// The SpeechT5 text encoder on the GPU: token ids -> encoder_last_hidden_state, the stage the reference runs once per sentence before its
// decoder loop (HelloSippyRTPipe.py:111-116; transformers modeling_speecht5.py SpeechT5EncoderWithTextPrenet, eval mode: no dropout)
//
//     prenet       x = embed_tokens[id] + alpha * pe[pos]                                        :765-781, scaled sinusoidal positions :400-422
//     layer_norm   x = LayerNorm(x), BEFORE the layers; there is no norm after the last one       :1292
//     12 layers    post-LN: h = LN1(x + out_proj(attn(x)));  x = LN2(h + W2 gelu(W1 h + b1) + b2)  :1013-1066
//     attention    12 heads of 64, q scaled by 1/8 (folded into the q weights at pack time, exact); score[i][j] = q_i.k_j +
//                  q_i.pe_k[clamp(i - j, -160, 159) + 160] (relative positions :425-442, :939-945), keys past the sentence masked (:1286)
//
// Ragged: only the valid tokens of a sentence are ever computed.  The sentences of a call are packed back to back ("rows") and cut into
// passes of at most max_tokens rows (a sentence is never split); every Linear of a pass is ONE GEMM over all its rows, attention runs per
// (sentence, head) over that sentence's rows only, and the last layer's output is scattered into the caller's (n, L, 768) grid with zeros at
// padded positions.  A row's arithmetic does not depend on its companions, so a sentence's output is bitwise the same alone, in a cohort, or
// in any pass.
//
// B2_MODE_FP32: every Linear through the CUDA-core conv kernel (as in decoder.cu).  B2_MODE_BF16: every Linear through the tcgen05 GEMM of
// gemm_tc.cuh (bf16 operands by TMA, fp32 accumulators, bias / GELU in the epilogue); fp32 residual stream, LayerNorm, q / k / v and attention.
#include "common.cuh"
#include "layers.cuh"
#include "serve.cuh"
#include "../../include/infernos_b200.h"

#include <math.h>
#include <stdlib.h>
#include <algorithm>
#include <string>
#include <vector>

using namespace b2;

namespace {

constexpr int H = 768, NL = 12, NH = 12, HD = 64, FFN = 3072, VOCAB = 81, MAXREL = 160, MAXPOS = 450;

// ---------------------------------------------------------------------------------------------------- kernels
// the sentence a packed row belongs to: off[] holds the packed start of every sentence of the call (off[n] = total rows)
__device__ __forceinline__ int row_session(const int32_t *off, int s0, int ns, int g) {
    int lo = s0, hi = s0 + ns - 1;
    while (lo < hi) {
        const int mid = (lo + hi + 1) >> 1;
        if (off[mid] <= g) lo = mid; else hi = mid - 1;
    }
    return lo;
}

// prologue, one CTA (256 threads) per packed row of the pass: x = E[id] + alpha * pe[pos], x = LayerNorm(x) -> fp32 residual stream h and
// (bf16 mode) its bf16 copy hb.  An id outside [0, 81) is embedded as zeros and flagged (bit 0 of *err).
__global__ void __launch_bounds__(256) k_enc_embed(const int32_t *__restrict__ ids, int L, const int32_t *__restrict__ off, int s0, int ns, int row0, int M,
                                                  const float *__restrict__ emb, const float *__restrict__ alpha, const float *__restrict__ pe,
                                                  const float *__restrict__ lnw, const float *__restrict__ lnb, float *__restrict__ h,
                                                  __nv_bfloat16 *__restrict__ hb, int *__restrict__ err) {
    pdl_trigger();
    pdl_wait(ids, off, emb, alpha, pe, lnw, lnb);
    __shared__ float red[8];
    const int r = blockIdx.x, tid = threadIdx.x;
    if (r >= M) return;
    const int g = row0 + r, s = row_session(off, s0, ns, g), pos = g - off[s];
    const int id = ids[(size_t)s * L + pos];
    const bool ok = id >= 0 && id < VOCAB;
    if (!ok && tid == 0) atomicOr(err, 1);
    const float a = alpha[0];
    float v[3], sum = 0.0f;
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const int c = tid + 256 * i;
        v[i] = (ok ? emb[(size_t)id * H + c] : 0.0f) + a * pe[(size_t)pos * H + c];
        sum += v[i];
    }
    const float mean = block_sum(sum, red) * (1.0f / H);
    float q = 0.0f;
#pragma unroll
    for (int i = 0; i < 3; i++) { const float d = v[i] - mean; q += d * d; }
    const float rstd = rsqrtf(block_sum(q, red) * (1.0f / H) + 1e-5f);
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const int c = tid + 256 * i;
        const float y = (v[i] - mean) * rstd * lnw[c] + lnb[c];
        h[(size_t)r * H + c] = y;
        if (hb) hb[(size_t)r * H + c] = __float2bfloat16_rn(y);
    }
}

// Bidirectional attention of one (sentence, head, tile of 64 queries): one thread per query, online softmax over key tiles of 32.
// qkv [rows][q 768 | k 768 | v 768] fp32 (q pre-scaled by 1/8); pe_k [320][64] (relative-position keys, shared by the heads).
// Per key tile the CTA stages the tile's keys and values and the 95 pe_k rows its (query, key) pairs use -- row (i - j) - (i0 - j0 - 31)
// of the tile holds pe_k[clamp(i - j, -160, 159) + 160] -- so no per-pair tensor ever exists in memory.  Keys and values are read by every
// lane at the same address (broadcast); pe_k rows differ per lane and are padded to 68 floats (17 x 16 bytes: conflict-free 128-bit loads).
// CUDA-core fp32 throughout: 3 x 64 FMAs per (query, key) pair (q.k, q.pe_k, p.v).
constexpr int kAttQ = 64, kAttK = 32, kAttKC = 8, kPeRows = kAttQ + kAttK - 1, kPeLd = 68;
template <bool BF>
__global__ void __launch_bounds__(kAttQ) k_enc_attend(const float *__restrict__ qkv, const int32_t *__restrict__ off, int s0, int row0,
                                                     const float *__restrict__ pe_k, float *__restrict__ ctx32, __nv_bfloat16 *__restrict__ ctxb) {
    pdl_trigger();
    pdl_wait(qkv, off, pe_k);
    __shared__ __align__(16) float ks[kAttK][HD];
    __shared__ __align__(16) float vs[kAttK][HD];
    __shared__ __align__(16) float ps[kPeRows][kPeLd];
    const int s = s0 + blockIdx.x, hh = blockIdx.y, i0 = blockIdx.z * kAttQ, t = threadIdx.x;
    const int b = off[s], len = off[s + 1] - b;
    if (i0 >= len) return;                                          // CTA-uniform
    const int i = i0 + t;
    const bool active = i < len;
    const float *base = qkv + (size_t)(b - row0) * (3 * H);
    float q[HD], acc[HD];
#pragma unroll
    for (int d4 = 0; d4 < HD / 4; d4++) {
        const float4 v = active ? *reinterpret_cast<const float4 *>(base + (size_t)i * (3 * H) + hh * HD + 4 * d4) : make_float4(0.f, 0.f, 0.f, 0.f);
        q[4 * d4] = v.x; q[4 * d4 + 1] = v.y; q[4 * d4 + 2] = v.z; q[4 * d4 + 3] = v.w;
    }
#pragma unroll
    for (int d = 0; d < HD; d++) acc[d] = 0.0f;
    float m = -INFINITY, l = 0.0f;
    for (int j0 = 0; j0 < len; j0 += kAttK) {
        __syncthreads();                                            // the previous tile is consumed
        for (int e = t; e < kAttK * (HD / 4); e += kAttQ) {
            const int r = e >> 4, c4 = (e & 15) * 4, j = j0 + r;
            float4 kv = make_float4(0.f, 0.f, 0.f, 0.f), vv = kv;
            if (j < len) {
                kv = *reinterpret_cast<const float4 *>(base + (size_t)j * (3 * H) + H + hh * HD + c4);
                vv = *reinterpret_cast<const float4 *>(base + (size_t)j * (3 * H) + 2 * H + hh * HD + c4);
            }
            *reinterpret_cast<float4 *>(&ks[r][c4]) = kv;
            *reinterpret_cast<float4 *>(&vs[r][c4]) = vv;
        }
        const int dlo = i0 - j0 - (kAttK - 1);
        for (int e = t; e < kPeRows * (HD / 4); e += kAttQ) {
            const int p = e >> 4, c4 = (e & 15) * 4;
            const int rel = min(max(dlo + p, -MAXREL), MAXREL - 1) + MAXREL;
            *reinterpret_cast<float4 *>(&ps[p][c4]) = *reinterpret_cast<const float4 *>(pe_k + (size_t)rel * HD + c4);
        }
        __syncthreads();
        if (!active) continue;
        const int nk = min(kAttK, len - j0);
        for (int jc = 0; jc < nk; jc += kAttKC) {
            float sc[kAttKC];
            float cmax = -INFINITY;
#pragma unroll
            for (int u = 0; u < kAttKC; u++) {
                const int jj = jc + u;
                sc[u] = -INFINITY;
                if (jj < nk) {
                    const float *kr = ks[jj], *pr = ps[t - jj + kAttK - 1];
                    float a0 = 0.0f, a1 = 0.0f, a2 = 0.0f, a3 = 0.0f;
#pragma unroll
                    for (int d4 = 0; d4 < HD / 4; d4++) {
                        const float4 kk = *reinterpret_cast<const float4 *>(kr + 4 * d4), pp = *reinterpret_cast<const float4 *>(pr + 4 * d4);
                        a0 = fmaf(q[4 * d4], kk.x, a0); a1 = fmaf(q[4 * d4 + 1], kk.y, a1); a2 = fmaf(q[4 * d4 + 2], kk.z, a2); a3 = fmaf(q[4 * d4 + 3], kk.w, a3);
                        a0 = fmaf(q[4 * d4], pp.x, a0); a1 = fmaf(q[4 * d4 + 1], pp.y, a1); a2 = fmaf(q[4 * d4 + 2], pp.z, a2); a3 = fmaf(q[4 * d4 + 3], pp.w, a3);
                    }
                    sc[u] = (a0 + a1) + (a2 + a3);
                    cmax = fmaxf(cmax, sc[u]);
                }
            }
            const float mn = fmaxf(m, cmax);
            const float corr = expf(m - mn);                        // 0 on the first chunk (m = -inf)
            l *= corr;
#pragma unroll
            for (int d = 0; d < HD; d++) acc[d] *= corr;
#pragma unroll
            for (int u = 0; u < kAttKC; u++) {
                const int jj = jc + u;
                if (jj < nk) {
                    const float p = expf(sc[u] - mn);
                    l += p;
                    const float *vr = vs[jj];
#pragma unroll
                    for (int d4 = 0; d4 < HD / 4; d4++) {
                        const float4 vv = *reinterpret_cast<const float4 *>(vr + 4 * d4);
                        acc[4 * d4] = fmaf(p, vv.x, acc[4 * d4]); acc[4 * d4 + 1] = fmaf(p, vv.y, acc[4 * d4 + 1]);
                        acc[4 * d4 + 2] = fmaf(p, vv.z, acc[4 * d4 + 2]); acc[4 * d4 + 3] = fmaf(p, vv.w, acc[4 * d4 + 3]);
                    }
                }
            }
            m = mn;
        }
    }
    if (!active) return;
    const float inv = 1.0f / l;
    const size_t o = (size_t)(b - row0 + i) * H + hh * HD;
#pragma unroll
    for (int d4 = 0; d4 < HD / 4; d4++) {
        const float x0 = acc[4 * d4] * inv, x1 = acc[4 * d4 + 1] * inv, x2 = acc[4 * d4 + 2] * inv, x3 = acc[4 * d4 + 3] * inv;
        if (BF) {
            __nv_bfloat162 lo = __floats2bfloat162_rn(x0, x1), hi = __floats2bfloat162_rn(x2, x3);
            *reinterpret_cast<uint2 *>(ctxb + o + 4 * d4) = make_uint2(*reinterpret_cast<uint32_t *>(&lo), *reinterpret_cast<uint32_t *>(&hi));
        } else {
            *reinterpret_cast<float4 *>(ctx32 + o + 4 * d4) = make_float4(x0, x1, x2, x3);
        }
    }
}

// the pass's sentences -> out (n, L, 768): the last layer's rows at valid positions, zeros at padded ones.  One CTA (192 threads, a float4
// each) per (sentence, position).
__global__ void __launch_bounds__(192) k_enc_out(const float *__restrict__ h, const int32_t *__restrict__ off, int s0, int row0, int L, float *__restrict__ out) {
    pdl_trigger();
    pdl_wait(h, off);
    const int s = s0 + blockIdx.x / L, pos = blockIdx.x % L, c4 = threadIdx.x * 4;
    const int b = off[s], len = off[s + 1] - b;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (pos < len) v = *reinterpret_cast<const float4 *>(h + (size_t)(b - row0 + pos) * H + c4);
    *reinterpret_cast<float4 *>(out + ((size_t)s * L + pos) * H + c4) = v;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------- host side
struct b2_enc : b2::LinearOwner {
    b2_enc() { what = "encoder"; }
    int max_tokens = 0, max_len = 0;
    bool finalized = false;
    DecLinear qkv[NL], o[NL], ff1[NL], ff2[NL];
    float *ln_w[NL][2] = {}, *ln_b[NL][2] = {};
    float *emb = nullptr, *alpha = nullptr, *pe = nullptr, *ln0_w = nullptr, *ln0_b = nullptr, *pe_k = nullptr;
    // rows of one pass
    float *h = nullptr, *tmp = nullptr, *qkv32 = nullptr, *ctx = nullptr, *f1 = nullptr;
    __nv_bfloat16 *hb = nullptr, *ctxb = nullptr, *f1b = nullptr;
    CUtensorMap tm_h, tm_ctx, tm_f1;
    // packed starts of a call's sentences: filled in pinned memory, copied to the device with one cudaMemcpyAsync; off_ev marks the copy done
    // so that the next call does not overwrite the pinned buffer before the copy engine has read it
    int32_t *h_off = nullptr, *d_off = nullptr;
    size_t off_cap = 0;
    cudaEvent_t off_ev = nullptr;
    int *err_h = nullptr, *err_d = nullptr;
};

namespace {

int finalize_enc(b2_enc *d) {
    const bool bf = d->mode == B2_MODE_BF16;
    const std::string P = "speecht5.encoder.prenet.", W = "speecht5.encoder.wrapped_encoder.";
    const HostTensor *t;
    if (!(t = need(d, P + "embed_tokens.weight", {VOCAB, H})) || upload_vec(d, &d->emb, *t)) return 1;
    if (!(t = need(d, P + "encode_positions.alpha", {}))) { if (!(t = need(d, P + "encode_positions.alpha", {1}))) return 1; }
    if (upload_vec(d, &d->alpha, *t)) return 1;
    if (!(t = need(d, "pe", {(int64_t)d->max_len, H})) || upload_vec(d, &d->pe, *t)) return 1;
    if (!(t = need(d, W + "layer_norm.weight", {H})) || upload_vec(d, &d->ln0_w, *t)) return 1;
    if (!(t = need(d, W + "layer_norm.bias", {H})) || upload_vec(d, &d->ln0_b, *t)) return 1;
    if (!(t = need(d, W + "embed_positions.pe_k.weight", {2 * MAXREL, HD})) || upload_vec(d, &d->pe_k, *t)) return 1;
    for (int i = 0; i < NL; i++) {
        const std::string L = W + "layers." + std::to_string(i) + ".";
        {   // q (pre-scaled by 1/sqrt(64): exact, a power of two; the relative-position term uses the scaled q too, :891, :939) | k | v
            std::vector<float> Wt((size_t)3 * H * H, 0.0f), B((size_t)3 * H, 0.0f);
            const char *nm[3] = {"q_proj", "k_proj", "v_proj"};
            for (int j = 0; j < 3; j++) {
                const HostTensor *w = need(d, L + "attention." + nm[j] + ".weight", {H, H}), *b = need(d, L + "attention." + nm[j] + ".bias", {H});
                if (!w || !b) return 1;
                fill_linear(Wt, B, H, 3 * H, j * H, *w, *b, j == 0 ? 0.125f : 1.0f);
            }
            if (upload_linear(d, d->qkv[i], H, 3 * H, Wt, B)) return 1;
        }
        if (pack_one(d, d->o[i], L + "attention.out_proj", H, H, H, H)) return 1;
        if (pack_one(d, d->ff1[i], L + "feed_forward.intermediate_dense", FFN, H, H, FFN)) return 1;
        if (pack_one(d, d->ff2[i], L + "feed_forward.output_dense", H, FFN, FFN, H)) return 1;
        const char *ln[2] = {"layer_norm", "final_layer_norm"};
        for (int j = 0; j < 2; j++) {
            const HostTensor *w = need(d, L + ln[j] + ".weight", {H}), *b = need(d, L + ln[j] + ".bias", {H});
            if (!w || !b) return 1;
            if (upload_vec(d, &d->ln_w[i][j], *w) || upload_vec(d, &d->ln_b[i][j], *b)) return 1;
        }
    }
    const size_t R = (size_t)d->max_tokens;
    if (dalloc(d, &d->h, R * H) || dalloc(d, &d->tmp, R * H) || dalloc(d, &d->qkv32, R * 3 * H)) return 1;
    if (bf) {
        if (dalloc(d, &d->hb, R * H) || dalloc(d, &d->ctxb, R * H) || dalloc(d, &d->f1b, R * FFN)) return 1;
        const int Ri = (int)R;
        if (make_map(&d->tm_h, d->hb, Ri, H, 128) || make_map(&d->tm_ctx, d->ctxb, Ri, H, 128) || make_map(&d->tm_f1, d->f1b, Ri, FFN, 128)) return 1;
    } else {
        if (dalloc(d, &d->ctx, R * H) || dalloc(d, &d->f1, R * FFN)) return 1;
    }
    B2_CUDA_OK(cudaEventCreateWithFlags(&d->off_ev, cudaEventDisableTiming));
    B2_CUDA_OK(cudaHostAlloc((void **)&d->err_h, sizeof(int), cudaHostAllocMapped));
    *d->err_h = 0;
    B2_CUDA_OK(cudaHostGetDevicePointer((void **)&d->err_d, d->err_h, 0));
    d->raw.clear();
    d->finalized = true;
    return 0;
}

int poll_enc_errors(b2_enc *d, const char *who) {
    if (!d->err_h) return 0;
    const int f = *(volatile int *)d->err_h;
    if (!f) return 0;
    *(volatile int *)d->err_h = 0;
    return set_error("%s: an earlier encoder call on this handle was given token ids outside [0, %d) (embedded as zeros)", who, VOCAB);
}

// one pass: sentences [s0, s0 + ns), packed rows [row0, row0 + M), the longest of them maxlen tokens
int pass_impl(b2_enc *d, const int32_t *d_ids, int L, int s0, int ns, int row0, int M, int maxlen, float *d_out, cudaStream_t st) {
    const bool bf = d->mode == B2_MODE_BF16, pdl = d->use_pdl;
    const int32_t *off = d->d_off;
    B2_CUDA_OK(launch_k(k_enc_embed, dim3((unsigned)M), dim3(256), 0, st, pdl, d_ids, L, off, s0, ns, row0, M, (const float *)d->emb, (const float *)d->alpha,
                        (const float *)d->pe, (const float *)d->ln0_w, (const float *)d->ln0_b, d->h, bf ? d->hb : (__nv_bfloat16 *)nullptr, d->err_d));
    B2_LAUNCH_OK("k_enc_embed");
    const dim3 gA((unsigned)ns, NH, (unsigned)cdiv(maxlen, kAttQ));
    for (int i = 0; i < NL; i++) {
        if (linear(d, d->qkv[i], d->h, &d->tm_h, M, 0, nullptr, d->qkv32, nullptr, st)) return 1;
        if (bf) B2_CUDA_OK(launch_k(k_enc_attend<true>, gA, dim3(kAttQ), 0, st, pdl, (const float *)d->qkv32, off, s0, row0, (const float *)d->pe_k, (float *)nullptr, d->ctxb));
        else B2_CUDA_OK(launch_k(k_enc_attend<false>, gA, dim3(kAttQ), 0, st, pdl, (const float *)d->qkv32, off, s0, row0, (const float *)d->pe_k, d->ctx, (__nv_bfloat16 *)nullptr));
        B2_LAUNCH_OK("k_enc_attend");
        if (linear(d, d->o[i], d->ctx, &d->tm_ctx, M, 0, nullptr, d->tmp, nullptr, st)) return 1;
        B2_CUDA_OK(launch_k(k_add_ln, dim3((unsigned)M), dim3(256), 0, st, pdl, d->h, (const float *)d->tmp, (const float *)d->ln_w[i][0], (const float *)d->ln_b[i][0],
                            bf ? d->hb : (__nv_bfloat16 *)nullptr, M));
        B2_LAUNCH_OK("k_add_ln");
        if (linear(d, d->ff1[i], d->h, &d->tm_h, M, 2, nullptr, bf ? nullptr : d->f1, bf ? d->f1b : nullptr, st)) return 1;
        if (linear(d, d->ff2[i], d->f1, &d->tm_f1, M, 0, nullptr, d->tmp, nullptr, st)) return 1;
        B2_CUDA_OK(launch_k(k_add_ln, dim3((unsigned)M), dim3(256), 0, st, pdl, d->h, (const float *)d->tmp, (const float *)d->ln_w[i][1], (const float *)d->ln_b[i][1],
                            bf ? d->hb : (__nv_bfloat16 *)nullptr, M));
        B2_LAUNCH_OK("k_add_ln");
    }
    B2_CUDA_OK(launch_k(k_enc_out, dim3((unsigned)(ns * L)), dim3(H / 4), 0, st, pdl, (const float *)d->h, off, s0, row0, L, d_out));
    B2_LAUNCH_OK("k_enc_out");
    return 0;
}

}  // namespace

void b2::enc_limits(const b2_enc *e, int *max_tokens, int *max_len, int *vocab) {
    *max_tokens = e->max_tokens; *max_len = e->max_len; *vocab = VOCAB;
}

#define ENC_GUARD(d)                                                                                  \
    if (!(d)) return set_error("null encoder handle");                                                \
    {                                                                                                 \
        cudaError_t _e = cudaSetDevice((d)->device);                                                  \
        if (_e != cudaSuccess) return set_error("cudaSetDevice(%d): %s", (d)->device, cudaGetErrorString(_e)); \
    }

extern "C" {

b2_enc *b2_enc_create(int device, int mode, int max_tokens, int max_len) {
    if (mode != B2_MODE_FP32 && mode != B2_MODE_BF16) { set_error("b2_enc_create: mode must be B2_MODE_FP32 or B2_MODE_BF16"); return nullptr; }
    if (max_tokens < 1 || max_len < 1 || max_len > MAXPOS) { set_error("b2_enc_create: need max_tokens >= 1 and 1 <= max_len <= %d", MAXPOS); return nullptr; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) { set_error("no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e)); return nullptr; }
    if (device < 0 || device >= ndev) { set_error("device %d out of range (%d devices)", device, ndev); return nullptr; }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major != 10) { set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor); return nullptr; }
    b2_enc *d = new b2_enc();
    d->device = device; d->mode = mode; d->max_tokens = max_tokens; d->max_len = max_len;
    d->use_pdl = pdl_enabled() && !(getenv("B2_ENC_PDL") && atoi(getenv("B2_ENC_PDL")) == 0);
    return d;
}

void b2_enc_destroy(b2_enc *d) {
    if (!d) return;
    cudaSetDevice(d->device);
    cudaDeviceSynchronize();
    for (void *p : d->allocs) cudaFree(p);
    if (d->d_off) cudaFree(d->d_off);
    if (d->h_off) cudaFreeHost(d->h_off);
    if (d->off_ev) cudaEventDestroy(d->off_ev);
    if (d->err_h) cudaFreeHost(d->err_h);
    delete d;
}

size_t b2_enc_device_bytes(const b2_enc *d) { return d ? d->device_bytes : 0; }

int b2_enc_load_tensor(b2_enc *d, const char *key, const float *h, const int64_t *shape, int ndim) {
    if (!d) return set_error("null encoder handle");
    if (d->finalized) return set_error("encoder weights are already finalized");
    if (!key || !h || ndim < 0 || ndim > 4 || (ndim > 0 && !shape)) return set_error("b2_enc_load_tensor: bad arguments");
    HostTensor t;
    size_t n = 1;
    for (int i = 0; i < ndim; i++) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
    t.data.assign(h, h + n);
    d->raw[key] = std::move(t);
    return 0;
}

int b2_enc_finalize(b2_enc *d) {
    ENC_GUARD(d);
    if (d->finalized) return set_error("encoder weights are already finalized");
    return finalize_enc(d);
}

int b2_enc_forward(b2_enc *d, const int32_t *d_ids, const int32_t *h_len, int n, int L, float *d_out, void *stream) {
    ENC_GUARD(d);
    if (!d->finalized) return set_error("b2_enc_finalize has not been called");
    if (n < 0 || L < 1) return set_error("b2_enc_forward: bad shape n=%d L=%d", n, L);
    if (L > d->max_len) return set_error("b2_enc_forward: %d positions exceed max_len=%d", L, d->max_len);
    if (n == 0) return 0;
    if (!d_ids || !d_out) return set_error("b2_enc_forward: null pointer");
    if (poll_enc_errors(d, "b2_enc_forward")) return 1;
    for (int s = 0; s < n; s++) {
        const int len = h_len ? h_len[s] : L;
        if (len < 1 || len > L) return set_error("b2_enc_forward: sentence %d has length %d outside [1, %d]", s, len, L);
        if (len > d->max_tokens) return set_error("b2_enc_forward: sentence %d has %d tokens, more than max_tokens=%d (a sentence is never split)", s, len, d->max_tokens);
    }
    cudaStream_t st = (cudaStream_t)stream;
    B2_CUDA_OK(cudaEventSynchronize(d->off_ev));                 // the previous call's copy has read the pinned buffer
    if ((size_t)n + 1 > d->off_cap) {
        const size_t cap = std::max<size_t>((size_t)n + 1, 2 * d->off_cap);
        B2_CUDA_OK(cudaDeviceSynchronize());                     // earlier passes may still read d_off
        if (d->d_off) { cudaFree(d->d_off); d->device_bytes -= d->off_cap * sizeof(int32_t); d->d_off = nullptr; }
        if (d->h_off) { cudaFreeHost(d->h_off); d->h_off = nullptr; }
        d->off_cap = 0;
        B2_CUDA_OK(cudaMalloc((void **)&d->d_off, cap * sizeof(int32_t)));
        B2_CUDA_OK(cudaHostAlloc((void **)&d->h_off, cap * sizeof(int32_t), cudaHostAllocDefault));
        d->off_cap = cap;
        d->device_bytes += cap * sizeof(int32_t);
    }
    d->h_off[0] = 0;
    for (int s = 0; s < n; s++) d->h_off[s + 1] = d->h_off[s] + (h_len ? h_len[s] : L);
    B2_CUDA_OK(cudaMemcpyAsync(d->d_off, d->h_off, ((size_t)n + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    B2_CUDA_OK(cudaEventRecord(d->off_ev, st));
    for (int s0 = 0; s0 < n;) {
        int s1 = s0, maxlen = 0;
        const int row0 = d->h_off[s0];
        while (s1 < n && d->h_off[s1 + 1] - row0 <= d->max_tokens) { maxlen = std::max(maxlen, d->h_off[s1 + 1] - d->h_off[s1]); s1++; }
        if (pass_impl(d, d_ids, L, s0, s1 - s0, row0, d->h_off[s1] - row0, maxlen, d_out, st)) return 1;
        s0 = s1;
    }
    return 0;
}

int b2_enc_poll_errors(b2_enc *d, void *stream) {
    ENC_GUARD(d);
    B2_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    return poll_enc_errors(d, "b2_enc_poll_errors");
}

}  // extern "C"
