// The autoregressive front half on the GPU (SURVEY.md section 8 f3): what HelloSippyRTPipe.infer() does before the tail,
// /root/reference/HelloSippyTTSRT/HelloSippyRTPipe.py:195-229, per decoder step and per session of the batch
//
//     prenet(output_sequence, speaker)[:, -1:]   transformers modeling_speecht5.py:648-697 (two Linear+ReLU+always-on dropout, final Linear,
//                                                scaled sinusoidal position :400-422, speaker projection)
//     wrapped_decoder(.., past_key_values)       six post-LN decoder layers :1070-1160: self-attention over a KV cache, cross-attention over
//                                                the encoder states (keys / values projected once per sentence), GELU feed-forward
//     feat_out -> 2 mel frames, prob_out -> 2 stop probabilities   :740-750
//
// batched over sessions that live in SLOTS (the same ids as the tail's pre_frames slots): per slot a self-attention KV cache
// [slot][layer][step][K 768 | V 768], the cross-attention keys / values [slot][layer][pos][K | V], the normalised speaker vector, the last
// emitted frame and the step counter.  Nothing of this leaves the device between steps; the mel frames of a call are written where
// b2_tts_tail2(B2_TAIL_APPLY_POSTNET) reads them.
//
// B2_MODE_FP32: every Linear through the CUDA-core conv kernel (a Linear is a 1-tap convolution), fp32 caches.
// B2_MODE_BF16: every Linear through k_gemm_tc below -- a tcgen05 GEMM whose BOTH operands arrive by TMA (activations [rows][K] and
//               weights [N][K], 128-byte swizzle, 4-stage mbarrier ring), fp32 accumulators in TMEM, bias / ReLU / GELU / dropout scale
//               fused into the epilogue; bf16 caches, fp32 residual stream and LayerNorm.
#include "common.cuh"
#include "ctx.cuh"
#include "conv_simt.cuh"
#include "conv_umma.cuh"
#include "umma_ptx.cuh"
#include "gemm_tc.cuh"
#include "layers.cuh"
#include "serve.cuh"
#include "../../include/infernos_b200.h"

#include <cuda.h>
#include <math.h>
#include <stdlib.h>
#include <utility>
#include <string.h>
#include <algorithm>
#include <map>
#include <string>
#include <vector>

using namespace b2;

namespace {

constexpr int H = 768, NL = 6, NH = 12, HD = 64, FFN = 3072, PRE = 256, SPK = 512, NMEL = 80, OUTP = 192;   // OUTP: feat 160 | prob 2 | pad

// ---------------------------------------------------------------------------------------------------- tcgen05 GEMM
struct GemmParams {
    const float *bias;        // [N]
    const float *colscale;    // optional [N]: multiplied in after the activation (the prenet's dropout keep-mask x 1/(1-p))
    float *out32;             // optional [M][ldo] fp32
    __nv_bfloat16 *outb;      // optional [M][ldo] bf16
    int M, N, K, ldo, act;    // act: 0 none, 1 relu, 2 gelu (erf)
};

__device__ __forceinline__ void tma_load_2d(uint32_t dst, const void *tmap, uint32_t bar, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
                 ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1) : "memory");
}

// C[m][n] = act(sum_k A[m][k] * W[n][k] + bias[n]) * colscale[n];  one 128 x NT tile per CTA.
// warps 0..3 epilogue (TMEM lane quadrant = warp), warp 4 TMA producer, warp 5 TMEM allocation + MMA issue.
// kGemmStages ring stages: with the decoder's K = 768 (12 K blocks) an 8-deep ring has two thirds of the tile's operands in flight at once
template <int NT, int kGemmStages>
__global__ void __launch_bounds__(192) k_gemm_tc(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB, const GemmParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    constexpr uint32_t kABytes = 128 * 64 * 2, kBBytes = NT * 64 * 2, kStage = kABytes + kBBytes;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem + kGemmStages * kStage);
    const uint32_t bar0 = smem_u32(bars);
    auto FULL = [&](int s) { return bar0 + 8u * (uint32_t)s; };
    auto EMPTY = [&](int s) { return bar0 + 8u * (uint32_t)(kGemmStages + s); };
    const uint32_t DONE = bar0 + 8u * (uint32_t)(2 * kGemmStages);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * kGemmStages + 1);
    const int m0 = blockIdx.x * 128, n0 = blockIdx.y * NT;
    const int nkb = p.K / 64;
    pdl_trigger();

    if (warp == 5) {
        if (lane == 0) {
            if (smem_u32(smem) & 1023u) __trap();
            for (int s = 0; s < kGemmStages; s++) { mbar_init(FULL(s), 1); mbar_init(EMPTY(s), 1); }
            mbar_init(DONE, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)NT) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (warp == 4 && lane == 0) {
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA) : "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmB) : "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = *tmem_slot;
    pdl_wait();                                   // everything above overlapped the previous kernel; its results are read from here on

    if (warp == 4) {
        if (lane == 0) {
            for (int kb = 0; kb < nkb; kb++) {
                const int s = kb % kGemmStages;
                mbar_wait(EMPTY(s), (uint32_t)(((kb / kGemmStages) & 1) ^ 1));
                mbar_expect_tx(FULL(s), kStage);
                const uint32_t dst = smem_u32(smem + (size_t)s * kStage);
                tma_load_2d(dst, &tmA, FULL(s), kb * 64, m0);
                tma_load_2d(dst + kABytes, &tmB, FULL(s), kb * 64, n0);
            }
        }
        __syncwarp();
    } else if (warp == 5) {
        if (elect_one()) {
            // kind::f16: D = f32, A = B = bf16, both K-major, N = NT, M = 128
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(NT >> 3) << 17) | ((128u >> 4) << 24);
            for (int kb = 0; kb < nkb; kb++) {
                const int s = kb % kGemmStages;
                mbar_wait(FULL(s), (uint32_t)((kb / kGemmStages) & 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                const uint32_t a_u32 = smem_u32(smem + (size_t)s * kStage);
                const uint64_t ad = smem_desc(a_u32, 0u, 1024u, 2u), bd = smem_desc(a_u32 + kABytes, 0u, 1024u, 2u);     // SWIZZLE_128B, 8-row groups 1 KB apart
#pragma unroll
                for (int ks = 0; ks < 4; ks++) umma_f16(tmem, ad + (uint64_t)(ks * 2), bd + (uint64_t)(ks * 2), idesc, (kb | ks) ? 1u : 0u);
                umma_commit(EMPTY(s));
            }
            umma_commit(DONE);
        }
        __syncwarp();
    } else {
        mbar_wait(DONE, 0);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        const int row = m0 + warp * 32 + lane;
        const uint32_t tm_lane = (uint32_t)(warp * 32) << 16;
#pragma unroll 1
        for (int c = 0; c < NT / 32; c++) {
            uint32_t v[32];
            tmem_ld32(tmem + tm_lane + (uint32_t)(c * 32), v);
            const int col = n0 + c * 32;
            if (row < p.M && col < p.N) {
                float o[32];
#pragma unroll
                for (int j = 0; j < 32; j++) {
                    float x = __uint_as_float(v[j]) + __ldg(p.bias + col + j);
                    if (p.act == 1) x = fmaxf(x, 0.0f);
                    else if (p.act == 2) x = gelu_erf(x);
                    if (p.colscale) x *= __ldg(p.colscale + col + j);
                    o[j] = x;
                }
                const size_t base = (size_t)row * p.ldo + col;
                if (p.out32) {
#pragma unroll
                    for (int j = 0; j < 8; j++) *reinterpret_cast<float4 *>(p.out32 + base + 4 * j) = make_float4(o[4 * j], o[4 * j + 1], o[4 * j + 2], o[4 * j + 3]);
                }
                if (p.outb) {
#pragma unroll
                    for (int j = 0; j < 4; j++) {
                        uint32_t pk[4];
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            __nv_bfloat162 h2 = __floats2bfloat162_rn(o[8 * j + 2 * e], o[8 * j + 2 * e + 1]);
                            pk[e] = *reinterpret_cast<uint32_t *>(&h2);
                        }
                        *reinterpret_cast<uint4 *>(p.outb + base + 8 * j) = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                    }
                }
            }
        }
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (warp == 5) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem), "r"((uint32_t)NT) : "memory");
}

// ---------------------------------------------------------------------------------------------------- small kernels
// row m of the step <- slot state: the last emitted frame (prenet input) and its position in output_sequence
// A slot id outside the pool is flagged (bit 0 of *err) and redirected to the scratch slot `max_sessions`, so that it can neither read
// nor corrupt another session's state; rowslot[] carries the sanitised ids to the rest of the step.
template <bool BF>
__global__ void k_dec_gather(const int32_t *__restrict__ slots, const float *__restrict__ last, const int32_t *__restrict__ step, int M,
                             float *__restrict__ x0, __nv_bfloat16 *__restrict__ x0b, int32_t *__restrict__ rowpos, int32_t *__restrict__ rowslot,
                             int max_sessions, int max_steps, int *__restrict__ err) {
    pdl_trigger();
    pdl_wait(slots, last, step);
    const int m = blockIdx.x, c = threadIdx.x;            // 128 threads
    if (m >= M) return;
    int sl = slots[m];
    if (sl == -1) sl = max_sessions;                       // padding row of a graph bucket: computed on the scratch slot, not an error
    else if (sl < 0 || sl >= max_sessions) { if (c == 0) atomicOr(err, 1); sl = max_sessions; }
    if (c == 0) rowslot[m] = sl;
    int t = step[sl];
    if (t >= max_steps) { if (c == 0 && sl != max_sessions) atomicOr(err, 4); t = max_steps - 1; }
    if (c == 0) rowpos[m] = t;
    const float v = c < NMEL ? last[(size_t)sl * NMEL + c] : 0.0f;
    if (BF) x0b[(size_t)m * 128 + c] = __float2bfloat16_rn(v);
    else if (c < NMEL) x0[(size_t)m * NMEL + c] = v;
}

// cat[m] = (fin[m] + alpha * pe[pos[m]]) | speaker[slot]      (modeling_speecht5.py:420, :696-698)
template <bool BF>
__global__ void k_pos_cat(const float *__restrict__ fin, const float *__restrict__ pe, const float *__restrict__ alpha, const int32_t *__restrict__ rowpos,
                          const int32_t *__restrict__ slots, const float *__restrict__ spk, int M, float *__restrict__ cat, __nv_bfloat16 *__restrict__ catb) {
    pdl_trigger();
    pdl_wait(fin, rowpos, slots, spk);
    const int m = blockIdx.x;
    if (m >= M) return;
    const int pos = rowpos[m], sl = slots[m];
    const float a = alpha[0];
    for (int c = threadIdx.x; c < H + SPK; c += blockDim.x) {
        const float v = c < H ? fin[(size_t)m * H + c] + a * pe[(size_t)pos * H + c] : spk[(size_t)sl * SPK + (c - H)];
        if (BF) catb[(size_t)m * (H + SPK) + c] = __float2bfloat16_rn(v);
        else cat[(size_t)m * (H + SPK) + c] = v;
    }
}

__device__ __forceinline__ void st_kv(float *p, float v) { *p = v; }
__device__ __forceinline__ void st_kv(__nv_bfloat16 *p, float v) { *p = __float2bfloat16_rn(v); }

// 8 consecutive cache elements (one 16-byte piece of a bf16 row, two of an fp32 row) as floats
__device__ __forceinline__ void ld_kv8(const float *p, float (&v)[8]) {
    const float4 a = *reinterpret_cast<const float4 *>(p), b = *reinterpret_cast<const float4 *>(p + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void ld_kv8(const __nv_bfloat16 *p, float (&v)[8]) {
    const uint4 u = *reinterpret_cast<const uint4 *>(p);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        v[2 * i] = __uint_as_float(w[i] << 16);
        v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}

// the same piece held as loaded (bf16: four registers instead of eight) until it is used
struct Raw8f { float4 a, b; };
__device__ __forceinline__ void ld_raw8(const float *p, Raw8f &r) { r.a = *reinterpret_cast<const float4 *>(p); r.b = *reinterpret_cast<const float4 *>(p + 4); }
__device__ __forceinline__ void ld_raw8(const __nv_bfloat16 *p, uint4 &r) { r = *reinterpret_cast<const uint4 *>(p); }
__device__ __forceinline__ void cvt_raw8(const Raw8f &r, float (&v)[8]) { v[0] = r.a.x; v[1] = r.a.y; v[2] = r.a.z; v[3] = r.a.w; v[4] = r.b.x; v[5] = r.b.y; v[6] = r.b.z; v[7] = r.b.w; }
__device__ __forceinline__ void cvt_raw8(const uint4 &u, float (&v)[8]) {
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
    for (int i = 0; i < 4; i++) {
        v[2 * i] = __uint_as_float(w[i] << 16);
        v[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
    }
}
#ifndef B2_ATT_U
#define B2_ATT_U 2          // measured: 2 positions in flight at 12 CTAs per SM (40 registers) beat 4 at 9 (56 registers): 22.2 vs 23.9 ms per call, same box
#endif
#ifndef B2_ATT_UQ
#define B2_ATT_UQ B2_ATT_U
#endif
#ifndef B2_ATT_UP
#define B2_ATT_UP B2_ATT_U
#endif
constexpr int kAttUQ = B2_ATT_UQ, kAttUP = B2_ATT_UP;            // cached positions per 8-lane group and trip (loads in flight per lane): scores, context
template <typename KV> struct RawOf { typedef Raw8f type; };
template <> struct RawOf<__nv_bfloat16> { typedef uint4 type; };

// One query position against a cached sequence, one CTA (128 threads) per (row, head)  (SpeechT5Attention.forward, :872-986; the 1/sqrt(64)
// scaling is folded into the q projection at pack time).  SELF: the row's new key / value (columns 768.. / 1536.. of qkv) are appended to
// the slot's cache at its step first, and the sequence is steps 0 .. step; otherwise keys / values are the sentence's cross-attention cache
// and the sequence is its first enc_len positions (the reference's padding mask).  ctx32 / ctxb: [M][768].
// Memory-bound (every cached key and value is read once per step): 8 lanes share one position, each owning 8 of the head's 64 dimensions,
// so a warp reads four whole 128-byte (bf16) rows per load instruction; scores are reduced over the 8 lanes by shuffles, the value sum is
// kept per lane and folded over positions at the end.
#ifndef B2_ATT_MINB
#define B2_ATT_MINB 12
#endif
template <typename KV, bool SELF>
__global__ void __launch_bounds__(128, B2_ATT_MINB) k_attend(const float *__restrict__ q, int ldq, const int32_t *__restrict__ slots, const int32_t *__restrict__ rowpos,
                                               const int32_t *__restrict__ enc_len, KV *__restrict__ cache, size_t slot_stride, size_t pos_stride,
                                               size_t layer_off, float *__restrict__ ctx32, __nv_bfloat16 *__restrict__ ctxb) {
    pdl_trigger();
    pdl_wait(q, slots, rowpos, enc_len, cache);
    extern __shared__ float sm[];                      // [T] scores | 64 q | 4 x 64 partial sums | 8 red
    const int m = blockIdx.x, h = blockIdx.y, tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31, grp = lane >> 3, c8 = (lane & 7) * 8;
    const int sl = slots[m];
    const int T = SELF ? rowpos[m] + 1 : enc_len[sl];
    float *sc = sm, *qs = sm + ((T + 3) & ~3), *part = qs + HD, *red = part + 4 * HD;
    KV *base = cache + (size_t)sl * slot_stride + layer_off + (size_t)h * HD;
    if (tid < HD) {
        qs[tid] = q[(size_t)m * ldq + h * HD + tid];
        if (SELF) {
            KV *dst = base + (size_t)(T - 1) * pos_stride;
            st_kv(dst + tid, q[(size_t)m * ldq + H + h * HD + tid]);
            st_kv(dst + H + tid, q[(size_t)m * ldq + 2 * H + h * HD + tid]);
        }
    }
    __syncthreads();
    float qv[8];
#pragma unroll
    for (int e = 0; e < 8; e++) qv[e] = qs[c8 + e];
    float mx = -INFINITY;
    // kAttUQ positions per 8-lane group and trip, all their loads issued before the first is used: with one 16-byte load in flight per lane the
    // kernel read the cache at 62 % of the HBM peak (ncu, round 2); the arithmetic and its order are unchanged
    for (int jb = warp * 4; jb < T; jb += 16 * kAttUQ) {
        typename RawOf<KV>::type raw[kAttUQ];
#pragma unroll
        for (int u = 0; u < kAttUQ; u++) {
            const int j = jb + 16 * u + grp;
            if (j < T) ld_raw8(base + (size_t)j * pos_stride + c8, raw[u]);
        }
#pragma unroll
        for (int u = 0; u < kAttUQ; u++) {
            if (jb + 16 * u >= T) break;                  // warp-uniform: a short sequence costs one position's arithmetic, not four
            const int j = jb + 16 * u + grp;
            float acc = 0.0f;
            if (j < T) {
                float kv[8];
                cvt_raw8(raw[u], kv);
#pragma unroll
                for (int e = 0; e < 8; e++) acc = fmaf(qv[e], kv[e], acc);
            }
            acc += __shfl_xor_sync(0xffffffffu, acc, 1);
            acc += __shfl_xor_sync(0xffffffffu, acc, 2);
            acc += __shfl_xor_sync(0xffffffffu, acc, 4);
            if (j < T) {
                if ((lane & 7) == 0) sc[j] = acc;
                mx = fmaxf(mx, acc);
            }
        }
    }
    mx = block_max(mx, red);                            // (its barriers also publish sc[])
    float sum = 0.0f;
    for (int j = tid; j < T; j += 128) {
        const float e = expf(sc[j] - mx);
        sc[j] = e;
        sum += e;
    }
    sum = block_sum(sum, red);
    float acc[8];
#pragma unroll
    for (int e = 0; e < 8; e++) acc[e] = 0.0f;
    for (int jb = warp * 4 + grp; jb < T; jb += 16 * kAttUP) {
        typename RawOf<KV>::type raw[kAttUP];
#pragma unroll
        for (int u = 0; u < kAttUP; u++)
            if (jb + 16 * u < T) ld_raw8(base + (size_t)(jb + 16 * u) * pos_stride + H + c8, raw[u]);
#pragma unroll
        for (int u = 0; u < kAttUP; u++) {
            if (jb + 16 * u < T) {
                float vv[8];
                cvt_raw8(raw[u], vv);
                const float pj = sc[jb + 16 * u];
#pragma unroll
                for (int e = 0; e < 8; e++) acc[e] = fmaf(pj, vv[e], acc[e]);
            }
        }
    }
#pragma unroll
    for (int e = 0; e < 8; e++) {
        acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 8);
        acc[e] += __shfl_xor_sync(0xffffffffu, acc[e], 16);
    }
    if (grp == 0) {
#pragma unroll
        for (int e = 0; e < 8; e++) part[warp * HD + c8 + e] = acc[e];
    }
    __syncthreads();
    if (tid < HD) {
        const float o = (part[tid] + part[HD + tid] + part[2 * HD + tid] + part[3 * HD + tid]) / sum;
        if (ctx32) ctx32[(size_t)m * H + h * HD + tid] = o;
        if (ctxb) ctxb[(size_t)m * H + h * HD + tid] = __float2bfloat16_rn(o);
    }
}

// after the speaker projection: h = relu(x) as fp32 residual stream + bf16 operand
__global__ void k_relu_dual(const float *__restrict__ x, float *__restrict__ h, __nv_bfloat16 *__restrict__ hb, size_t n) {
    pdl_trigger();
    pdl_wait(x);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const float v = fmaxf(x[i], 0.0f);
        h[i] = v;
        if (hb) hb[i] = __float2bfloat16_rn(v);
    }
}

// out[m] = feat (2 x 80) | prob logits (2) -> the call's mel [M][2*nsteps][80], the stop probabilities [M][nsteps][2], the slot's last frame and step
__global__ void k_dec_finish(const float *__restrict__ out, const int32_t *__restrict__ slots, int M, int s, int nsteps,
                             float *__restrict__ mel, float *__restrict__ prob, float *__restrict__ last, int32_t *__restrict__ step, int max_sessions) {
    pdl_trigger();
    pdl_wait(out, slots, last, step);
    const int m = blockIdx.x, c = threadIdx.x;           // 192 threads
    if (m >= M) return;
    const int sl = slots[m];
    const float v = out[(size_t)m * OUTP + c];
    if (c < 2 * NMEL) {
        mel[((size_t)m * 2 * nsteps + 2 * s) * NMEL + c] = v;
        if (c >= NMEL) last[(size_t)sl * NMEL + (c - NMEL)] = v;
    } else if (c < 2 * NMEL + 2) {
        prob[((size_t)m * nsteps + s) * 2 + (c - 2 * NMEL)] = 1.0f / (1.0f + expf(-v));
    }
    if (c == 0 && sl != max_sessions) step[sl] += 1;       // the scratch slot (padding rows, rejected ids) stays at step 0
}

// start of a sentence: zero frame, step 0, normalised speaker vector (F.normalize: x / max(||x||, 1e-12)), encoder length
__global__ void __launch_bounds__(256) k_dec_init(const int32_t *__restrict__ slots, const float *__restrict__ speaker, const int32_t *__restrict__ enc_len_in, int L,
                                                 int max_enc, float *__restrict__ last, int32_t *__restrict__ step, float *__restrict__ spk,
                                                 int32_t *__restrict__ enc_len, int max_sessions, int *__restrict__ err) {
    __shared__ float red[8];
    const int m = blockIdx.x, tid = threadIdx.x;
    const int sl = slots[m];
    if (sl < 0 || sl >= max_sessions) { if (tid == 0) atomicOr(err, 1); return; }
    float a = speaker[(size_t)m * SPK + tid], c = speaker[(size_t)m * SPK + 256 + tid];
    const float nrm = fmaxf(sqrtf(block_sum(a * a + c * c, red)), 1e-12f);
    spk[(size_t)sl * SPK + tid] = a / nrm;
    spk[(size_t)sl * SPK + 256 + tid] = c / nrm;
    if (tid < NMEL) last[(size_t)sl * NMEL + tid] = 0.0f;
    if (tid == 0) {
        step[sl] = 0;
        int n = enc_len_in ? enc_len_in[m] : L;
        if (n < 1 || n > L || n > max_enc) { atomicOr(err, 8); n = min(max(n, 1), min(L, max_enc)); }
        enc_len[sl] = n;
    }
}

// xkv rows [r0, r0 + rows) of the flattened (session, position) grid -> the slots' cross-attention caches
template <typename KV>
__global__ void k_xkv_scatter(const float *__restrict__ xkv, const int32_t *__restrict__ slots, int r0, int rows, int L, KV *__restrict__ xcache,
                              size_t slot_stride, size_t layer_stride, int max_sessions) {
    const int r = blockIdx.x;
    if (r >= rows) return;
    const int g = r0 + r, m = g / L, j = g - m * L;
    const int sl = slots[m];
    if (sl < 0 || sl >= max_sessions) return;
    KV *dst = xcache + (size_t)sl * slot_stride + (size_t)j * (2 * H);                 // + layer * max_enc * 2H
    const float *src = xkv + (size_t)r * (NL * 2 * H);
    for (int c = threadIdx.x; c < NL * 2 * H; c += blockDim.x) st_kv(dst + (size_t)(c / (2 * H)) * layer_stride + (c % (2 * H)), src[c]);
}

__global__ void k_f32_to_bf16(const float *__restrict__ x, __nv_bfloat16 *__restrict__ y, size_t n) {
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) y[i] = __float2bfloat16_rn(x[i]);
}

// the prenet's dropout when the caller supplies no masks: Bernoulli(1/2) keep-mask per (call, step, layer, unit), shared by the batch like
// the reference's _consistent_dropout (:671-674), scaled by 1/(1-p) = 2.  Counter-based (splitmix64 of the coordinates): no state to carry.
__global__ void k_make_scales(const float *__restrict__ masks, unsigned long long seed, unsigned long long call, int nsteps, float *__restrict__ scales) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nsteps * 2 * PRE) return;
    float keep;
    if (masks) keep = masks[i];
    else {
        unsigned long long z = seed + 0x9E3779B97F4A7C15ull * (call * 0x10001ull + (unsigned long long)i + 1ull);
        z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
        z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
        z ^= z >> 31;
        keep = (z >> 63) ? 1.0f : 0.0f;
    }
    scales[i] = keep == 1.0f ? 2.0f : 0.0f;
}

}  // namespace

// ---------------------------------------------------------------------------------------------------- host side
struct b2_dec : b2::LinearOwner {
    b2_dec() { what = "decoder"; }
    int max_sessions = 0, max_rows = 0, max_steps = 0, max_enc = 0;
    bool finalized = false;
    DecLinear pre0, pre1, fin, spkl, qkv[NL], so[NL], xq[NL], xo[NL], ff1[NL], ff2[NL], xkv, outl;
    float *ln_w[NL][3] = {}, *ln_b[NL][3] = {};
    float *alpha = nullptr, *pe = nullptr;
    // slot state
    float *last = nullptr, *spk = nullptr;
    int32_t *step = nullptr, *enc_len = nullptr;
    void *self_cache = nullptr, *x_cache = nullptr;        // fp32 or bf16
    // per-call rows
    int32_t *rowpos = nullptr, *rowslot = nullptr;
    float *x0 = nullptr, *p1 = nullptr, *p2 = nullptr, *fin32 = nullptr, *cat = nullptr, *h = nullptr, *tmp = nullptr, *qkv32 = nullptr, *ctx = nullptr,
          *f1 = nullptr, *out = nullptr, *scales = nullptr, *xkv32 = nullptr;
    __nv_bfloat16 *x0b = nullptr, *p1b = nullptr, *p2b = nullptr, *catb = nullptr, *hb = nullptr, *ctxb = nullptr, *f1b = nullptr, *encb = nullptr;
    CUtensorMap tm_x0, tm_p1, tm_p2, tm_cat, tm_h, tm_ctx, tm_f1, tm_enc;
    int *err_h = nullptr, *err_d = nullptr;
    unsigned long long calls = 0;
    // one CUDA graph per (padded batch size, steps per call): a call is ~74 launches per step, 16 steps (b2_dec_steps); programmatic dependent
    // launch between the kernels of a step unless B2_DEC_PDL=0 (LinearOwner::use_pdl)
    bool use_graphs = true;
    std::map<unsigned long long, std::pair<cudaGraphExec_t, int>> graphs;    // key -> (exec, kernel nodes); exec == nullptr: seen once, run eagerly
    cudaStream_t g_stream = nullptr;           // captures run here: the caller's stream may be the legacy default stream, which cannot capture
    int32_t *g_slots = nullptr;
    float *g_mel = nullptr, *g_prob = nullptr;
    size_t g_cap_rows = 0;
};

namespace {

typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn g_enc = nullptr;

int get_encoder() {
    if (g_enc) return 0;
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
    if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) return set_error("cuTensorMapEncodeTiled is not available from the driver");
    g_enc = reinterpret_cast<EncodeTiledFn>(fn);
    return 0;
}

}  // namespace

namespace b2 {

int make_tma_2d_bf16(CUtensorMap *tm, const void *ptr, long long rows, int K, long long row_stride, int box_rows) {
    if (get_encoder()) return 1;
    cuuint64_t gdim[2] = {(cuuint64_t)K, (cuuint64_t)rows};
    cuuint64_t gstr[1] = {(cuuint64_t)row_stride * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = g_enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void *>(ptr), gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                       CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) return set_error("cuTensorMapEncodeTiled failed with CUresult %d (rows %lld K %d stride %lld)", (int)r, rows, K, row_stride);
    return 0;
}

static bool g_gemm_attr[64][5] = {};

// ring depth: deep (8 x 24 KB / 6 x 32 KB) when the K loop is long enough to use it, 4 otherwise (B2_GEMM_DEEP=0: always 4)
int gemm_tc_stages(int K, int nt) {
    static const bool deep_on = !(getenv("B2_GEMM_DEEP") && atoi(getenv("B2_GEMM_DEEP")) == 0);
    const bool deep = deep_on && K >= 512 && nt != 256;                 // 128 x 256 tiles: 4 x 48 KB is all the shared memory there is
    return deep ? (nt == 128 ? 6 : 8) : 4;
}

int launch_gemm_tc(const GemmTcArgs &a, cudaStream_t st) {
    if (a.M <= 0) return 0;
    if (!a.tmA || !a.tmB || !a.bias || (a.nt != 64 && a.nt != 128 && a.nt != 256) || a.N % a.nt || a.K % 64 || a.K < 64) return set_error("gemm_tc: bad arguments (N %d nt %d K %d)", a.N, a.nt, a.K);
    GemmParams p;
    p.bias = a.bias; p.colscale = a.colscale; p.out32 = a.out32; p.outb = a.outb; p.M = a.M; p.N = a.N; p.K = a.K; p.ldo = a.N; p.act = a.act;
    dim3 grid((unsigned)cdiv(a.M, 128), (unsigned)(a.N / a.nt));
    const int stages = gemm_tc_stages(a.K, a.nt);
    const bool deep = stages != 4;
    const int slot = a.nt == 256 ? 4 : (a.nt == 128 ? 1 : 0) + (deep ? 2 : 0);
    const size_t smem = (size_t)stages * (128 * 64 * 2 + (size_t)a.nt * 64 * 2) + (2 * stages + 1) * 8 + 16;
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 64 && !g_gemm_attr[dev][slot]) {
        if (a.nt == 256) B2_CUDA_OK(cudaFuncSetAttribute(k_gemm_tc<256, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        else if (a.nt == 128) B2_CUDA_OK(deep ? cudaFuncSetAttribute(k_gemm_tc<128, 6>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                                         : cudaFuncSetAttribute(k_gemm_tc<128, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        else B2_CUDA_OK(deep ? cudaFuncSetAttribute(k_gemm_tc<64, 8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                             : cudaFuncSetAttribute(k_gemm_tc<64, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        g_gemm_attr[dev][slot] = true;
    }
    const GemmParams cp = p;
    if (a.nt == 256) {
        B2_CUDA_OK(launch_k(k_gemm_tc<256, 4>, grid, dim3(192), smem, st, a.pdl, *a.tmA, *a.tmB, cp));
    } else if (a.nt == 128) {
        if (deep) B2_CUDA_OK(launch_k(k_gemm_tc<128, 6>, grid, dim3(192), smem, st, a.pdl, *a.tmA, *a.tmB, cp));
        else B2_CUDA_OK(launch_k(k_gemm_tc<128, 4>, grid, dim3(192), smem, st, a.pdl, *a.tmA, *a.tmB, cp));
    } else {
        if (deep) B2_CUDA_OK(launch_k(k_gemm_tc<64, 8>, grid, dim3(192), smem, st, a.pdl, *a.tmA, *a.tmB, cp));
        else B2_CUDA_OK(launch_k(k_gemm_tc<64, 4>, grid, dim3(192), smem, st, a.pdl, *a.tmA, *a.tmB, cp));
    }
    B2_LAUNCH_OK("k_gemm_tc");
    return 0;
}

}  // namespace b2

namespace {

int finalize_dec(b2_dec *d) {
    const bool bf = d->mode == B2_MODE_BF16;
    if (bf && get_encoder()) return 1;
    const std::string P = "speecht5.decoder.prenet.", Dp = "speecht5.decoder.wrapped_decoder.layers.";
    if (pack_one(d, d->pre0, P + "layers.0", PRE, NMEL, bf ? 128 : NMEL, PRE)) return 1;
    if (pack_one(d, d->pre1, P + "layers.1", PRE, PRE, PRE, PRE)) return 1;
    if (pack_one(d, d->fin, P + "final_layer", H, PRE, PRE, H)) return 1;
    if (pack_one(d, d->spkl, P + "speaker_embeds_layer", H, H + SPK, H + SPK, H)) return 1;
    const HostTensor *t;
    if (!(t = need(d, P + "encode_positions.alpha", {}))) { if (!(t = need(d, P + "encode_positions.alpha", {1}))) return 1; }
    if (upload_vec(d, &d->alpha, *t)) return 1;
    if (!(t = need(d, "pe", {(int64_t)d->max_steps, H}))) return 1;
    if (upload_vec(d, &d->pe, *t)) return 1;
    std::vector<float> XW((size_t)NL * 2 * H * H, 0.0f), XB((size_t)NL * 2 * H, 0.0f);
    for (int i = 0; i < NL; i++) {
        const std::string L = Dp + std::to_string(i) + ".";
        {   // q (pre-scaled by 1/sqrt(64): exact, a power of two) | k | v in one N = 2304 projection
            std::vector<float> W((size_t)3 * H * H, 0.0f), B((size_t)3 * H, 0.0f);
            const char *nm[3] = {"q_proj", "k_proj", "v_proj"};
            for (int j = 0; j < 3; j++) {
                const HostTensor *w = need(d, L + "self_attn." + nm[j] + ".weight", {H, H}), *b = need(d, L + "self_attn." + nm[j] + ".bias", {H});
                if (!w || !b) return 1;
                fill_linear(W, B, H, 3 * H, j * H, *w, *b, j == 0 ? 0.125f : 1.0f);
            }
            if (upload_linear(d, d->qkv[i], H, 3 * H, W, B)) return 1;
        }
        if (pack_one(d, d->so[i], L + "self_attn.out_proj", H, H, H, H)) return 1;
        if (pack_one(d, d->xq[i], L + "encoder_attn.q_proj", H, H, H, H, 0.125f)) return 1;
        if (pack_one(d, d->xo[i], L + "encoder_attn.out_proj", H, H, H, H)) return 1;
        if (pack_one(d, d->ff1[i], L + "feed_forward.intermediate_dense", FFN, H, H, FFN)) return 1;
        if (pack_one(d, d->ff2[i], L + "feed_forward.output_dense", H, FFN, FFN, H)) return 1;
        const char *kv[2] = {"k_proj", "v_proj"};
        for (int j = 0; j < 2; j++) {
            const HostTensor *w = need(d, L + "encoder_attn." + kv[j] + ".weight", {H, H}), *b = need(d, L + "encoder_attn." + kv[j] + ".bias", {H});
            if (!w || !b) return 1;
            fill_linear(XW, XB, H, NL * 2 * H, (i * 2 + j) * H, *w, *b, 1.0f);
        }
        const char *ln[3] = {"self_attn_layer_norm", "encoder_attn_layer_norm", "final_layer_norm"};
        for (int j = 0; j < 3; j++) {
            const HostTensor *w = need(d, L + ln[j] + ".weight", {H}), *b = need(d, L + ln[j] + ".bias", {H});
            if (!w || !b) return 1;
            if (upload_vec(d, &d->ln_w[i][j], *w) || upload_vec(d, &d->ln_b[i][j], *b)) return 1;
        }
    }
    if (upload_linear(d, d->xkv, H, NL * 2 * H, XW, XB)) return 1;
    {
        const HostTensor *fw = need(d, "speech_decoder_postnet.feat_out.weight", {2 * NMEL, H}), *fb = need(d, "speech_decoder_postnet.feat_out.bias", {2 * NMEL});
        const HostTensor *pw = need(d, "speech_decoder_postnet.prob_out.weight", {2, H}), *pb = need(d, "speech_decoder_postnet.prob_out.bias", {2});
        if (!fw || !fb || !pw || !pb) return 1;
        std::vector<float> W((size_t)OUTP * H, 0.0f), B((size_t)OUTP, 0.0f);
        fill_linear(W, B, H, OUTP, 0, *fw, *fb, 1.0f);
        fill_linear(W, B, H, OUTP, 2 * NMEL, *pw, *pb, 1.0f);
        if (upload_linear(d, d->outl, H, OUTP, W, B)) return 1;
    }
    // slot state
    const size_t S = (size_t)d->max_sessions + 1, R = (size_t)d->max_rows;          // + the scratch slot bad ids are redirected to
    if (dalloc(d, &d->last, S * NMEL) || dalloc(d, &d->spk, S * SPK) || dalloc(d, &d->step, S) || dalloc(d, &d->enc_len, S)) return 1;
    const size_t self_n = S * NL * (size_t)d->max_steps * 2 * H, x_n = S * (size_t)d->max_enc * NL * 2 * H;
    if (bf) {
        __nv_bfloat16 *a = nullptr, *b = nullptr;
        if (dalloc(d, &a, self_n) || dalloc(d, &b, x_n)) return 1;
        d->self_cache = a; d->x_cache = b;
    } else {
        float *a = nullptr, *b = nullptr;
        if (dalloc(d, &a, self_n) || dalloc(d, &b, x_n)) return 1;
        d->self_cache = a; d->x_cache = b;
    }
    // per-call rows
    if (dalloc(d, &d->rowpos, R) || dalloc(d, &d->rowslot, R) || dalloc(d, &d->fin32, R * H) || dalloc(d, &d->h, R * H) || dalloc(d, &d->tmp, R * H) || dalloc(d, &d->qkv32, R * 3 * H) ||
        dalloc(d, &d->out, R * OUTP) || dalloc(d, &d->scales, (size_t)64 * 2 * PRE) || dalloc(d, &d->xkv32, R * NL * 2 * H)) return 1;
    if (bf) {
        if (dalloc(d, &d->x0b, R * 128) || dalloc(d, &d->p1b, R * PRE) || dalloc(d, &d->p2b, R * PRE) || dalloc(d, &d->catb, R * (H + SPK)) ||
            dalloc(d, &d->hb, R * H) || dalloc(d, &d->ctxb, R * H) || dalloc(d, &d->f1b, R * FFN) || dalloc(d, &d->encb, R * H)) return 1;
        const int Ri = (int)R;
        if (make_map(&d->tm_x0, d->x0b, Ri, 128, 128) || make_map(&d->tm_p1, d->p1b, Ri, PRE, 128) || make_map(&d->tm_p2, d->p2b, Ri, PRE, 128) ||
            make_map(&d->tm_cat, d->catb, Ri, H + SPK, 128) || make_map(&d->tm_h, d->hb, Ri, H, 128) || make_map(&d->tm_ctx, d->ctxb, Ri, H, 128) ||
            make_map(&d->tm_f1, d->f1b, Ri, FFN, 128) || make_map(&d->tm_enc, d->encb, Ri, H, 128)) return 1;
    } else {
        if (dalloc(d, &d->x0, R * NMEL) || dalloc(d, &d->p1, R * PRE) || dalloc(d, &d->p2, R * PRE) || dalloc(d, &d->cat, R * (H + SPK)) ||
            dalloc(d, &d->ctx, R * H) || dalloc(d, &d->f1, R * FFN)) return 1;
    }
    B2_CUDA_OK(cudaHostAlloc((void **)&d->err_h, sizeof(int), cudaHostAllocMapped));
    *d->err_h = 0;
    B2_CUDA_OK(cudaHostGetDevicePointer((void **)&d->err_d, d->err_h, 0));
    d->raw.clear();
    d->finalized = true;
    return 0;
}

int poll_dec_errors(b2_dec *d, const char *who) {
    if (!d->err_h) return 0;
    const int f = *(volatile int *)d->err_h;
    if (!f) return 0;
    *(volatile int *)d->err_h = 0;
    return set_error("%s: an earlier decoder call on this handle failed on the device:%s%s%s", who, (f & 1) ? " slot id outside the pool;" : "",
                     (f & 4) ? " a session ran past max_steps (its step was clamped);" : "", (f & 8) ? " encoder length outside [1, min(L, max_enc_len)];" : "");
}

template <typename KV>
int steps_impl(b2_dec *d, const int32_t *d_slots, int n, int nsteps, float *d_mel, float *d_prob, cudaStream_t st) {
    const bool bf = d->mode == B2_MODE_BF16;
    KV *self_cache = reinterpret_cast<KV *>(d->self_cache), *x_cache = reinterpret_cast<KV *>(d->x_cache);
    const size_t self_slot = (size_t)NL * d->max_steps * 2 * H, self_pos = 2 * H;
    const size_t x_slot = (size_t)NL * d->max_enc * 2 * H, x_pos = 2 * H;            // [slot][layer][pos][K | V], like the self-attention cache
    const size_t attn_smem_self = ((size_t)((d->max_steps + 3) & ~3) + HD + 4 * HD + 8) * sizeof(float);
    const size_t attn_smem_x = ((size_t)((d->max_enc + 3) & ~3) + HD + 4 * HD + 8) * sizeof(float);
    if (attn_smem_self > 200 * 1024 || attn_smem_x > 200 * 1024) return set_error("decoder: max_steps / max_enc_len too large for the attention kernel");
    static bool attr_done[64][2] = {};
    if (d->device < 64 && !attr_done[d->device][bf ? 1 : 0]) {
        B2_CUDA_OK(cudaFuncSetAttribute(k_attend<KV, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        B2_CUDA_OK(cudaFuncSetAttribute(k_attend<KV, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
        attr_done[d->device][bf ? 1 : 0] = true;
    }
    for (int r0 = 0; r0 < n; r0 += d->max_rows) {
        const int M = std::min(d->max_rows, n - r0);
        const int32_t *slots = d->rowslot;               // sanitised by k_dec_gather at the top of every step
        float *mel = d_mel + (size_t)r0 * 2 * nsteps * NMEL, *prob = d_prob + (size_t)r0 * nsteps * 2;
        for (int s = 0; s < nsteps; s++) {
            const float *sc0 = d->scales + (size_t)(s * 2) * PRE, *sc1 = sc0 + PRE;
            const bool pdl = d->use_pdl;
            const dim3 gM((unsigned)M);
            if (bf) B2_CUDA_OK(launch_k(k_dec_gather<true>, gM, dim3(128), 0, st, pdl, d_slots + r0, (const float *)d->last, (const int32_t *)d->step, M, (float *)nullptr, d->x0b, d->rowpos, d->rowslot, d->max_sessions, d->max_steps, d->err_d));
            else B2_CUDA_OK(launch_k(k_dec_gather<false>, gM, dim3(128), 0, st, pdl, d_slots + r0, (const float *)d->last, (const int32_t *)d->step, M, d->x0, (__nv_bfloat16 *)nullptr, d->rowpos, d->rowslot, d->max_sessions, d->max_steps, d->err_d));
            B2_LAUNCH_OK("k_dec_gather");
            // prenet (:689-692)
            if (linear(d, d->pre0, d->x0, &d->tm_x0, M, 1, sc0, bf ? nullptr : d->p1, bf ? d->p1b : nullptr, st)) return 1;
            if (linear(d, d->pre1, d->p1, &d->tm_p1, M, 1, sc1, bf ? nullptr : d->p2, bf ? d->p2b : nullptr, st)) return 1;
            if (linear(d, d->fin, d->p2, &d->tm_p2, M, 0, nullptr, d->fin32, nullptr, st)) return 1;
            if (bf) B2_CUDA_OK(launch_k(k_pos_cat<true>, gM, dim3(256), 0, st, pdl, (const float *)d->fin32, (const float *)d->pe, (const float *)d->alpha, (const int32_t *)d->rowpos, slots, (const float *)d->spk, M, (float *)nullptr, d->catb));
            else B2_CUDA_OK(launch_k(k_pos_cat<false>, gM, dim3(256), 0, st, pdl, (const float *)d->fin32, (const float *)d->pe, (const float *)d->alpha, (const int32_t *)d->rowpos, slots, (const float *)d->spk, M, d->cat, (__nv_bfloat16 *)nullptr));
            B2_LAUNCH_OK("k_pos_cat");
            if (linear(d, d->spkl, d->cat, &d->tm_cat, M, 0, nullptr, d->tmp, nullptr, st)) return 1;
            {
                const size_t ne = (size_t)M * H;
                B2_CUDA_OK(launch_k(k_relu_dual, dim3((unsigned)std::min<size_t>((ne + 255) / 256, (size_t)sm_count() * 8)), dim3(256), 0, st, pdl, (const float *)d->tmp, d->h, bf ? d->hb : (__nv_bfloat16 *)nullptr, ne));
                B2_LAUNCH_OK("k_relu_dual");
            }
            for (int i = 0; i < NL; i++) {
                // self-attention (:1125-1134)
                if (linear(d, d->qkv[i], d->h, &d->tm_h, M, 0, nullptr, d->qkv32, nullptr, st)) return 1;
                B2_CUDA_OK(launch_k(k_attend<KV, true>, dim3((unsigned)M, NH), dim3(128), attn_smem_self, st, pdl, (const float *)d->qkv32, 3 * H, slots, (const int32_t *)d->rowpos,
                                    (const int32_t *)d->enc_len, self_cache, self_slot, self_pos, (size_t)i * d->max_steps * 2 * H, bf ? (float *)nullptr : d->ctx,
                                    bf ? d->ctxb : (__nv_bfloat16 *)nullptr));
                B2_LAUNCH_OK("k_attend(self)");
                if (linear(d, d->so[i], d->ctx, &d->tm_ctx, M, 0, nullptr, d->tmp, nullptr, st)) return 1;
                B2_CUDA_OK(launch_k(k_add_ln, gM, dim3(256), 0, st, pdl, d->h, (const float *)d->tmp, (const float *)d->ln_w[i][0], (const float *)d->ln_b[i][0], bf ? d->hb : (__nv_bfloat16 *)nullptr, M));
                B2_LAUNCH_OK("k_add_ln");
                // cross-attention (:1137-1147)
                if (linear(d, d->xq[i], d->h, &d->tm_h, M, 0, nullptr, d->qkv32, nullptr, st)) return 1;
                B2_CUDA_OK(launch_k(k_attend<KV, false>, dim3((unsigned)M, NH), dim3(128), attn_smem_x, st, pdl, (const float *)d->qkv32, H, slots, (const int32_t *)d->rowpos,
                                    (const int32_t *)d->enc_len, x_cache, x_slot, x_pos, (size_t)i * d->max_enc * 2 * H, bf ? (float *)nullptr : d->ctx,
                                    bf ? d->ctxb : (__nv_bfloat16 *)nullptr));
                B2_LAUNCH_OK("k_attend(cross)");
                if (linear(d, d->xo[i], d->ctx, &d->tm_ctx, M, 0, nullptr, d->tmp, nullptr, st)) return 1;
                B2_CUDA_OK(launch_k(k_add_ln, gM, dim3(256), 0, st, pdl, d->h, (const float *)d->tmp, (const float *)d->ln_w[i][1], (const float *)d->ln_b[i][1], bf ? d->hb : (__nv_bfloat16 *)nullptr, M));
                B2_LAUNCH_OK("k_add_ln");
                // feed-forward (:1150-1151)
                if (linear(d, d->ff1[i], d->h, &d->tm_h, M, 2, nullptr, bf ? nullptr : d->f1, bf ? d->f1b : nullptr, st)) return 1;
                if (linear(d, d->ff2[i], d->f1, &d->tm_f1, M, 0, nullptr, d->tmp, nullptr, st)) return 1;
                B2_CUDA_OK(launch_k(k_add_ln, gM, dim3(256), 0, st, pdl, d->h, (const float *)d->tmp, (const float *)d->ln_w[i][2], (const float *)d->ln_b[i][2], bf ? d->hb : (__nv_bfloat16 *)nullptr, M));
                B2_LAUNCH_OK("k_add_ln");
            }
            if (linear(d, d->outl, d->h, &d->tm_h, M, 0, nullptr, d->out, nullptr, st)) return 1;
            B2_CUDA_OK(launch_k(k_dec_finish, gM, dim3(OUTP), 0, st, pdl, (const float *)d->out, slots, M, s, nsteps, mel, prob, d->last, d->step, d->max_sessions));
            B2_LAUNCH_OK("k_dec_finish");
        }
    }
    return 0;
}

template <typename KV>
int start_impl(b2_dec *d, const int32_t *d_slots, const float *d_enc, int n, int L, cudaStream_t st) {
    const bool bf = d->mode == B2_MODE_BF16;
    KV *x_cache = reinterpret_cast<KV *>(d->x_cache);
    const size_t x_slot = (size_t)NL * d->max_enc * 2 * H, x_layer = (size_t)d->max_enc * 2 * H;
    const long long rows_total = (long long)n * L;
    for (long long r0 = 0; r0 < rows_total; r0 += d->max_rows) {
        const int rows = (int)std::min<long long>(d->max_rows, rows_total - r0);
        const float *A = d_enc + (size_t)r0 * H;
        if (bf) {
            const size_t ne = (size_t)rows * H;
            k_f32_to_bf16<<<(unsigned)std::min<size_t>((ne + 255) / 256, (size_t)sm_count() * 8), 256, 0, st>>>(A, d->encb, ne);
            B2_LAUNCH_OK("k_f32_to_bf16");
        }
        if (linear(d, d->xkv, A, &d->tm_enc, rows, 0, nullptr, d->xkv32, nullptr, st)) return 1;
        k_xkv_scatter<KV><<<rows, 256, 0, st>>>(d->xkv32, d_slots, (int)r0, rows, L, x_cache, x_slot, x_layer, d->max_sessions);
        B2_LAUNCH_OK("k_xkv_scatter");
    }
    return 0;
}

}  // namespace

#define DEC_GUARD(d)                                                                                  \
    if (!(d)) return set_error("null decoder handle");                                                \
    {                                                                                                 \
        cudaError_t _e = cudaSetDevice((d)->device);                                                  \
        if (_e != cudaSuccess) return set_error("cudaSetDevice(%d): %s", (d)->device, cudaGetErrorString(_e)); \
    }

void b2::dec_limits(const b2_dec *d, int *max_sessions, int *max_steps, int *max_enc_len) {
    *max_sessions = d->max_sessions; *max_steps = d->max_steps; *max_enc_len = d->max_enc;
}

extern "C" {

b2_dec *b2_dec_create(int device, int mode, int max_sessions, int max_rows, int max_steps, int max_enc_len) {
    if (mode != B2_MODE_FP32 && mode != B2_MODE_BF16) { set_error("b2_dec_create: mode must be B2_MODE_FP32 or B2_MODE_BF16"); return nullptr; }
    if (max_sessions < 1 || max_rows < 1 || max_steps < 1 || max_enc_len < 1) { set_error("b2_dec_create: sizes must be >= 1"); return nullptr; }
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) { set_error("no CUDA device: %s (this library has no CPU fallback)", cudaGetErrorString(e)); return nullptr; }
    if (device < 0 || device >= ndev) { set_error("device %d out of range (%d devices)", device, ndev); return nullptr; }
    cudaDeviceProp prop;
    cudaGetDeviceProperties(&prop, device);
    if (prop.major != 10) { set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major, prop.minor); return nullptr; }
    b2_dec *d = new b2_dec();
    d->device = device; d->mode = mode; d->max_sessions = max_sessions; d->max_rows = max_rows; d->max_steps = max_steps; d->max_enc = max_enc_len;
    d->use_pdl = pdl_enabled() && !(getenv("B2_DEC_PDL") && atoi(getenv("B2_DEC_PDL")) == 0);
    return d;
}

void b2_dec_destroy(b2_dec *d) {
    if (!d) return;
    cudaSetDevice(d->device);
    cudaDeviceSynchronize();
    for (auto &kv : d->graphs) if (kv.second.first) cudaGraphExecDestroy(kv.second.first);
    if (d->g_stream) cudaStreamDestroy(d->g_stream);
    for (void *p : d->allocs) cudaFree(p);
    if (d->err_h) cudaFreeHost(d->err_h);
    delete d;
}

size_t b2_dec_device_bytes(const b2_dec *d) { return d ? d->device_bytes : 0; }

int b2_dec_load_tensor(b2_dec *d, const char *key, const float *h, const int64_t *shape, int ndim) {
    if (!d) return set_error("null decoder handle");
    if (d->finalized) return set_error("decoder weights are already finalized");
    if (!key || !h || ndim < 0 || ndim > 4 || (ndim > 0 && !shape)) return set_error("b2_dec_load_tensor: bad arguments");
    HostTensor t;
    size_t n = 1;
    for (int i = 0; i < ndim; i++) { t.shape.push_back(shape[i]); n *= (size_t)shape[i]; }
    t.data.assign(h, h + n);
    d->raw[key] = std::move(t);
    return 0;
}

int b2_dec_finalize(b2_dec *d) {
    DEC_GUARD(d);
    if (d->finalized) return set_error("decoder weights are already finalized");
    return finalize_dec(d);
}

int b2_dec_start(b2_dec *d, const int32_t *d_slots, const float *d_enc, const int32_t *d_enc_len, const float *d_speaker, int n, int L, void *stream) {
    DEC_GUARD(d);
    if (!d->finalized) return set_error("b2_dec_finalize has not been called");
    if (n < 0 || L < 1) return set_error("b2_dec_start: bad shape n=%d L=%d", n, L);
    if (L > d->max_enc) return set_error("b2_dec_start: %d encoder positions exceed max_enc_len=%d", L, d->max_enc);
    if (n == 0) return 0;
    if (!d_slots || !d_enc || !d_speaker) return set_error("b2_dec_start: null pointer");
    if (poll_dec_errors(d, "b2_dec_start")) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    k_dec_init<<<n, 256, 0, st>>>(d_slots, d_speaker, d_enc_len, L, d->max_enc, d->last, d->step, d->spk, d->enc_len, d->max_sessions, d->err_d);
    B2_LAUNCH_OK("k_dec_init");
    return d->mode == B2_MODE_BF16 ? start_impl<__nv_bfloat16>(d, d_slots, d_enc, n, L, st) : start_impl<float>(d, d_slots, d_enc, n, L, st);
}

int b2_dec_steps(b2_dec *d, const int32_t *d_slots, int n, int nsteps, const float *d_masks, uint64_t seed, float *d_mel, float *d_prob, void *stream) {
    DEC_GUARD(d);
    if (!d->finalized) return set_error("b2_dec_finalize has not been called");
    if (n < 0 || nsteps < 1 || nsteps > 64) return set_error("b2_dec_steps: bad arguments n=%d nsteps=%d (1..64)", n, nsteps);
    if (n == 0) return 0;
    if (!d_slots || !d_mel || !d_prob) return set_error("b2_dec_steps: null pointer");
    if (poll_dec_errors(d, "b2_dec_steps")) return 1;
    cudaStream_t st = (cudaStream_t)stream;
    k_make_scales<<<cdiv(nsteps * 2 * PRE, 256), 256, 0, st>>>(d_masks, (unsigned long long)seed, d->calls++, nsteps, d->scales);
    B2_LAUNCH_OK("k_make_scales");
    auto run = [&](const int32_t *sl, int rows, float *mel, float *prob) {
        return d->mode == B2_MODE_BF16 ? steps_impl<__nv_bfloat16>(d, sl, rows, nsteps, mel, prob, st) : steps_impl<float>(d, sl, rows, nsteps, mel, prob, st);
    };
    if (!d->use_graphs) return run(d_slots, n, d_mel, d_prob);
    // Graph path.  The batch is padded to a bucket size with rows on the scratch slot (id -1) so that a few graphs cover every batch size;
    // slots and outputs go through fixed staging buffers (a graph replays fixed addresses).  A (bucket, nsteps) pair runs eagerly the first
    // time it is seen (every kernel sets its attributes outside a capture) and is captured on its second use.
    const int nb = n <= 64 ? ((n + 7) / 8) * 8 : n <= 512 ? ((n + 31) / 32) * 32 : ((n + 127) / 128) * 128;
    if ((size_t)nb > d->g_cap_rows) {
        B2_CUDA_OK(cudaStreamSynchronize(st));
        for (auto &kv : d->graphs) if (kv.second.first) cudaGraphExecDestroy(kv.second.first);
        d->graphs.clear();                                   // they point into the old staging buffers
        const size_t cap = std::max<size_t>((size_t)nb, std::min<size_t>((size_t)d->max_sessions + 128, d->g_cap_rows * 2));
        if (dalloc(d, &d->g_slots, cap) || dalloc(d, &d->g_mel, cap * 2 * 64 * NMEL) || dalloc(d, &d->g_prob, cap * 64 * 2)) return 1;
        d->g_cap_rows = cap;
    }
    const unsigned long long key = ((unsigned long long)nb << 8) | (unsigned long long)nsteps;
    B2_CUDA_OK(cudaMemsetAsync(d->g_slots, 0xFF, (size_t)nb * sizeof(int32_t), st));          // -1 = padding row
    B2_CUDA_OK(cudaMemcpyAsync(d->g_slots, d_slots, (size_t)n * sizeof(int32_t), cudaMemcpyDeviceToDevice, st));
    auto it = d->graphs.find(key);
    if (it == d->graphs.end()) {
        d->graphs.emplace(key, std::make_pair((cudaGraphExec_t) nullptr, 0));
        if (run(d->g_slots, nb, d->g_mel, d->g_prob)) return 1;
    } else {
        if (!it->second.first) {
            cudaGraph_t g = nullptr;
            cudaGraphExec_t ge = nullptr;
            const uint64_t l0 = g_launches.load();
            if (!d->g_stream) B2_CUDA_OK(cudaStreamCreateWithFlags(&d->g_stream, cudaStreamNonBlocking));
            cudaStream_t cs = d->g_stream;
            auto run_on = [&](cudaStream_t s2) {
                return d->mode == B2_MODE_BF16 ? steps_impl<__nv_bfloat16>(d, d->g_slots, nb, nsteps, d->g_mel, d->g_prob, s2)
                                               : steps_impl<float>(d, d->g_slots, nb, nsteps, d->g_mel, d->g_prob, s2);
            };
            B2_CUDA_OK(cudaStreamBeginCapture(cs, cudaStreamCaptureModeRelaxed));
            const int rc = run_on(cs);
            cudaError_t e = cudaStreamEndCapture(cs, &g);
            if (rc) { if (g) cudaGraphDestroy(g); return 1; }
            if (e != cudaSuccess) return set_error("b2_dec_steps: cudaStreamEndCapture: %s", cudaGetErrorString(e));
            e = cudaGraphInstantiate(&ge, g, 0);
            cudaGraphDestroy(g);
            if (e != cudaSuccess) return set_error("b2_dec_steps: cudaGraphInstantiate: %s", cudaGetErrorString(e));
            const int nk = (int)(g_launches.load() - l0);
            g_launches.fetch_sub((uint64_t)nk);
            it->second = std::make_pair(ge, nk);
        }
        B2_CUDA_OK(cudaGraphLaunch(it->second.first, st));
        count_launch(it->second.second);
    }
    B2_CUDA_OK(cudaMemcpyAsync(d_mel, d->g_mel, (size_t)n * 2 * nsteps * NMEL * sizeof(float), cudaMemcpyDeviceToDevice, st));
    B2_CUDA_OK(cudaMemcpyAsync(d_prob, d->g_prob, (size_t)n * nsteps * 2 * sizeof(float), cudaMemcpyDeviceToDevice, st));
    return 0;
}

int b2_dec_set_graphs(b2_dec *d, int on) {
    if (!d) return set_error("null decoder handle");
    d->use_graphs = on != 0;
    return 0;
}

int b2_dec_poll_errors(b2_dec *d, void *stream) {
    DEC_GUARD(d);
    B2_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    return poll_dec_errors(d, "b2_dec_poll_errors");
}

int b2_dec_get_step(b2_dec *d, int slot, int32_t *h_step, void *stream) {
    DEC_GUARD(d);
    if (!d->finalized || slot < 0 || slot >= d->max_sessions || !h_step) return set_error("b2_dec_get_step: bad arguments");
    B2_CUDA_OK(cudaMemcpyAsync(h_step, d->step + slot, sizeof(int32_t), cudaMemcpyDeviceToHost, (cudaStream_t)stream));
    B2_CUDA_OK(cudaStreamSynchronize((cudaStream_t)stream));
    return 0;
}

int b2_linear(int device, int mode, const void *d_in, int M, int a_rows, const float *h_weight, const float *h_bias, int N, int K, int act,
              const float *d_colscale, float *d_out32, void *d_outb, int *h_launched, void *stream) {
    if (mode != B2_MODE_FP32 && mode != B2_MODE_BF16) return set_error("b2_linear: mode must be B2_MODE_FP32 or B2_MODE_BF16");
    if (M < 0 || a_rows < M || K < 64 || K % 64 || N < 64 || N % 64 || act < 0 || act > 2)
        return set_error("b2_linear: bad arguments (M %d a_rows %d N %d K %d act %d; need a_rows >= M, K and N multiples of 64, act 0..2)", M, a_rows, N, K, act);
    if (mode == B2_MODE_FP32 && (d_outb || !d_out32)) return set_error("b2_linear: fp32 mode writes d_out32 only");
    if (h_launched) h_launched[0] = h_launched[1] = 0;
    if (M == 0) return 0;
    if (!d_in || !h_weight || !h_bias || (!d_out32 && !d_outb)) return set_error("b2_linear: null pointer");
    B2_CUDA_OK(cudaSetDevice(device));
    cudaStream_t st = (cudaStream_t)stream;
    LinearOwner o;
    o.what = "b2_linear"; o.device = device; o.mode = mode; o.use_pdl = pdl_enabled();
    DecLinear l;
    std::vector<float> W(h_weight, h_weight + (size_t)N * K), B(h_bias, h_bias + N);
    CUtensorMap tmA;
    int rc = mode == B2_MODE_BF16 ? get_encoder() : 0;
    if (!rc) rc = upload_linear(&o, l, K, N, W, B);
    if (!rc && mode == B2_MODE_BF16) rc = make_map(&tmA, d_in, a_rows, K, 128);
    if (!rc) rc = linear(&o, l, static_cast<const float *>(d_in), &tmA, M, act, d_colscale, d_out32, static_cast<__nv_bfloat16 *>(d_outb), st);
    const cudaError_t e = cudaStreamSynchronize(st);
    if (!rc && e != cudaSuccess) rc = set_error("b2_linear: %s", cudaGetErrorString(e));
    if (!rc && h_launched && mode == B2_MODE_BF16) {
        h_launched[0] = gemm_tile_n(l, M);
        h_launched[1] = gemm_tc_stages(K, h_launched[0]);
    }
    for (void *p : o.allocs) cudaFree(p);
    return rc;
}

}  // extern "C"
