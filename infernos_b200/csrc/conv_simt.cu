// fp32 CUDA-core kernels of the TTS tail (see conv_simt.cuh).  Restates, never copies:
//   transformers SpeechT5HifiGan.forward / HifiGanResidualBlock.forward (modeling_speecht5.py:2954-2962, 3055-3085)
//   AmendmentNetwork1.forward (HelloSippyTTSRT/HelloSippyRT.py:219-237)
//   window builder (HelloSippyTTSRT/HelloSippyRTPipe.py:231-235)
#include "conv_simt.cuh"
#include <algorithm>

namespace b2 {

__device__ __forceinline__ float lrelu(float v, float slope) { return v > 0.0f ? v : v * slope; }

// ---------------------------------------------------------------------------------------------------
// generic conv1d as a tiled SGEMM: M = W*Tout flattened rows, N = Cout, K = taps*Cin.
// CTA tile 128 x BN, 256 threads, 8 x (BN/16) outputs per thread, K chunk 16.
// ---------------------------------------------------------------------------------------------------
template <int BN>
__global__ void __launch_bounds__(256) k_conv_simt(ConvArgs a) {
    constexpr int BM = 128, KC = 16, TN = BN / 16;
    __shared__ __align__(16) float As[KC][BM];
    __shared__ __align__(16) float Bs[KC][BN];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const long long M = (long long)a.W * a.Tout;
    const long long m0 = (long long)blockIdx.x * BM;
    const int n0 = blockIdx.y * BN;

    // the row this thread loads for the A tile
    const int lrow = tid & 127;
    const int lc4 = tid >> 7;                     // 0..1 (+2 on the second pass)
    const long long lr = m0 + lrow;
    const bool lvalid = lr < M;
    const int lw = lvalid ? (int)(lr / a.Tout) : 0;
    const int lt = lvalid ? (int)(lr - (long long)lw * a.Tout) : 0;
    const float *in_w = a.in + (long long)lw * a.Tin * a.Cin;

    float acc[8][TN];
#pragma unroll
    for (int i = 0; i < 8; i++)
#pragma unroll
        for (int e = 0; e < TN; e++) acc[i][e] = 0.0f;

    for (int j = 0; j < a.taps; j++) {
        const int tin = lt * a.stride + j * a.dil - a.pad;
        const bool rvalid = lvalid && tin >= 0 && tin < a.Tin;
        const float *in_row = in_w + (long long)tin * a.Cin;
        const float *w_tap = a.wt + (long long)j * a.Cin * a.Cout;
        for (int c0 = 0; c0 < a.Cin; c0 += KC) {
#pragma unroll
            for (int q = 0; q < 2; q++) {
                const int c = c0 + (lc4 + 2 * q) * 4;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (rvalid && c < a.Cin) v = __ldg(reinterpret_cast<const float4 *>(in_row + c));
                const int cc = (lc4 + 2 * q) * 4;
                As[cc + 0][lrow] = lrelu(v.x, a.pre_slope);
                As[cc + 1][lrow] = lrelu(v.y, a.pre_slope);
                As[cc + 2][lrow] = lrelu(v.z, a.pre_slope);
                As[cc + 3][lrow] = lrelu(v.w, a.pre_slope);
            }
            if (BN == 64 || tid < 128) {
                constexpr int N4 = BN / 4;
                const int kk = tid / N4, n4 = tid % N4;
                float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
                if (c0 + kk < a.Cin && n0 + n4 * 4 < a.Cout)
                    v = __ldg(reinterpret_cast<const float4 *>(w_tap + (long long)(c0 + kk) * a.Cout + n0 + n4 * 4));
                *reinterpret_cast<float4 *>(&Bs[kk][n4 * 4]) = v;
            }
            __syncthreads();
#pragma unroll
            for (int kk = 0; kk < KC; kk++) {
                const float4 a0 = *reinterpret_cast<const float4 *>(&As[kk][ty * 8]);
                const float4 a1 = *reinterpret_cast<const float4 *>(&As[kk][ty * 8 + 4]);
                const float av[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
                float bv[TN];
                if constexpr (TN == 4) {
                    const float4 b = *reinterpret_cast<const float4 *>(&Bs[kk][tx * 4]);
                    bv[0] = b.x; bv[1] = b.y; bv[2] = b.z; bv[3] = b.w;
                } else {
                    const float2 b = *reinterpret_cast<const float2 *>(&Bs[kk][tx * 2]);
                    bv[0] = b.x; bv[1] = b.y;
                }
#pragma unroll
                for (int i = 0; i < 8; i++)
#pragma unroll
                    for (int e = 0; e < TN; e++) acc[i][e] = fmaf(av[i], bv[e], acc[i][e]);
            }
            __syncthreads();
        }
    }

    const int col = n0 + tx * TN;
    if (col >= a.Cout) return;
    float bias[TN];
#pragma unroll
    for (int e = 0; e < TN; e++) bias[e] = a.bias ? __ldg(a.bias + col + e) : 0.0f;
#pragma unroll
    for (int i = 0; i < 8; i++) {
        const long long r = m0 + ty * 8 + i;
        if (r >= M) continue;
        const long long o = r * a.Cout + col;
        float v[TN];
#pragma unroll
        for (int e = 0; e < TN; e++) v[e] = acc[i][e] + bias[e];
        if (a.residual) {
#pragma unroll
            for (int e = 0; e < TN; e++) v[e] += a.residual[o + e];
        }
        if (a.accumulate) {
#pragma unroll
            for (int e = 0; e < TN; e++) v[e] = a.out[o + e] + v[e];
        }
        if (a.div != 1.0f) {
#pragma unroll
            for (int e = 0; e < TN; e++) v[e] = __fdiv_rn(v[e], a.div);
        }
        if (a.out) {
            if constexpr (TN == 4) *reinterpret_cast<float4 *>(a.out + o) = make_float4(v[0], v[1], v[2], v[3]);
            else *reinterpret_cast<float2 *>(a.out + o) = make_float2(v[0], v[1]);
        }
        if (a.out_bf16) {
#pragma unroll
            for (int e = 0; e < TN; e += 2) {
                __nv_bfloat162 p = __floats2bfloat162_rn(lrelu(v[e], a.bf16_slope), lrelu(v[e + 1], a.bf16_slope));
                *reinterpret_cast<__nv_bfloat162 *>(a.out_bf16 + o + e) = p;
            }
        }
    }
}

int launch_conv_simt(const ConvArgs &a, cudaStream_t st) {
    if (a.W <= 0 || a.Tout <= 0) return 0;
    if (a.Cin % 4 || a.Cout % 4) return set_error("conv_simt: Cin (%d) and Cout (%d) must be multiples of 4", a.Cin, a.Cout);
    const long long M = (long long)a.W * a.Tout;
    if (a.Cout % 64 == 0) {
        dim3 grid((unsigned)cdiv(M, 128), (unsigned)(a.Cout / 64));
        k_conv_simt<64><<<grid, 256, 0, st>>>(a);
    } else {
        dim3 grid((unsigned)cdiv(M, 128), (unsigned)cdiv(a.Cout, 32));
        k_conv_simt<32><<<grid, 256, 0, st>>>(a);
    }
    B2_LAUNCH_OK("k_conv_simt");
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// conv_post: leaky_relu(0.01) -> Conv1d(32 -> 1, k7, pad 3) -> tanh.   Memory-bound (128 B in, 4 B out per sample).
// One CTA = 512 consecutive samples of one window: the 518 x 32 input patch is read once with coalesced 128-bit
// loads (leaky-ReLU applied on the way), transposed into shared memory as [channel][time]; each thread then
// slides over 4 consecutive outputs reading three 128-bit words per channel, conflict-free.
// ---------------------------------------------------------------------------------------------------
static constexpr int kPostTile = 512;
static constexpr int kPostLd = kPostTile + 8;      // [c][4 halo | 512 | 4 halo], 16-byte aligned rows

__global__ void __launch_bounds__(128) k_conv_post(const float *__restrict__ in, const float *__restrict__ wt, const float *__restrict__ bias,
                                                  float *__restrict__ out, int T, int tiles_per_win) {
    extern __shared__ __align__(16) float xs[];    // [32][kPostLd]
    __shared__ float ws[7 * 32];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    for (int i = tid; i < 224; i += 128) ws[i] = wt[i];
    const int w = blockIdx.x / tiles_per_win;
    const int t0 = (blockIdx.x - w * tiles_per_win) * kPostTile;
    const float *inw = in + (long long)w * T * 32;
    // rows t0-4 .. t0+515 -> xs[c][0 .. 519]
    for (int rb = warp * 32; rb < kPostLd; rb += 128) {
        const int rl = rb + lane;
        const int t = t0 - 4 + rl;
        const bool ok = rl < kPostLd && t >= 0 && t < T;
#pragma unroll
        for (int c4 = 0; c4 < 8; c4++) {
            float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
            if (ok) v = __ldg(reinterpret_cast<const float4 *>(inw + (long long)t * 32 + c4 * 4));
            if (rl < kPostLd) {
                xs[(c4 * 4 + 0) * kPostLd + rl] = lrelu(v.x, 0.01f);
                xs[(c4 * 4 + 1) * kPostLd + rl] = lrelu(v.y, 0.01f);
                xs[(c4 * 4 + 2) * kPostLd + rl] = lrelu(v.z, 0.01f);
                xs[(c4 * 4 + 3) * kPostLd + rl] = lrelu(v.w, 0.01f);
            }
        }
    }
    __syncthreads();
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll 4
    for (int c = 0; c < 32; c++) {
        const float *row = xs + c * kPostLd + tid * 4;           // row[4 + e + j - 3] is x[t0 + 4*tid + e + j - 3]
        const float4 a = *reinterpret_cast<const float4 *>(row);
        const float4 b = *reinterpret_cast<const float4 *>(row + 4);
        const float4 d = *reinterpret_cast<const float4 *>(row + 8);
        const float x[12] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w, d.x, d.y, d.z, d.w};
#pragma unroll
        for (int j = 0; j < 7; j++) {
            const float wv = ws[j * 32 + c];
#pragma unroll
            for (int e = 0; e < 4; e++) acc[e] = fmaf(wv, x[1 + e + j], acc[e]);
        }
    }
    const int t = t0 + tid * 4;
    if (t < T) {      // T is a multiple of 4 (256 samples per frame)
        const float b = bias[0];
        *reinterpret_cast<float4 *>(out + (long long)w * T + t) = make_float4(tanhf(acc[0] + b), tanhf(acc[1] + b), tanhf(acc[2] + b), tanhf(acc[3] + b));
    }
}

int launch_conv_post(const float *in, const float *wt, const float *bias, float *out, int W, int T, cudaStream_t st) {
    if (W <= 0 || T <= 0) return 0;
    if (T % 4) return set_error("conv_post: T must be a multiple of 4");
    static bool attr_set[64] = {false};
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    const size_t smem = (size_t)32 * kPostLd * sizeof(float);
    if (dev < 64 && !attr_set[dev]) {
        B2_CUDA_OK(cudaFuncSetAttribute(k_conv_post, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set[dev] = true;
    }
    const int tiles = cdiv(T, kPostTile);
    k_conv_post<<<(unsigned)((long long)W * tiles), 128, smem, st>>>(in, wt, bias, out, T, tiles);
    B2_LAUNCH_OK("k_conv_post");
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// window builder: one CTA per session
// ---------------------------------------------------------------------------------------------------
// Slot ids arrive from the caller in device memory, so they are checked HERE: an id outside [0, max_sessions) would read and
// write pre_pool out of bounds, and the same id twice in one call races the read of pre[] against its overwrite.  A bad session
// gets zero pre_frames, writes nothing back and raises bit 0 (range) / bit 1 (duplicate) of *err_flag (host-mapped memory that
// the C-ABI reads after the stream has been synchronised, tail.cu:poll_slot_errors).  claim[slot] holds the epoch (one per launch) of the
// last call that used the slot.
__global__ void __launch_bounds__(256) k_build_windows(const int32_t *__restrict__ slots, const float *__restrict__ mel, float *__restrict__ pre_pool,
                                                      const float *__restrict__ mean, const float *__restrict__ scale,
                                                      float *__restrict__ win_raw, float *__restrict__ win_norm, __nv_bfloat16 *__restrict__ win_norm_b,
                                                      int B, int nframes, int max_sessions, unsigned *__restrict__ claim, unsigned epoch,
                                                      int *__restrict__ err_flag) {
    pdl_trigger();
    pdl_wait(slots, mel, pre_pool);
    const int nwin = nframes / 8;
    __shared__ int s_ok;
    for (int b = blockIdx.x; b < B; b += gridDim.x) {
        const int slot = slots[b];
        if (threadIdx.x == 0) {
            int ok = 1;
            if (slot < 0 || slot >= max_sessions) { ok = 0; atomicOr(err_flag, 1); }
            else if (claim && atomicExch(claim + slot, epoch) == epoch) { ok = 0; atomicOr(err_flag, 2); }
            s_ok = ok;
        }
        __syncthreads();
        const bool ok = s_ok != 0;
        float *pre = pre_pool + (long long)(ok ? slot : 0) * 320;
        const float *m = mel + (long long)b * nframes * 80;
        const long long wbase = (long long)b * nwin * 960;
        // spec frame f (0 .. nframes+3): f < 4 -> pre[f], else mel[f-4]; window i covers frames 8i .. 8i+11
        for (int e = threadIdx.x; e < nwin * 960; e += blockDim.x) {
            const int i = e / 960, rem = e - i * 960;
            const int fr = rem / 80, bin = rem - fr * 80;
            const int f = 8 * i + fr;
            const float v = (f < 4) ? (ok ? pre[f * 80 + bin] : 0.0f) : m[(f - 4) * 80 + bin];
            win_raw[wbase + e] = v;
            const float nv = __fdiv_rn(v - mean[bin], scale[bin]);
            win_norm[wbase + e] = nv;
            if (win_norm_b) win_norm_b[((long long)b * nwin * 12 + i * 12 + fr) * 128 + bin] = __float2bfloat16_rn(nv);
        }
        if (win_norm_b)
            for (int e = threadIdx.x; e < nwin * 12 * 48; e += blockDim.x)
                win_norm_b[((long long)b * nwin * 12 + e / 48) * 128 + 80 + e % 48] = __float2bfloat16_rn(0.0f);
        __syncthreads();   // every read of pre[] is done before it is overwritten
        if (ok)
            for (int e = threadIdx.x; e < 320; e += blockDim.x) pre[e] = m[(nframes - 4) * 80 + e];
        __syncthreads();
    }
}

int launch_build_windows(const int32_t *slots, const float *mel, float *pre_pool, const float *mean, const float *scale,
                         float *win_raw, float *win_norm, __nv_bfloat16 *win_norm_b, int B, int nframes,
                         int max_sessions, unsigned *claim, unsigned epoch, int *err_flag, cudaStream_t st) {
    if (B <= 0) return 0;
    B2_CUDA_OK(launch_k(k_build_windows, dim3(B), dim3(256), 0, st, pdl_enabled(), slots, mel, pre_pool, mean, scale, win_raw, win_norm, win_norm_b, B, nframes, max_sessions, claim, epoch, err_flag));
    B2_LAUNCH_OK("k_build_windows");
    return 0;
}

__global__ void __launch_bounds__(256) k_normalise(const float *__restrict__ mel, const float *__restrict__ mean, const float *__restrict__ scale,
                                                  float *__restrict__ out, __nv_bfloat16 *__restrict__ out_b, size_t n) {
    size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const size_t row = i / 80;
        const int bin = (int)(i - row * 80);
        const float nv = __fdiv_rn(mel[i] - mean[bin], scale[bin]);
        out[i] = nv;
        if (out_b) {
            out_b[row * 128 + bin] = __float2bfloat16_rn(nv);
            if (bin < 48) out_b[row * 128 + 80 + bin] = __float2bfloat16_rn(0.0f);
        }
    }
}

int launch_normalise(const float *mel, const float *mean, const float *scale, float *out, __nv_bfloat16 *out_b, size_t rows, cudaStream_t st) {
    size_t n = rows * 80;
    if (n == 0) return 0;
    size_t blocks = (n + 255) / 256, cap = (size_t)sm_count() * 16;
    k_normalise<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(mel, mean, scale, out, out_b, n);
    B2_LAUNCH_OK("k_normalise");
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// chunker prologue: one CTA (192 threads) per window; thread = output channel, 12 accumulators (time).
// warp 0 = the 32 mel channels (Cin 80), warps 1..5 = the 160 audio channels (Cin 256).
// mel_view[ci][t] = mel_window_flat[ci*12 + t]; audio_view[ci][t] = audio[ci*12 + t]  (raw .view, not a transpose)
// ---------------------------------------------------------------------------------------------------
// NW windows per trip: every weight is fetched once per NW windows (the 491 KB of conv_pre_a weights do not fit L1, so at one
// window per trip the kernel was bound by re-reading them from L2: 2 GB per call at 4,096 windows)
template <int NW>
__global__ void __launch_bounds__(192) k_chunker_pre(const float *__restrict__ mel, const float *__restrict__ audio,
                                                    const float *__restrict__ wm, const float *__restrict__ bm,
                                                    const float *__restrict__ wa, const float *__restrict__ ba,
                                                    float *__restrict__ z0, int W) {
    extern __shared__ __align__(16) float smem_f[];
    float *sm = smem_f;                       // [NW][80 * 12]
    float *sa = smem_f + NW * 960;            // [NW][256 * 12]
    const int tid = threadIdx.x;
    const int ngroups = (W + NW - 1) / NW;
    for (int g = blockIdx.x; g < ngroups; g += gridDim.x) {
        const int w0 = g * NW;
        for (int e = tid; e < NW * 960; e += 192) { const int q = e / 960; sm[e] = (w0 + q < W) ? mel[(long long)w0 * 960 + e] : 0.0f; }
        for (int e = tid; e < NW * 3072; e += 192) { const int q = e / 3072; sa[e] = (w0 + q < W) ? audio[(long long)w0 * 3072 + e] : 0.0f; }
        __syncthreads();
        float acc[NW][12];
        const bool is_mel = tid < 32;
        const int co = is_mel ? tid : tid - 32;
        const int Cin = is_mel ? 80 : 256, Cout = is_mel ? 32 : 160;
        const float *src = is_mel ? sm : sa;
        const int wstride = is_mel ? 960 : 3072;
        const float *wt = is_mel ? wm : wa;
        const float b = is_mel ? bm[co] : ba[co];
#pragma unroll
        for (int q = 0; q < NW; q++)
#pragma unroll
            for (int t = 0; t < 12; t++) acc[q][t] = b;
        for (int ci = 0; ci < Cin; ci++) {
            float wv[3];
#pragma unroll
            for (int k = 0; k < 3; k++) wv[k] = __ldg(wt + ((long long)k * Cin + ci) * Cout + co);
#pragma unroll
            for (int q = 0; q < NW; q++) {
                const float *row = src + q * wstride + ci * 12;
                const float4 x0 = *reinterpret_cast<const float4 *>(row);
                const float4 x1 = *reinterpret_cast<const float4 *>(row + 4);
                const float4 x2 = *reinterpret_cast<const float4 *>(row + 8);
                const float x[14] = {0.f, x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w, x2.x, x2.y, x2.z, x2.w, 0.f};
#pragma unroll
                for (int k = 0; k < 3; k++)
#pragma unroll
                    for (int t = 0; t < 12; t++) acc[q][t] = fmaf(wv[k], x[t + k], acc[q][t]);
            }
        }
#pragma unroll
        for (int q = 0; q < NW; q++) {
            if (w0 + q >= W) break;
            float *o = z0 + (long long)(w0 + q) * 12 * 192 + tid;
#pragma unroll
            for (int t = 0; t < 12; t++) o[t * 192] = acc[q][t];
        }
        __syncthreads();
    }
}

// Operand of the chunker prologue on tensor cores: inb[w][t][ci] = audio[w][12 ci + t] (ci < 256), mel_flat[w][12 (ci - 256) + t] (ci < 336),
// 0 (ci < 384) -- the two raw `.view` reinterpretations of HelloSippyRT.py:221-224 side by side as one channels-last bf16 tensor [W][12][384].
__global__ void __launch_bounds__(384) k_chunker_in(const float *__restrict__ mel, const float *__restrict__ audio, __nv_bfloat16 *__restrict__ inb, int W) {
    pdl_trigger();
    pdl_wait(mel, audio);
    const int ci = threadIdx.x;
    for (int w = blockIdx.x; w < W; w += gridDim.x) {
        float v[12];
        const float *src = ci < 256 ? audio + (long long)w * 3072 + 12 * ci : (ci < 336 ? mel + (long long)w * 960 + 12 * (ci - 256) : nullptr);
#pragma unroll
        for (int q = 0; q < 3; q++) {
            const float4 f = src ? __ldg(reinterpret_cast<const float4 *>(src) + q) : make_float4(0.f, 0.f, 0.f, 0.f);
            v[4 * q] = f.x; v[4 * q + 1] = f.y; v[4 * q + 2] = f.z; v[4 * q + 3] = f.w;
        }
        __nv_bfloat16 *o = inb + (long long)w * 12 * 384 + ci;
#pragma unroll
        for (int t = 0; t < 12; t++) o[t * 384] = __float2bfloat16_rn(v[t]);
    }
}

int launch_chunker_in(const float *mel, const float *audio, __nv_bfloat16 *inb, int W, cudaStream_t st) {
    if (W <= 0) return 0;
    B2_CUDA_OK(launch_k(k_chunker_in, dim3((unsigned)std::min<long long>(W, (long long)sm_count() * 8)), dim3(384), 0, st, pdl_enabled(), mel, audio, inb, W));
    B2_LAUNCH_OK("k_chunker_in");
    return 0;
}

int launch_chunker_pre(const float *mel, const float *audio, const float *wm, const float *bm, const float *wa, const float *ba,
                       float *z0, int W, cudaStream_t st) {
    if (W <= 0) return 0;
    constexpr int NW = 4;
    static bool attr_set[64] = {};
    const size_t smem = (size_t)NW * (960 + 3072) * sizeof(float);
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 64 && !attr_set[dev]) {
        B2_CUDA_OK(cudaFuncSetAttribute(k_chunker_pre<NW>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_set[dev] = true;
    }
    const int groups = (W + NW - 1) / NW;
    const int cap = sm_count() * 3;
    k_chunker_pre<NW><<<groups < cap ? groups : cap, 192, smem, st>>>(mel, audio, wm, bm, wa, ba, z0, W);
    B2_LAUNCH_OK("k_chunker_pre");
    return 0;
}

__global__ void __launch_bounds__(256) k_chunker_final(const float *__restrict__ audio, const float *__restrict__ post, float *__restrict__ out, long long n) {
    pdl_trigger();
    pdl_wait(audio, post);
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
        const long long w = e >> 11;
        const int i = (int)(e & 2047);
        const float g = lrelu(post[w * 2048 + (i & 7) * 256 + (i >> 3)], 0.01f);
        out[e] = tanhf(audio[w * 3072 + 512 + i] * g);
    }
}

int launch_chunker_final(const float *audio, const float *post, float *out, int W, cudaStream_t st) {
    const long long n = (long long)W * 2048;
    if (n <= 0) return 0;
    long long blocks = (n + 255) / 256, cap = (long long)sm_count() * 16;
    B2_CUDA_OK(launch_k(k_chunker_final, dim3((unsigned)(blocks < cap ? blocks : cap)), dim3(256), 0, st, pdl_enabled(), audio, post, out, n));
    B2_LAUNCH_OK("k_chunker_final");
    return 0;
}

__global__ void __launch_bounds__(256) k_trim(const float *__restrict__ audio, float *__restrict__ out, long long n, int Lin, int lo, int Lout) {
    const long long stride = (long long)gridDim.x * blockDim.x;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += stride) {
        const long long w = e / Lout;
        const int i = (int)(e - w * Lout);
        out[e] = audio[w * Lin + lo + i];
    }
}

int launch_trim(const float *audio, float *out, int W, int Lin, int lo, int Lout, cudaStream_t st) {
    const long long n = (long long)W * Lout;
    if (n <= 0) return 0;
    long long blocks = (n + 255) / 256, cap = (long long)sm_count() * 16;
    k_trim<<<(unsigned)(blocks < cap ? blocks : cap), 256, 0, st>>>(audio, out, n, Lin, lo, Lout);
    B2_LAUNCH_OK("k_trim");
    return 0;
}

// ---------------------------------------------------------------------------------------------------
// post-net element-wise steps (see conv_simt.cuh).  All HBM-bound, 128-bit accesses, grid-stride.
// ---------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pn_prep(const float *__restrict__ mel, __nv_bfloat16 *__restrict__ outb, size_t rows) {
    // one thread = 8 output bins (one 16-byte store); 16 threads per row
    const size_t total = rows * 16;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i >> 4;
        const int q = (int)(i & 15);
        uint4 o = make_uint4(0u, 0u, 0u, 0u);
        if (q < 10) {
            const float4 a = __ldg(reinterpret_cast<const float4 *>(mel + r * 80 + q * 8));
            const float4 b = __ldg(reinterpret_cast<const float4 *>(mel + r * 80 + q * 8 + 4));
            __nv_bfloat162 h0 = __floats2bfloat162_rn(a.x, a.y), h1 = __floats2bfloat162_rn(a.z, a.w);
            __nv_bfloat162 h2 = __floats2bfloat162_rn(b.x, b.y), h3 = __floats2bfloat162_rn(b.z, b.w);
            o = make_uint4(*reinterpret_cast<uint32_t *>(&h0), *reinterpret_cast<uint32_t *>(&h1), *reinterpret_cast<uint32_t *>(&h2), *reinterpret_cast<uint32_t *>(&h3));
        }
        reinterpret_cast<uint4 *>(outb)[i] = o;
    }
}

__global__ void __launch_bounds__(256) k_pn_tanh(const float *__restrict__ in, float *__restrict__ out32, __nv_bfloat16 *__restrict__ outb, size_t n4) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
        float4 v = reinterpret_cast<const float4 *>(in)[i];
        v.x = tanhf(v.x); v.y = tanhf(v.y); v.z = tanhf(v.z); v.w = tanhf(v.w);
        if (out32) reinterpret_cast<float4 *>(out32)[i] = v;
        if (outb) {
            __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
            reinterpret_cast<uint2 *>(outb)[i] = make_uint2(*reinterpret_cast<uint32_t *>(&h0), *reinterpret_cast<uint32_t *>(&h1));
        }
    }
}

__global__ void __launch_bounds__(256) k_pn_out(const float *__restrict__ mel, const float *__restrict__ y, int ystride, float *__restrict__ out, size_t rows) {
    const size_t total = rows * 20;                 // 20 float4 per row of 80 bins
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const size_t r = i / 20;
        const int q = (int)(i - r * 20);
        const float4 m = __ldg(reinterpret_cast<const float4 *>(mel) + i);
        const float4 v = __ldg(reinterpret_cast<const float4 *>(y + r * ystride) + q);
        reinterpret_cast<float4 *>(out)[i] = make_float4(m.x + v.x, m.y + v.y, m.z + v.z, m.w + v.w);
    }
}

static inline int ew_grid(size_t items) {
    long long b = (long long)((items + 255) / 256);
    const long long cap = (long long)sm_count() * 8;
    return (int)(b < 1 ? 1 : (b > cap ? cap : b));
}

int launch_pn_prep(const float *mel, __nv_bfloat16 *outb, size_t rows, cudaStream_t st) {
    if (!rows) return 0;
    k_pn_prep<<<ew_grid(rows * 16), 256, 0, st>>>(mel, outb, rows);
    B2_LAUNCH_OK("k_pn_prep");
    return 0;
}

int launch_pn_tanh(const float *in, float *out32, __nv_bfloat16 *outb, size_t n, cudaStream_t st) {
    if (!n) return 0;
    if (n % 4) return set_error("pn_tanh: element count must be a multiple of 4");
    k_pn_tanh<<<ew_grid(n / 4), 256, 0, st>>>(in, out32, outb, n / 4);
    B2_LAUNCH_OK("k_pn_tanh");
    return 0;
}

int launch_pn_out(const float *mel, const float *y, int ystride, float *out, size_t rows, cudaStream_t st) {
    if (!rows) return 0;
    if (ystride % 4) return set_error("pn_out: row stride must be a multiple of 4");
    k_pn_out<<<ew_grid(rows * 20), 256, 0, st>>>(mel, y, ystride, out, rows);
    B2_LAUNCH_OK("k_pn_out");
    return 0;
}

}  // namespace b2
