// Transformer building blocks shared by the SpeechT5 speech decoder (decoder.cu) and text encoder (encoder.cu): a Linear packed for both
// precision modes (fp32 [K][N] for the CUDA-core conv kernel; bf16 [N][K] + TMA maps for the tcgen05 GEMM of gemm_tc.cuh), its packing
// from torch state_dict tensors, the launch of one Linear in either mode, and the residual + LayerNorm kernel.
#pragma once
#include "common.cuh"
#include "ctx.cuh"
#include "conv_simt.cuh"
#include "gemm_tc.cuh"
#include "../../include/infernos_b200.h"

#include <cuda.h>
#include <math.h>
#include <stdlib.h>
#include <algorithm>
#include <initializer_list>
#include <map>
#include <string>
#include <vector>

namespace b2 {

struct DecLinear {
    int K = 0, N = 0;                      // padded sizes
    float *w32 = nullptr, *bias = nullptr; // fp32 [K][N] (1-tap conv layout), [N]
    __nv_bfloat16 *wbf = nullptr;          // bf16 [N][K]
    CUtensorMap tmB;                       // box 64 x NT over wbf
    int nt = 128;
    CUtensorMap tmB256;                    // box 64 x 256 over wbf (N % 256 == 0, N >= 2048): 128 x 256 tiles when 128 x 128 ones would not fit one wave
    bool has256 = false;
};

// what a handle that owns packed Linears keeps for them: the state_dict tensors until finalize, its device allocations, mode and launch style
struct LinearOwner {
    const char *what = "";                 // "decoder" / "encoder": prefix of error messages
    int device = 0, mode = 0;
    bool use_pdl = true;                   // programmatic dependent launch between the kernels of a pass
    std::map<std::string, HostTensor> raw;
    std::vector<void *> allocs;
    size_t device_bytes = 0;
};

}  // namespace b2

namespace {

using namespace b2;

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }

__device__ __forceinline__ float block_max(float v, float *red) {
    for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = red[0];
    for (int i = 1; i < (int)(blockDim.x >> 5); i++) r = fmaxf(r, red[i]);
    __syncthreads();
    return r;
}
__device__ __forceinline__ float block_sum(float v, float *red) {
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    float r = 0.0f;
    for (int i = 0; i < (int)(blockDim.x >> 5); i++) r += red[i];
    __syncthreads();
    return r;
}

// fp32 mode: x = act(x) * colscale[col], in place (the bf16 GEMM does this in its epilogue)
__global__ void k_act_scale(float *__restrict__ x, const float *__restrict__ colscale, size_t n, int N, int act) {
    pdl_trigger();
    pdl_wait(x, colscale);
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        float v = x[i];
        if (act == 1) v = fmaxf(v, 0.0f);
        else if (act == 2) v = gelu_erf(v);
        if (colscale) v *= colscale[i % (size_t)N];
        x[i] = v;
    }
}

// h = LayerNorm(h + o) * w + b over 768 columns, eps 1e-5, biased variance (torch.nn.LayerNorm); 256 threads per row
__global__ void __launch_bounds__(256) k_add_ln(float *__restrict__ h, const float *__restrict__ o, const float *__restrict__ w, const float *__restrict__ b,
                                               __nv_bfloat16 *__restrict__ hb, int M) {
    constexpr int H = 768;
    pdl_trigger();
    pdl_wait(h, o);
    __shared__ float red[8];
    const int m = blockIdx.x, tid = threadIdx.x;
    if (m >= M) return;
    float v[3];
    float s = 0.0f;
#pragma unroll
    for (int i = 0; i < 3; i++) { v[i] = h[(size_t)m * H + tid + 256 * i] + o[(size_t)m * H + tid + 256 * i]; s += v[i]; }
    const float mean = block_sum(s, red) * (1.0f / H);
    float q = 0.0f;
#pragma unroll
    for (int i = 0; i < 3; i++) { const float d = v[i] - mean; q += d * d; }
    const float rstd = rsqrtf(block_sum(q, red) * (1.0f / H) + 1e-5f);
#pragma unroll
    for (int i = 0; i < 3; i++) {
        const int c = tid + 256 * i;
        const float y = (v[i] - mean) * rstd * w[c] + b[c];
        h[(size_t)m * H + c] = y;
        if (hb) hb[(size_t)m * H + c] = __float2bfloat16_rn(y);
    }
}

// ---------------------------------------------------------------------------------------------------- host side
inline int make_map(CUtensorMap *tm, const void *ptr, int rows, int K, int box_rows) { return b2::make_tma_2d_bf16(tm, ptr, rows, K, K, box_rows); }

template <typename T>
int dalloc(LinearOwner *d, T **p, size_t n, bool zero = true) {
    void *q = nullptr;
    const size_t bytes = std::max<size_t>(n * sizeof(T), 16);
    cudaError_t e = cudaMalloc(&q, bytes);
    if (e != cudaSuccess) return b2::set_error("%s: cudaMalloc of %zu bytes failed: %s", d->what, bytes, cudaGetErrorString(e));
    if (zero) cudaMemset(q, 0, bytes);
    d->allocs.push_back(q);
    d->device_bytes += bytes;
    *p = reinterpret_cast<T *>(q);
    return 0;
}

inline const HostTensor *need(LinearOwner *d, const std::string &k, std::initializer_list<int64_t> shape) {
    auto it = d->raw.find(k);
    if (it == d->raw.end()) { b2::set_error("%s weight '%s' was not loaded", d->what, k.c_str()); return nullptr; }
    if (it->second.shape != std::vector<int64_t>(shape)) { b2::set_error("%s weight '%s' has an unexpected shape", d->what, k.c_str()); return nullptr; }
    return &it->second;
}

// packs rows [n_lo, n_lo + n) of the destination from a torch Linear weight [n][k] (+ bias), scaled; K and N are the padded sizes
inline void fill_linear(std::vector<float> &W, std::vector<float> &B, int Kp, int Np, int n_lo, const HostTensor &w, const HostTensor &b, float scale) {
    const int n = (int)w.shape[0], k = (int)w.shape[1];
    for (int i = 0; i < n; i++) {
        for (int j = 0; j < k; j++) W[(size_t)(n_lo + i) * Kp + j] = w.data[(size_t)i * k + j] * scale;
        B[(size_t)n_lo + i] = b.data[i] * scale;
    }
    (void)Np;
}

inline int upload_linear(LinearOwner *d, DecLinear &l, int Kp, int Np, const std::vector<float> &W, const std::vector<float> &B) {
    l.K = Kp; l.N = Np;
    l.nt = (Np % 128 == 0 && Np >= 2048) ? 128 : 64;        // N = 768 layers: 64-wide tiles double the CTA count (8 x 12 at 1,024 rows)
    if (dalloc(d, &l.bias, (size_t)Np)) return 1;
    B2_CUDA_OK(cudaMemcpy(l.bias, B.data(), (size_t)Np * sizeof(float), cudaMemcpyHostToDevice));
    if (d->mode == B2_MODE_BF16) {
        std::vector<__nv_bfloat16> hb((size_t)Np * Kp);
        for (size_t i = 0; i < hb.size(); i++) hb[i] = __float2bfloat16_rn(W[i]);
        if (dalloc(d, &l.wbf, hb.size(), false)) return 1;
        B2_CUDA_OK(cudaMemcpy(l.wbf, hb.data(), hb.size() * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice));
        if (make_map(&l.tmB, l.wbf, Np, Kp, l.nt)) return 1;
        if (l.nt == 128 && Np % 256 == 0) {
            if (make_map(&l.tmB256, l.wbf, Np, Kp, 256)) return 1;
            l.has256 = true;
        }
    } else {
        std::vector<float> t((size_t)Kp * Np);
        for (int n = 0; n < Np; n++)
            for (int k = 0; k < Kp; k++) t[(size_t)k * Np + n] = W[(size_t)n * Kp + k];
        if (dalloc(d, &l.w32, t.size(), false)) return 1;
        B2_CUDA_OK(cudaMemcpy(l.w32, t.data(), t.size() * sizeof(float), cudaMemcpyHostToDevice));
    }
    return 0;
}

inline int pack_one(LinearOwner *d, DecLinear &l, const std::string &key, int n, int k, int Kp, int Np, float scale = 1.0f) {
    const HostTensor *w = need(d, key + ".weight", {n, k}), *b = need(d, key + ".bias", {n});
    if (!w || !b) return 1;
    std::vector<float> W((size_t)Np * Kp, 0.0f), B((size_t)Np, 0.0f);
    fill_linear(W, B, Kp, Np, 0, *w, *b, scale);
    return upload_linear(d, l, Kp, Np, W, B);
}

inline int upload_vec(LinearOwner *d, float **dst, const HostTensor &t) {
    if (dalloc(d, dst, t.data.size(), false)) return 1;
    B2_CUDA_OK(cudaMemcpy(*dst, t.data.data(), t.data.size() * sizeof(float), cudaMemcpyHostToDevice));
    return 0;
}

// Tile width of a bf16-mode Linear's GEMM over M rows.  One tile per CTA: when the 128 x 128 tiles of a wide layer do not fit one wave (ffn1 at
// 1,024 rows: 8 x 24 = 192 CTAs on 148 SMs, the second wave 30 % full: 46 us against 21 us for the 144-CTA qkv GEMM), 128 x 256 tiles do (96 CTAs).
// B2_GEMM_NT256=0 keeps 128.
inline int gemm_tile_n(const DecLinear &l, int M) {
    static const bool nt256_on = !(getenv("B2_GEMM_NT256") && atoi(getenv("B2_GEMM_NT256")) == 0);
    return nt256_on && l.has256 && (long long)cdiv(M, 128) * (l.N / 128) > sm_count() ? 256 : l.nt;
}

// C = act(A W^T + bias) * colscale.  fp32 mode: A32 [M][K] through the CUDA-core conv kernel (+ k_act_scale); bf16 mode: tmA over the bf16 A buffer.
inline int linear(LinearOwner *d, const DecLinear &l, const float *A32, const CUtensorMap *tmA, int M, int act, const float *colscale,
                  float *out32, __nv_bfloat16 *outb, cudaStream_t st) {
    using namespace b2;
    if (M <= 0) return 0;
    if (d->mode == B2_MODE_BF16) {
        GemmTcArgs g;
        g.tmA = tmA; g.bias = l.bias; g.colscale = colscale; g.out32 = out32; g.outb = outb; g.M = M; g.N = l.N; g.K = l.K; g.act = act; g.pdl = d->use_pdl;
        g.nt = gemm_tile_n(l, M);
        g.tmB = g.nt == 256 ? &l.tmB256 : &l.tmB;
        return launch_gemm_tc(g, st);
    }
    ConvArgs a;
    a.in = A32; a.wt = l.w32; a.bias = l.bias; a.residual = nullptr; a.out = out32; a.out_bf16 = nullptr;
    a.W = 1; a.Tin = M; a.Tout = M; a.Cin = l.K; a.Cout = l.N; a.taps = 1; a.dil = 1; a.pad = 0; a.stride = 1;
    a.pre_slope = 1.0f; a.bf16_slope = 1.0f; a.div = 1.0f; a.accumulate = 0;
    if (launch_conv_simt(a, st)) return 1;
    if (act || colscale) {
        const size_t n = (size_t)M * l.N;
        B2_CUDA_OK(launch_k(k_act_scale, dim3((unsigned)std::min<size_t>((n + 255) / 256, (size_t)sm_count() * 8)), dim3(256), 0, st, d->use_pdl, out32, colscale, n, l.N, act));
        B2_LAUNCH_OK("k_act_scale");
    }
    return 0;
}

}  // namespace
