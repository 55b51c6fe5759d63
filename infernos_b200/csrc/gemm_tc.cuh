// tcgen05 GEMM with both operands by TMA (decoder.cu): C[m][n] = act(sum_k A[m][k] * W[n][k] + bias[n]) * colscale[n].
#pragma once
#include "common.cuh"
#include <cuda.h>

namespace b2 {

struct GemmTcArgs {
    const CUtensorMap *tmA = nullptr;   // bf16 [rows][K] (any 16-byte-multiple row stride), box 64 x 128, 128-byte swizzle
    const CUtensorMap *tmB = nullptr;   // bf16 [N][K] row-major, box 64 x nt
    const float *bias = nullptr;        // [N]
    const float *colscale = nullptr;    // optional [N]
    float *out32 = nullptr;             // optional [M][N]
    __nv_bfloat16 *outb = nullptr;      // optional [M][N]
    int M = 0, N = 0, K = 0, nt = 128, act = 0;   // N % nt == 0, K % 64 == 0; act: 0 none, 1 relu, 2 gelu (erf)
    bool pdl = false;                   // launch with the programmatic-stream-serialization attribute (the decoder's kernel chain)
};
int launch_gemm_tc(const GemmTcArgs &a, cudaStream_t st);
// stages of the shared-memory operand ring launch_gemm_tc uses for K and tile width nt
int gemm_tc_stages(int K, int nt);
// TMA map over row-major bf16 [rows][K] with `row_stride` ELEMENTS between rows (>= K), box 64 x box_rows, 128-byte swizzle
int make_tma_2d_bf16(CUtensorMap *tm, const void *ptr, long long rows, int K, long long row_stride, int box_rows);

}  // namespace b2
