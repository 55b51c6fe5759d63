// The C = 32 HiFiGAN ResBlock (stage 3: T = 3,072 per window, a third of the step) with FOUR OUTPUT TIME STEPS STACKED INTO THE MMA's N
// dimension ("block-Toeplitz" form; modeling_speecht5.py:2903-2962 is the arithmetic, conv_resblock.cu the time-as-M kernel this replaces).
//
// Why.  With time as M and the 32 output channels as N, one tcgen05.mma (M128 x N32 x K16) occupies the tensor pipe for 40 cycles -- 32 of
// them fetching the 4 KB activation slice from shared memory -- for 8 cycles of math (profiles/r1b_mma_rate_microbench.txt), and the k = 7 / 11
// launches of stage 3 are bound by exactly that (phase timestamps: with two CTAs per SM the pipe is saturated during the conv phases).
// Here one A row serves four outputs:
//
//     D[m][(r', co)] = sum_{j', ci} A[m][(j', ci)] * B[(j', ci)][(r', co)]          r' = 0..3 stacked outputs, j' = 0..k+2 extended taps
//     A[m][(j', ci)] = act[ci][ d*(4v + j' - half) + rho ]                           m = (v, rho): rho = time mod d, v = (time div d) div 4
//     B[(j', ci)][(r', co)] = W[co][ci][j' - r']   (zero when j' - r' is not a tap)
//     D[m][(r', co)] = conv(time = d*(4v + r') + rho)[co]
//
// i.e. N = 128 at 64 cycles per K16 step = the tensor pipe's full rate, (k + 3) extended taps instead of 4 x k: 2.2x / 1.75x / 1.25x fewer
// pipe cycles for k = 11 / 7 / 3 (the edge taps j' < 3 and j' >= k touch fewer r' and run as N = 32 / 64 / 96 MMAs on a column sub-range).
//
// Layouts.  Operand buffers (shared, bf16) are de-interleaved so that the rows of ONE extended tap are 16 bytes apart, as the un-swizzled
// K-major UMMA layout wants:  [ci / 8][b = (time div d) mod 4][row = kTG + v*d + rho][8 ch]; extended tap j' reads block (j' - half) mod 4 at
// a row offset of ((j' - half) div 4) * d.  The mapping depends on the dilation of the conv that READS the buffer, so every epilogue scatters
// its rows by the next conv's mapping (16-byte stores, conflict-free because kTBR = 1 mod 8).  B: the k taps of the conv in REVERSE order,
// one 2 KB TMA slot each (SWIZZLE_64B); the four stacked outputs of extended tap j' are the consecutive slots k-1-j'+r', so a B tile is a
// sliding window over the slots and nothing is replicated.  Accumulators (TMEM): X = the fp32 residual stream, 128 lanes x (4 x 32) columns,
// lane m <-> times 4m..4m+3 (conv2 has dilation 1); T1 = conv1's output in ITS dilation's mapping.  T1 is pre-loaded with conv1's bias by
// tcgen05.st (exact fp32, and the conv epilogue loses its bias add), so every MMA accumulates.
//
// One CTA = one slab of S <= 512 time steps of one window (halo H as in conv_resblock.cu), one 128-lane accumulator tile; two CTAs share an SM
// (2 x 256 TMEM columns, 2 x 99 KB shared memory) and fill each other's epilogue phases.  Warps: 0-3 load + epilogues (TMEM lane quadrants),
// 4 TMEM alloc + TMA weight ring, 5 MMA issue (one elected thread, everything in uniform registers).
#include "conv_umma.cuh"
#include "umma_ptx.cuh"

#include <cuda.h>
#include <stdlib.h>
#include <algorithm>
#include <vector>

namespace b2 {

static constexpr int kTG = 10;                              // guard rows in front of a block's data rows (>= 2 * largest dilation)
static constexpr int kTBR = 153;                            // rows per block: 10 + 128 + 15, and 153 = 1 (mod 8): scattered 16-byte stores spread over the banks
static constexpr int kTChunk16 = 4 * kTBR;                  // 16-byte units between two 8-channel chunks
static constexpr uint32_t kTABytes = 4u * kTChunk16 * 16u;  // 39,168 bytes per operand buffer
static constexpr uint32_t kTTapBytes = 2048;                // one tap: [32 co][32 ci] bf16
static constexpr int kTMaxTaps = 11;
static constexpr int kTGrp = 4;                             // taps per TMA box / per full-empty barrier pair
static constexpr int kTMaxGrp = (kTMaxTaps + kTGrp - 1) / kTGrp;
static constexpr uint32_t kTRingBytes = kTMaxGrp * kTGrp * kTTapBytes;      // 24,576
static constexpr int kTBars = 2 * kTMaxGrp + 4;
static constexpr uint32_t kTSmemBytes = kTRingBytes + 2 * kTABytes + kTBars * 8 + 16;
static constexpr int kTStageLd = 36;                        // floats per staged row of the output transpose

struct RbtParams {
    const float *x;          // [W][T][32] fp32
    const float *acc_src;    // optional fp32 [W][T][32] added to the result (MRF sum); may alias out32
    float *out32;
    __nv_bfloat16 *outb;
    const float *post_w;     // EPI 5: conv_post weights [7][32] fp32 and bias [1] (device), output audio [W][T] fp32
    const float *post_b;
    float *audio;
    float slope, outb_slope, div, rdiv;
    int W, T, taps, H, V, S, tiles_per_win;
    int dil[3], off[3], lim[3];       // conv1 of pair i reads rows [off, off + lim) of the slab through the mapping of dil[i]
    unsigned mdiv[3];                 // ceil(2^20 / dil[i])
    unsigned long long m_tpw;
    // the extended-tap loop of the MMA thread, tabulated on the host (one entry per conv and step, jp = taps + 2 - step): everything the issuing
    // thread needs is ONE uniform load away.  Computed in the loop (min / max / shifts of the step index) the compiler left the uniform datapath
    // and every tcgen05.mma dragged seven R2UR moves behind it (~200 cycles per MMA, measured).
    //   x: A row offset (16-byte units): block * kTBR + kTG + a * d      y: B window start: first slot * (tap bytes / 16)
    //   z: accumulator column of the N sub-range | (group to wait for + 1) << 8 | (group to hand back + 1) << 12      w: instruction descriptor
    int nsteps, ngroups;
    uint4 st[6][kTMaxTaps + 4];
    // UP: the stage's upsampler computed in place of the slab load (x never goes through HBM): its bf16 input [W][up_T][64] (already
    // leaky-ReLU'd by its producer), up_T = T / 4, and its bias per output channel
    const __nv_bfloat16 *up_in;
    int up_T;
    float up_bias[32];
    float bias1[96];                  // conv1 biases
    float cbias[96];                  // running sums of the conv2 biases
};

__device__ __forceinline__ void rbt_tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]),
          "r"(v[8]), "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15]),
          "r"(v[16]), "r"(v[17]), "r"(v[18]), "r"(v[19]), "r"(v[20]), "r"(v[21]), "r"(v[22]), "r"(v[23]),
          "r"(v[24]), "r"(v[25]), "r"(v[26]), "r"(v[27]), "r"(v[28]), "r"(v[29]), "r"(v[30]), "r"(v[31])
        : "memory");
}

__device__ __forceinline__ unsigned long long rbt_pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}

// slab row r under the mapping (d, off, lim): index (in 16-byte units, inside 8-channel chunk 0) of its operand row, or -1 when the
// mapping does not hold the row (it then lies in the halo zone that is already invalid, or outside the slab)
__device__ __forceinline__ int rbt_map(int r, int d, unsigned md, int off, int lim) {
    const int rr = r - off;
    if ((unsigned)rr >= (unsigned)lim) return -1;
    const int u = (int)(((unsigned)rr * md) >> 20);
    const int rho = rr - u * d;
    return (u & 3) * kTBR + kTG + (u >> 2) * d + rho;
}

// 32 channels of one time step -> bf16(lrelu(v (+ bias))) (zeros when !keep) at operand row `row16` (all four 8-channel chunks).
// slope is in (0, 1): leaky_relu(v) == max(v, slope * v).  Bias add and slope multiply on packed pairs (add/mul.rn.f32x2: same IEEE results).
template <bool BIAS>
__device__ __forceinline__ void rbt_operand_row(uint32_t a_u32, int row16, const uint32_t (&v)[32], const float (&bias)[32], float slope, bool keep) {
    const unsigned long long slope2 = rbt_pack2(slope, slope);
    const bool all_keep = __all_sync(0xffffffffu, keep);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        uint32_t pk[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const int c = 8 * i + 2 * e;
            unsigned long long x2 = rbt_pack2(__uint_as_float(v[c]), __uint_as_float(v[c + 1]));
            if (BIAS) asm("add.rn.f32x2 %0, %1, %2;" : "=l"(x2) : "l"(x2), "l"(rbt_pack2(bias[c], bias[c + 1])));
            unsigned long long m2;
            asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(m2) : "l"(x2), "l"(slope2));
            float v0, v1, m0, m1;
            asm("mov.b64 {%0, %1}, %2;" : "=f"(v0), "=f"(v1) : "l"(x2));
            asm("mov.b64 {%0, %1}, %2;" : "=f"(m0), "=f"(m1) : "l"(m2));
            __nv_bfloat162 h2 = __floats2bfloat162_rn(fmaxf(v0, m0), fmaxf(v1, m1));
            pk[e] = *reinterpret_cast<uint32_t *>(&h2);
        }
        if (!all_keep) {
#pragma unroll
            for (int e = 0; e < 4; e++) pk[e] = keep ? pk[e] : 0u;
        }
        if (row16 >= 0) {
            const uint32_t dst = a_u32 + (uint32_t)((i * kTChunk16 + row16) * 16);
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
        }
    }
}

// predicated 16-byte stores: the row loops of the final epilogues stay branch-free (with `if (row is an output) { load; ...; store; }` the
// compiler emitted a divergent branch and a load -> store round trip per row, one after the other: ~1.4k cycles per 32-row piece, measured)
__device__ __forceinline__ void rbt_stg_v4(float *ptr, const float4 &v, bool pred) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %5, 0;\n\t@p st.global.v4.f32 [%0], {%1, %2, %3, %4};\n\t}"
                 ::"l"(ptr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w), "r"((int)pred) : "memory");
}
__device__ __forceinline__ void rbt_stg_v2(void *ptr, uint32_t a, uint32_t b, bool pred) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %3, 0;\n\t@p st.global.v2.b32 [%0], {%1, %2};\n\t}" ::"l"(ptr), "r"(a), "r"(b), "r"((int)pred) : "memory");
}
__device__ __forceinline__ void rbt_sts_v4(uint32_t addr, float a, float b, float c, float d, bool pred) {
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %5, 0;\n\t@p st.shared.v4.f32 [%0], {%1, %2, %3, %4};\n\t}" ::"r"(addr), "f"(a), "f"(b), "f"(c), "f"(d), "r"((int)pred));
}

// this warp's operand rows (and TMEM accesses) of the phase are done: publish them to the MMA thread (one arrival per warp)
__device__ __forceinline__ void rbt_publish(uint32_t bar, int lane) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");          // generic-proxy writes -> UMMA (async proxy) reads
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncwarp();
    if (lane == 0) mbar_arrive(bar);
}

// The extended-tap loop of ONE conv for a compile-time tap count, fully unrolled: block, row multiple, slot window, column sub-range and N of
// every step are constants, so a step is two tcgen05.mma whose descriptors are a uniform base plus an immediate (plus a multiple of the
// run-time dilation) -- no table loads, no R2UR moves in front of the MMAs.  (The table-driven loop below serves the other tap counts; with
// it one thread issued an MMA every ~135 cycles, twice what the tensor pipe needs for N = 128.)
template <int K>
__device__ __forceinline__ void rbt_issue_conv(uint64_t adesc_c, uint64_t bdesc0, uint32_t acc_base, int d, uint32_t wpar, uint32_t bar_full0, uint32_t bar_empty0) {
    constexpr int half = (K - 1) / 2;
    const uint32_t idesc0 = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 4) << 24);
#pragma unroll
    for (int s = 0; s < K + 3; s++) {
        const int jp = K + 2 - s;
        const int rlo = jp - (K - 1) > 0 ? jp - (K - 1) : 0, rhi = jp < 3 ? jp : 3;
        const int qlo = K - 1 - jp + rlo, qhi = K - 1 - jp + rhi;
        const int e = jp - half, a = (e >= 0) ? e / 4 : -((-e + 3) / 4), bq = e - 4 * a;
        const int pjp = jp + 1, prhi = pjp < 3 ? pjp : 3, pqhi = (s == 0) ? -1 : K - 1 - pjp + prhi;          // previous step's window end
        const int njp = jp - 1, nqlo = jp > 0 ? (K - 1 - njp + (njp - (K - 1) > 0 ? njp - (K - 1) : 0)) : K;   // next step's window start
        if (qhi > pqhi && qhi % kTGrp == 0) mbar_wait(bar_full0 + 8u * (uint32_t)(qhi / kTGrp), wpar);
        const uint64_t ad = adesc_c + (uint64_t)(uint32_t)(bq * kTBR + kTG + a * d);
        const uint64_t bd = bdesc0 + (uint64_t)(uint32_t)(qlo * (int)(kTTapBytes >> 4));
        const uint32_t tacc = acc_base + (uint32_t)(rlo * 32);
        const uint32_t idesc = idesc0 | ((uint32_t)((rhi - rlo + 1) * 4) << 17);
        umma_f16(tacc, ad, bd, idesc, 1u);
        umma_f16(tacc, ad + (uint64_t)(uint32_t)(2 * kTChunk16), bd + 2ull, idesc, 1u);
        if (nqlo > qlo && (nqlo % kTGrp == 0 || nqlo == K)) umma_commit(bar_empty0 + 8u * (uint32_t)(qlo / kTGrp));
    }
}

static constexpr int kRbtDbgEvents = 32, kRbtDbgCtas = 4096;
#define RBT_DBG(k) do { if (DBG && dbg && blockIdx.x < kRbtDbgCtas) dbg[(size_t)blockIdx.x * kRbtDbgEvents + (k)] = clock64(); } while (0)

// EPI: 0 out32 = r;  1 out32 = acc + r;  2 outb = bf16(lrelu((acc + r) / div));  3 out32 = (acc + r) / div;  4 decided at run time;
// 5 the vocoder's last step fused in: audio = tanh(conv_post(lrelu((acc + r) / div, 0.01))), nothing else written.
// UP: x = upsampler(up_in) is computed by this kernel (ConvTranspose1d k8 s4 p2, 64 -> 32 channels, restated as a 3-tap conv with 4 x 32
// outputs per input time step, tail.cu:pack_convT): output times 4t..4t+3 of input step t are exactly accumulator row m = t - t_base/4 in X's
// layout, so the upsampler is twelve more MMAs into X (pre-loaded with its bias) on a 17 KB operand instead of a 64 KB fp32 slab load, and
// the separate upsampler launch with its 1.6 GB round trip through HBM disappears.  Needs t_base = 0 (mod 4): the plan rounds H and V.
template <int EPI, bool DBG, bool UP>
__global__ void __launch_bounds__(192, 2) k_resblock_t(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_up,
                                                       const __grid_constant__ RbtParams p, unsigned long long *dbg) {
    extern __shared__ __align__(1024) uint8_t smem[];
    pdl_trigger();
    constexpr int C = 32;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint8_t *sW = smem;
    uint8_t *sA1 = smem + kTRingBytes;
    uint8_t *sA2 = sA1 + kTABytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sA2 + kTABytes);
    // barriers: [0,3) w_full[g]  [3,6) w_empty[g]  6 a1_ready  7 t1_full  8 a2_ready  9 x_full
    const uint32_t bar0 = smem_u32(bars);
#define W_FULL(g) (bar0 + 8u * (uint32_t)(g))
#define W_EMPTY(g) (bar0 + 8u * (uint32_t)(kTMaxGrp + (g)))
#define A1_READY (bar0 + 8u * (uint32_t)(2 * kTMaxGrp))
#define T1_FULL (bar0 + 8u * (uint32_t)(2 * kTMaxGrp + 1))
#define A2_READY (bar0 + 8u * (uint32_t)(2 * kTMaxGrp + 2))
#define X_FULL (bar0 + 8u * (uint32_t)(2 * kTMaxGrp + 3))
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + kTBars);

    const int w = fdiv(blockIdx.x, p.m_tpw);
    const int tile = blockIdx.x - w * p.tiles_per_win;
    const int t_base = tile * p.V - p.H;               // time of slab row 0
    const int S = p.S;
    if (threadIdx.x == 0) RBT_DBG(0);

    // the slab's x rows start their way from HBM into L2 before anything else: one 128-byte line per row
    if (!UP && warp < 4) {
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int r = 4 * (int)threadIdx.x + q, t = t_base + r;
            if (r < S && t >= 0 && t < p.T) {
                const size_t off = ((size_t)w * p.T + t) * C;
                asm volatile("prefetch.global.L2 [%0];" ::"l"(p.x + off));
            }
        }
    }
    // ---- prologue
    if (warp == 4) {
        if (lane == 0) {
            if (smem_u32(smem) & 1023u) __trap();
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w) : "memory");
            if (UP) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_up) : "memory");
            for (int g = 0; g < kTMaxGrp; g++) { mbar_init(W_FULL(g), 1); mbar_init(W_EMPTY(g), 1); }
            mbar_init(A1_READY, 4); mbar_init(T1_FULL, 1); mbar_init(A2_READY, 4); mbar_init(X_FULL, 1);
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(256u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    // The operand buffers are NOT cleared: every row a valid output reads is written by an epilogue first (rows outside the window as zeros);
    // guard rows and rows the current mapping does not hold are only ever read on behalf of outputs the halo has already invalidated, and
    // whatever they contain (NaN bit patterns included) stays in those rows -- an accumulator row depends on its own operand rows only.
    // tests/test_resblock_t_model.py runs the index-exact model with NaN-filled buffers to pin this.  (-DB2_RBT_ZERO_INIT clears them.)
#ifdef B2_RBT_ZERO_INIT
    {
        const uint32_t a1 = smem_u32(sA1);
        for (uint32_t q = threadIdx.x; q < 2u * kTABytes / 16u; q += 192u)
            asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(a1 + q * 16u), "r"(0u) : "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
#endif
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_X = *tmem_slot;
    const uint32_t tmem_T1 = tmem_X + 128u;
    if (threadIdx.x == 0) RBT_DBG(1);
    // PDL: everything above ran while the previous kernel drained; its output (x, the MRF partial sum) is only touched by the epilogue warps
    if (warp < 4) pdl_wait();

    if (warp < 4) {
        // ======================================================================================= slab load + epilogues
        const int m = warp * 32 + lane;                        // TMEM lane == accumulator row
        const uint32_t tm_lane = (uint32_t)(warp * 32) << 16;
        const uint32_t a1_u32 = smem_u32(sA1), a2_u32 = smem_u32(sA2);
        uint32_t inside_mask = 0;                              // bit q: row 4m + q of the slab exists and lies inside the window
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int r = 4 * m + q, t = t_base + r;
            inside_mask |= (r < S && t >= 0 && t < p.T) ? (1u << q) : 0u;
        }
        const int sub_r = lane >> 3, c4 = lane & 7;

        if constexpr (UP) {
            // ---- the upsampler's operand: input steps [t_base/4 - 1, t_base/4 + 129) x 64 channels, [ci/8][row][8 ch] in A2 (rows 16 bytes
            // apart: its three taps are row offsets 0 / 1 / 2); steps outside the window are the transposed conv's zero padding
            const int t0 = t_base >> 2;                            // t_base is a multiple of 4 (possibly negative)
            for (int idx = (int)threadIdx.x; idx < 130 * 8; idx += 128) {
                const int row = idx >> 3, ch = idx & 7, tin = t0 - 1 + row;
                const bool ok = tin >= 0 && tin < p.up_T;
                const __nv_bfloat16 *src = ok ? p.up_in + ((size_t)w * p.up_T + tin) * 64 + ch * 8 : p.up_in;
                cp_async16(a2_u32 + (uint32_t)((ch * 130 + row) * 16), src, ok ? 16u : 0u);
            }
            asm volatile("cp.async.commit_group;" ::: "memory");
            {
                // X <- the upsampler's bias, T1 <- conv1's bias: both accumulators are pre-loaded, every MMA accumulates
#pragma unroll 1
                for (int which = 0; which < 2; which++) {
                    const float *bsrc = which ? p.bias1 : p.up_bias;
                    const uint32_t dstc = which ? tmem_T1 : tmem_X;
                    uint32_t bv[32];
#pragma unroll
                    for (int c = 0; c < 32; c++) bv[c] = __float_as_uint(bsrc[c]);
#pragma unroll 1
                    for (int q = 0; q < 4; q++) rbt_tmem_st32(dstc + tm_lane + (uint32_t)(q * 32), bv);
                }
            }
            asm volatile("cp.async.wait_group 0;" ::: "memory");
            asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
            rbt_publish(A2_READY, lane);
            // ---- x (X, after the upsampler's MMAs) -> lrelu -> A1 in the first conv's mapping
            const int d0 = p.dil[0], off0 = p.off[0], lim0 = p.lim[0];
            const unsigned md0 = p.mdiv[0];
            const float nob[32] = {};
            mbar_wait(X_FULL, 0u);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll 1
            for (int q = 0; q < 4; q++) {
                uint32_t acc[32];
                tmem_ld32(tmem_X + tm_lane + (uint32_t)(q * 32), acc);
                rbt_operand_row<false>(a1_u32, rbt_map(4 * m + q, d0, md0, off0, lim0), acc, nob, p.slope, ((inside_mask >> q) & 1u) != 0u);
            }
            rbt_publish(A1_READY, lane);
        } else {
        // ---- x -> X (TMEM), conv1's bias -> T1, lrelu(x) -> A1 in the first conv's mapping.  Global memory is read coalesced (8 lanes per 128
            // contiguous bytes of a row, one 32x32 piece ahead) and turned into the lane-owns-a-row order by a per-warp transpose through shared
            // memory (A2 is free until the first epilogue).  Piece q = rows 4m + q of this warp's 32 accumulator rows.
            {
                const uint32_t stg_u32 = a2_u32 + (uint32_t)warp * 8192u;
                const float *xw = p.x + ((size_t)w * p.T + t_base) * C + c4 * 4;      // row 0 of the slab (may lie before the window: only dereferenced when ok)
                auto issue_piece = [&](int q) {
                    const uint32_t dst0 = stg_u32 + (uint32_t)((q & 1) * 4096);
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const int row = j * 4 + sub_r;                                // staged row == lane that will own it
                        const int r = 4 * (warp * 32 + row) + q, t = t_base + r;
                        const bool ok = r < S && t >= 0 && t < p.T;
                        const float *src = ok ? xw + (ptrdiff_t)r * C : p.x;
                        cp_async16(dst0 + (uint32_t)(row * 128 + ((c4 ^ (row & 7)) << 4)), src, ok ? 16u : 0u);     // zero-fill outside the window
                    }
                    asm volatile("cp.async.commit_group;" ::: "memory");
                };
                issue_piece(0);
                {
                    uint32_t b1[32];
#pragma unroll
                    for (int c = 0; c < 32; c++) b1[c] = __float_as_uint(p.bias1[c]);
#pragma unroll
                    for (int q = 0; q < 4; q++) rbt_tmem_st32(tmem_T1 + tm_lane + (uint32_t)(q * 32), b1);
                }
                const int d0 = p.dil[0], off0 = p.off[0], lim0 = p.lim[0];
                const unsigned md0 = p.mdiv[0];
                const float nob[32] = {};
#pragma unroll 1
                for (int q = 0; q < 4; q++) {
                    if (q + 1 < 4) {
                        issue_piece(q + 1);
                        asm volatile("cp.async.wait_group 1;" ::: "memory");
                    } else {
                        asm volatile("cp.async.wait_group 0;" ::: "memory");
                    }
                    __syncwarp();
                    uint32_t v[32];
                    {
                        const uint32_t src0 = stg_u32 + (uint32_t)((q & 1) * 4096) + (uint32_t)(lane * 128);
#pragma unroll
                        for (int j = 0; j < 8; j++)
                            asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v[4 * j]), "=r"(v[4 * j + 1]), "=r"(v[4 * j + 2]), "=r"(v[4 * j + 3])
                                         : "r"(src0 + (uint32_t)((j ^ (lane & 7)) << 4)) : "memory");
                    }
                    __syncwarp();                  // the buffer is refilled two pieces later
                    rbt_tmem_st32(tmem_X + tm_lane + (uint32_t)(q * 32), v);
                    rbt_operand_row<false>(a1_u32, rbt_map(4 * m + q, d0, md0, off0, lim0), v, nob, p.slope, ((inside_mask >> q) & 1u) != 0u);
                }
                asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                rbt_publish(A1_READY, lane);
            }
            // every warp's staging area lies in rows of A2 that OTHER warps write in epilogue 1: nobody starts it before all are done
            asm volatile("bar.sync 1, 128;" ::: "memory");
        }
        if (threadIdx.x == 0) RBT_DBG(2);

#pragma unroll 1
        // (UP: A2_READY and X_FULL have completed once more -- the upsampler's operand and its MMAs -- so their parities are flipped)
        constexpr uint32_t xph = UP ? 1u : 0u;
        for (int i = 0; i < 3; i++) {
            const uint32_t par = (uint32_t)(i & 1);
            if (i == 2 && p.acc_src) {
                // the MRF partial sum of the output rows: into L2 NOW, two convs (~5k cycles) before the final epilogue reads it.  Requested at CTA
                // start (30-45k cycles ahead) the lines were gone again by the time they were needed -- the final epilogue ran at HBM latency with
                // 16 KB in flight per CTA, 6-9k cycles for 56 KB (phase timestamps, profiles/).
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const int r = 4 * m + q, t = t_base + r;
                    if (r + 3 >= p.H && r < p.H + p.V + 3 && r < S && t >= 0 && t < p.T)
                        asm volatile("prefetch.global.L2 [%0];" ::"l"(p.acc_src + ((size_t)w * p.T + t) * C));
                }
            }
            {
                // ---- epilogue 1: T1 (conv1 + b1, in the mapping of dil[i]) -> lrelu -> A2 in conv2's mapping (dilation 1); T1 <- conv1's bias of the next pair
                const int d = p.dil[i], off = p.off[i], lim = p.lim[i];
                const int v = (int)(((unsigned)m * p.mdiv[i]) >> 20), rho = m - v * d;
                uint32_t b1[32];
                if (i < 2) {
#pragma unroll
                    for (int c = 0; c < 32; c++) b1[c] = __float_as_uint(p.bias1[(i + 1) * 32 + c]);
                }
                const float nob[32] = {};
                mbar_wait(T1_FULL, par);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (threadIdx.x == 0) RBT_DBG(3 + 4 * i);
#pragma unroll 1
                for (int q = 0; q < 4; q++) {
                    uint32_t acc[32];
                    tmem_ld32(tmem_T1 + tm_lane + (uint32_t)(q * 32), acc);
                    if (i < 2) rbt_tmem_st32(tmem_T1 + tm_lane + (uint32_t)(q * 32), b1);
                    const int rr = d * (4 * v + q) + rho, r = rr + off, t = t_base + r;
                    const bool valid = rr < lim;
                    const int row16 = valid ? ((r & 3) * kTBR + kTG + (r >> 2)) : -1;
                    rbt_operand_row<false>(a2_u32, row16, acc, nob, p.slope, valid && t >= 0 && t < p.T);
                }
                if (i < 2) asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                rbt_publish(A2_READY, lane);
                if (threadIdx.x == 0) RBT_DBG(4 + 4 * i);
            }
            if (i < 2) {
                // ---- epilogue 2: X (+ running conv2 bias) -> lrelu -> A1 in the mapping of the next pair's conv1
                const int d = p.dil[i + 1], off = p.off[i + 1], lim = p.lim[i + 1];
                const unsigned md = p.mdiv[i + 1];
                float cb[32];
#pragma unroll
                for (int c = 0; c < 32; c++) cb[c] = p.cbias[i * 32 + c];
                mbar_wait(X_FULL, par ^ xph);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                if (threadIdx.x == 0) RBT_DBG(5 + 4 * i);
#pragma unroll 1
                for (int q = 0; q < 4; q++) {
                    uint32_t acc[32];
                    tmem_ld32(tmem_X + tm_lane + (uint32_t)(q * 32), acc);
                    rbt_operand_row<true>(a1_u32, rbt_map(4 * m + q, d, md, off, lim), acc, cb, p.slope, ((inside_mask >> q) & 1u) != 0u);
                }
                rbt_publish(A1_READY, lane);
                if (threadIdx.x == 0) RBT_DBG(6 + 4 * i);
            }
        }
        // ---- the result: X + cbias[2]
        if constexpr (EPI == 5) {
            // last ResBlock of the vocoder: MRF mean -> lrelu(0.01) -> conv_post (32 -> 1, 7 taps) -> tanh, in place of writing the fp32 mean and
            // reading it back (modeling_speecht5.py:3074-3078).  Every MMA of the CTA is complete: the S x 32 fp32 slab V is laid over the weight
            // ring and the operand buffers (rows of 128 bytes, 16-byte pieces XOR-ed with row & 7), the conv_post weights behind it.
            const uint32_t v_u32 = smem_u32(smem);
            float *wp = reinterpret_cast<float *>(smem + 65536);
            // the MRF partial sum of the rows conv_post reads, 8 lanes per row, kPB rows per thread and batch; the first batch is requested before
            // the last conv2 has finished (it does not depend on it)
            const int r_lo = max(0, p.H - 3), r_hi = min(S, p.H + p.V + 3);
            const float *aq = p.acc_src + ((size_t)w * p.T + t_base) * C + c4 * 4;
            auto ld_row = [&](int r) {
                const int t = t_base + r;
                return (r < r_hi && t >= 0 && t < p.T) ? *reinterpret_cast<const float4 *>(aq + (ptrdiff_t)r * C) : make_float4(0.f, 0.f, 0.f, 0.f);
            };
            constexpr int kPB = 13;                      // rows per thread and batch: two batches cover the 390 rows of a k = 11 slab
            float4 pa[kPB];
            const int rb0 = r_lo + ((int)threadIdx.x >> 3);
#pragma unroll
            for (int u = 0; u < kPB; u++) pa[u] = ld_row(rb0 + 16 * u);
            mbar_wait(X_FULL, xph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (threadIdx.x == 0) RBT_DBG(13);
            for (int q = threadIdx.x; q < 7 * 32; q += 128) wp[q] = __ldg(p.post_w + q);
            // pass A (lane owns four rows): X + running bias -> V
#pragma unroll 1
            for (int q = 0; q < 4; q++) {
                uint32_t a32[32];
                tmem_ld32(tmem_X + tm_lane + (uint32_t)(q * 32), a32);
                const float *cb = p.cbias + 2 * C;
                const int r = 4 * m + q;
                if (r < S) {
#pragma unroll
                    for (int j = 0; j < 8; j++) {
                        const uint32_t dst = v_u32 + (uint32_t)(r * 128 + ((j ^ ((r >> 2) & 7)) << 4));
                        asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "f"(__uint_as_float(a32[4 * j]) + cb[4 * j]),
                                     "f"(__uint_as_float(a32[4 * j + 1]) + cb[4 * j + 1]), "f"(__uint_as_float(a32[4 * j + 2]) + cb[4 * j + 2]),
                                     "f"(__uint_as_float(a32[4 * j + 3]) + cb[4 * j + 3]) : "memory");
                    }
                }
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (threadIdx.x == 0) RBT_DBG(28);
            // pass B (8 lanes per row, coalesced): + MRF partial sum, mean, lrelu(0.01), zero outside the window; only the rows conv_post reads.
            // The next batch's partial sums are requested row by row as the current batch's registers are consumed.
            {
                const float rcp = p.rdiv, nd = -p.div;
#pragma unroll 1
                for (int rb = rb0; rb < r_hi; rb += 16 * kPB) {
#pragma unroll
                    for (int u = 0; u < kPB; u++) {
                        const int r = rb + 16 * u, t = t_base + r;
                        const float4 a4 = pa[u];
                        pa[u] = ld_row(r + 16 * kPB);
                        // (no memory clobber on the accesses of V in passes B and C: rows are independent, a row's store depends on its load
                        // through the data, and volatile asm statements keep their order against the named barriers around the passes.  Rows
                        // past r_hi are read (inside the CTA's shared memory) but not written.)
                        const bool in = t >= 0 && t < p.T;
                        const uint32_t a = v_u32 + (uint32_t)(r * 128 + ((c4 ^ ((r >> 2) & 7)) << 4));
                        float4 v;
                        asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
                        float o[4] = {a4.x + v.x, a4.y + v.y, a4.z + v.z, a4.w + v.w};
#pragma unroll
                        for (int e = 0; e < 4; e++) {
                            const float q0 = o[e] * rcp;
                            const float mm = fmaf(fmaf(nd, q0, o[e]), rcp, q0);       // (acc + r) / 3: reciprocal multiply + one Newton correction
                            o[e] = in ? fmaxf(mm, 0.01f * mm) : 0.0f;
                        }
                        rbt_sts_v4(a, o[0], o[1], o[2], o[3], r < r_hi);
                    }
                }
            }
            asm volatile("bar.sync 1, 128;" ::: "memory");
            if (threadIdx.x == 0) RBT_DBG(29);
            // pass C: FOUR consecutive output samples per thread (V <= 512 - 2H: at most 128 threads' worth), channel-chunk-major.  The four
            // outputs share their input rows: 10 row reads per 4 outputs instead of 28 -- shared-memory bandwidth is what the co-resident CTA's
            // MMAs live on.  Lanes read rows four apart, which the (row >> 2) swizzle of V spreads over all banks.
            {
                const float pb = __ldg(p.post_b);
                const int r0 = p.H + 4 * (int)threadIdx.x;
                if (r0 < p.H + p.V) {
                    float acc[4] = {pb, pb, pb, pb};
#pragma unroll 1
                    for (int ch = 0; ch < 8; ch++) {
                        float4 wv[7];
#pragma unroll
                        for (int j = 0; j < 7; j++) wv[j] = *reinterpret_cast<const float4 *>(wp + j * 32 + ch * 4);
#pragma unroll
                        for (int ri = 0; ri < 10; ri++) {
                            const int rr = r0 - 3 + ri;
                            float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
                            if ((unsigned)rr < (unsigned)S)                              // outside the slab == outside the window here
                                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w)
                                             : "r"(v_u32 + (uint32_t)(rr * 128 + ((ch ^ ((rr >> 2) & 7)) << 4))));
#pragma unroll
                            for (int o = 0; o < 4; o++) {
                                const int j = ri - o;
                                if (j >= 0 && j < 7) {
                                    acc[o] = fmaf(wv[j].x, x.x, acc[o]); acc[o] = fmaf(wv[j].y, x.y, acc[o]);
                                    acc[o] = fmaf(wv[j].z, x.z, acc[o]); acc[o] = fmaf(wv[j].w, x.w, acc[o]);
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int o = 0; o < 4; o++) {
                        const int r = r0 + o, t = t_base + r;
                        if (r < p.H + p.V && t < p.T) p.audio[(size_t)w * p.T + t] = tanhf(acc[o]);
                    }
                }
            }
        } else {
            // rows [H, H+V) leave through a per-warp transpose (A1 is dead: every conv has retired), 8 lanes per 128 contiguous bytes of an
            // output row.  The MRF partial sum (acc_src) is read in that same coalesced order, one piece ahead.
            float *stg = reinterpret_cast<float *>(sA1) + warp * 32 * kTStageLd;
            const bool has_acc = (EPI == 4) ? (p.acc_src != nullptr) : (EPI >= 1);
            const bool has_div = (EPI == 4) ? (p.div != 1.0f) : (EPI >= 2);
            const bool has_o32 = (EPI == 4) ? (p.out32 != nullptr) : (EPI != 2);
            const bool has_ob = (EPI == 4) ? (p.outb != nullptr) : (EPI == 2);
            const size_t row0 = (size_t)w * p.T + t_base;                          // global row of slab row 0 (only used for rows inside the window)
            auto is_out = [&](int q, int j) {
                const int r = 4 * (warp * 32 + j * 4 + sub_r) + q;
                return r >= p.H && r < p.H + p.V && t_base + r < p.T;
            };
            auto ld_acc = [&](int q, float4 (&b)[8]) {
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int r = 4 * (warp * 32 + j * 4 + sub_r) + q;
                    b[j] = is_out(q, j) ? *reinterpret_cast<const float4 *>(p.acc_src + (row0 + r) * C + c4 * 4) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
            };
            float4 accA[8], accB[8];
            if (has_acc) ld_acc(0, accA);                 // requested before the last conv2 has finished
            mbar_wait(X_FULL, xph);
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            if (threadIdx.x == 0) RBT_DBG(13);
            const float rcp = p.rdiv, nd = -p.div;
            // one 32-column piece: X + running bias -> staging -> (8 lanes per row) + partial sum, mean, store.  `cur` holds this piece's partial
            // sums, the next piece's are requested into `nxt` while this one is worked on; the two buffers swap roles from piece to piece (a copy
            // from one into the other would wait for the loads at the end of every piece: ~1k cycles of L2 latency, measured)
            auto piece = [&](int q, float4 (&cur)[8], float4 (&nxt)[8]) {
                {
                    uint32_t a32[32];
                    tmem_ld32(tmem_X + tm_lane + (uint32_t)(q * 32), a32);
                    const float *cb = p.cbias + 2 * C;
#pragma unroll
                    for (int j = 0; j < 32; j++) a32[j] = __float_as_uint(__uint_as_float(a32[j]) + cb[j]);
#pragma unroll
                    for (int j = 0; j < 8; j++)
                        *reinterpret_cast<uint4 *>(stg + lane * kTStageLd + j * 4) = make_uint4(a32[4 * j], a32[4 * j + 1], a32[4 * j + 2], a32[4 * j + 3]);
                }
                __syncwarp();
                if (has_acc && q + 1 < 4) ld_acc(q + 1, nxt);
                float4 v[8];
#pragma unroll
                for (int j = 0; j < 8; j++) v[j] = *reinterpret_cast<const float4 *>(stg + (j * 4 + sub_r) * kTStageLd + c4 * 4);
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    if (has_acc) { v[j].x = cur[j].x + v[j].x; v[j].y = cur[j].y + v[j].y; v[j].z = cur[j].z + v[j].z; v[j].w = cur[j].w + v[j].w; }
                    if (has_div) {
                        float q0;
                        q0 = v[j].x * rcp; v[j].x = fmaf(fmaf(nd, q0, v[j].x), rcp, q0);
                        q0 = v[j].y * rcp; v[j].y = fmaf(fmaf(nd, q0, v[j].y), rcp, q0);
                        q0 = v[j].z * rcp; v[j].z = fmaf(fmaf(nd, q0, v[j].z), rcp, q0);
                        q0 = v[j].w * rcp; v[j].w = fmaf(fmaf(nd, q0, v[j].w), rcp, q0);
                    }
                    const int r = 4 * (warp * 32 + j * 4 + sub_r) + q;
                    const bool out = is_out(q, j);
                    const size_t o = out ? (row0 + r) * C + (size_t)(c4 * 4) : 0;
                    if (has_o32) rbt_stg_v4(p.out32 + o, v[j], out);
                    if (has_ob) {
                        __nv_bfloat162 h0 = __floats2bfloat162_rn(lrelu_f(v[j].x, p.outb_slope), lrelu_f(v[j].y, p.outb_slope));
                        __nv_bfloat162 h1 = __floats2bfloat162_rn(lrelu_f(v[j].z, p.outb_slope), lrelu_f(v[j].w, p.outb_slope));
                        rbt_stg_v2(p.outb + o, *reinterpret_cast<uint32_t *>(&h0), *reinterpret_cast<uint32_t *>(&h1), out);
                    }
                }
                __syncwarp();
            };
#pragma unroll 1
            for (int q = 0; q < 4; q += 2) {
                piece(q, accA, accB);
                piece(q + 1, accB, accA);
            }
        }
        if (threadIdx.x == 0) RBT_DBG(14);
    } else if (warp == 4) {
        // ======================================================================================= weight ring (TMA): slot q <-> tap k-1-q of every conv,
        // four slots per box and barrier pair; a conv walks the ring exactly once, so the producer runs up to one conv ahead of the MMA thread
        if (lane == 0) {
            const int k = p.taps, ng = p.ngroups;
            if constexpr (UP) {
                // the upsampler's weights first: 3 taps x 2 halves of its 64 input channels, [128 (phase, co)][32 ci] = 8 KB each, two passes over
                // the three ring groups (an even number of passes: the conv passes keep their parities)
                for (int b = 0; b < 6; b++) {
                    const int g = b % kTMaxGrp;
                    mbar_wait(W_EMPTY(g), (uint32_t)(((b / kTMaxGrp) & 1) ^ 1));
                    mbar_expect_tx(W_FULL(g), kTGrp * kTTapBytes);
                    tma_load_3d(smem_u32(sW + (size_t)g * kTGrp * kTTapBytes), &tmap_up, W_FULL(g), (b & 1) * 32, 0, b >> 1);
                }
            }
            for (int c = 0; c < 6; c++)
                for (int g = 0; g < ng; g++) {
                    mbar_wait(W_EMPTY(g), (uint32_t)((c & 1) ^ 1));
                    mbar_expect_tx(W_FULL(g), kTGrp * kTTapBytes);
                    tma_load_3d(smem_u32(sW + (size_t)g * kTGrp * kTTapBytes), &tmap_w, W_FULL(g), 0, 0, c * k + g * kTGrp);
                }
        }
        __syncwarp();
    } else {
        // ======================================================================================= MMA issue (one elected thread, uniform datapath)
        const uint32_t tX = __shfl_sync(0xffffffffu, tmem_X, 0);
        if (elect_one()) {
            const uint64_t adesc_1 = smem_desc(smem_u32(sA1), (uint32_t)kTChunk16 * 16u, 128u, 0u);
            const uint64_t adesc_2 = smem_desc(smem_u32(sA2), (uint32_t)kTChunk16 * 16u, 128u, 0u);
            const uint64_t bdesc0 = smem_desc(smem_u32(sW), 0u, 512u, 4u);        // SWIZZLE_64B: a weight row is 32 bf16
            const int nsteps = p.nsteps, k = p.taps;
            if constexpr (UP) {
                // x = upsampler(up_in) into X: tap j of input step t = accumulator row m reads operand row m + j; tap 0 only feeds output phases
                // 0-1 (columns 0..63), tap 2 phases 2-3 (columns 64..127): N = 64 MMAs there (tail.cu:pack_convT)
                const uint64_t adesc_u = smem_desc(smem_u32(sA2), 130u * 16u, 128u, 0u);
                const uint32_t idesc0 = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 4) << 24);
                mbar_wait(A2_READY, 0u);
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
                for (int b = 0; b < 6; b++) {
                    const int tap = b >> 1, h = b & 1, g = b % kTMaxGrp;
                    mbar_wait(W_FULL(g), (uint32_t)((b / kTMaxGrp) & 1));
                    const int col = (tap == 2) ? 64 : 0, nn = (tap == 1) ? 128 : 64;
                    const uint32_t idesc = idesc0 | ((uint32_t)(nn >> 3) << 17);
                    const uint64_t bd = bdesc0 + (uint64_t)(uint32_t)(g * (int)((kTGrp * kTTapBytes) >> 4) + col * 4);      // 64 bytes per weight row
                    const uint64_t ad = adesc_u + (uint64_t)(uint32_t)(4 * h * 130 + tap);
                    umma_f16(tX + (uint32_t)col, ad, bd, idesc, 1u);
                    umma_f16(tX + (uint32_t)col, ad + (uint64_t)(uint32_t)(2 * 130), bd + 2ull, idesc, 1u);
                    umma_commit(W_EMPTY(g));
                }
                umma_commit(X_FULL);
            }
#pragma unroll 1
            for (int cidx = 0; cidx < 6; cidx++) {
                const int i = cidx >> 1, cv = cidx & 1;
                const int d = cv ? 1 : p.dil[i];
                const uint64_t adesc_c = cv ? adesc_2 : adesc_1;
                const uint32_t acc_base = cv ? tX : tX + 128u;
                const uint32_t wpar = (uint32_t)cv;                          // conv index 2i + cv: its parity
                mbar_wait(cv ? A2_READY : A1_READY, (uint32_t)(i & 1) ^ ((UP && cv) ? 1u : 0u));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                RBT_DBG(16 + 2 * cidx);
                if (k == 11) rbt_issue_conv<11>(adesc_c, bdesc0, acc_base, d, wpar, W_FULL(0), W_EMPTY(0));
                else if (k == 7) rbt_issue_conv<7>(adesc_c, bdesc0, acc_base, d, wpar, W_FULL(0), W_EMPTY(0));
                else if (k == 3) rbt_issue_conv<3>(adesc_c, bdesc0, acc_base, d, wpar, W_FULL(0), W_EMPTY(0));
                else {
#pragma unroll 1
                    for (int s = 0; s < nsteps; s++) {
                        const uint4 e = p.st[cidx][s];
                        const uint32_t wg = (e.z >> 8) & 15u, fg = (e.z >> 12) & 15u;
                        if (wg) mbar_wait(W_FULL(wg - 1u), wpar);
                        const uint64_t ad = adesc_c + (uint64_t)e.x;
                        const uint64_t bd = bdesc0 + (uint64_t)e.y;
                        const uint32_t tacc = acc_base + (e.z & 255u);
                        umma_f16(tacc, ad, bd, e.w, 1u);
                        umma_f16(tacc, ad + (uint64_t)(uint32_t)(2 * kTChunk16), bd + 2ull, e.w, 1u);
                        if (fg) umma_commit(W_EMPTY(fg - 1u));
                    }
                }
                umma_commit(cv ? X_FULL : T1_FULL);
                RBT_DBG(17 + 2 * cidx);
            }
        }
        __syncwarp();
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) RBT_DBG(15);
    if (warp == 4) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_X), "r"(256u) : "memory");
    }
}

#undef W_FULL
#undef W_EMPTY
#undef A1_READY
#undef T1_FULL
#undef A2_READY
#undef X_FULL
#undef RBT_DBG

// ---------------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// the stacked-output kernel covers C = 32 with taps and dilations whose extended taps stay inside the guard rows
bool resblock_t_supported(int C, int taps, const int dil[3]) {
    if (C != 32 || !(taps & 1) || taps < 3 || taps > kTMaxTaps) return false;
    const int half = (taps - 1) / 2, amax = std::max((half + 3) / 4, (half + 3) / 4);      // |(j' - half) div 4| <= ceil(half / 4) <= (half + 3) / 4
    for (int i = 0; i < 3; i++)
        if (dil[i] < 1 || dil[i] > 16 || amax * dil[i] > kTG) return false;
    return true;
}

// weights of the six convs with the taps of each conv in reverse order: wt[(c * k + q)][co][ci] = W_c[tap k-1-q][co][ci]
int resblock_t_pack(ResBlockPack &out, std::vector<void *> &allocs, size_t &bytes) {
    const int C = out.C, k = out.taps;
    if (!resblock_t_supported(C, k, out.dil)) return 0;                 // not an error: the time-as-M kernel runs instead
    const size_t per_tap = (size_t)C * C, total = (size_t)(6 * k + kTGrp) * per_tap;      // + zero taps: the last TMA box stays in bounds
    void *q = nullptr;
    B2_CUDA_OK(cudaMalloc(&q, total * sizeof(__nv_bfloat16)));
    allocs.push_back(q); bytes += total * sizeof(__nv_bfloat16);
    out.wt = reinterpret_cast<__nv_bfloat16 *>(q);
    B2_CUDA_OK(cudaMemset(q, 0, total * sizeof(__nv_bfloat16)));
    for (int c = 0; c < 6; c++)
        for (int j = 0; j < k; j++)
            B2_CUDA_OK(cudaMemcpy(out.wt + ((size_t)c * k + (k - 1 - j)) * per_tap, out.w + ((size_t)c * k + j) * per_tap, per_tap * sizeof(__nv_bfloat16),
                                  cudaMemcpyDeviceToDevice));
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) return set_error("cuTensorMapEncodeTiled is not available from the driver");
    CUtensorMap *tm = new CUtensorMap();
    cuuint64_t gdim[3] = {(cuuint64_t)C, (cuuint64_t)C, (cuuint64_t)(6 * k + kTGrp)};
    cuuint64_t gstr[2] = {(cuuint64_t)C * 2, (cuuint64_t)C * C * 2};
    cuuint32_t box[3] = {(cuuint32_t)C, (cuuint32_t)C, (cuuint32_t)kTGrp};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = reinterpret_cast<EncodeTiledFn>(fn)(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void *)out.wt, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                                     CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { delete tm; return set_error("resblock_t: cuTensorMapEncodeTiled failed with CUresult %d (k %d)", (int)r, k); }
    out.tmap_t = tm;
    return 0;
}

void resblock_t_free(ResBlockPack &p) {
    if (p.tmap_t) { delete reinterpret_cast<CUtensorMap *>(p.tmap_t); p.tmap_t = nullptr; }
}

// slab geometry: S rows per slab, halo H, V output rows per tile, and for every pair the row range its conv1 mapping holds
int resblock_t_plan(int k, const int dil[3], int T, bool post, int &S, int &H, int &V, int &tiles, int off[3], int lim[3], bool align4) {
    const int half = (k - 1) / 2;
    int cap[3], dsum = 0;
    for (int i = 0; i < 3; i++) {
        cap[i] = 4 * dil[i] * (128 / dil[i]);                  // rows the mapping of dil[i] can hold in 128 accumulator rows
        dsum += dil[i] + 1;
    }
    // Always tiled, also when the window is shorter than a slab: the halo rows then lie outside the window and are written as the zeros the
    // reference pads with.  (A no-halo slab would need every physical row a NEW mapping does not write cleared first: an operand buffer keeps
    // the rows of the previous pair's mapping, which are harmless only where the halo has already invalidated them.)
    H = half * dsum + (post ? 3 : 0);                          // conv_post reaches three more rows either side
    // rows closer than g_i to a slab end are already invalid when pair i starts: its mapping may drop them
    int g[3], acc = 0;
    S = 512;
    for (int i = 0; i < 3; i++) { g[i] = acc; S = std::min(S, cap[i] + 2 * g[i]); acc += half * (dil[i] + 1); }
    for (int i = 0; i < 3; i++) {
        off[i] = std::max(0, (S - cap[i] + 1) / 2);
        lim[i] = std::min(cap[i], S - off[i]);
        if (off[i] > g[i] || S - off[i] - lim[i] > g[i]) return set_error("resblock_t: no slab geometry for k=%d dil=%d", k, dil[i]);
    }
    if (align4) H = (H + 3) & ~3;          // fused upsampler: a tile starts on an input step (t_base = tile * V - H = 0 mod 4)
    const int vmax = align4 ? ((S - 2 * H) & ~3) : S - 2 * H;
    if (vmax < 64) return set_error("resblock_t: halo %d leaves no room in a %d-row slab", H, S);
    tiles = cdiv(T, vmax);
    V = cdiv(T, tiles);
    if (align4) V = (V + 3) & ~3;
    return 0;
}

static bool g_rbt_attr[64][32] = {};
static unsigned long long *g_rbt_dbg = nullptr;

template <int EPI, bool DBG, bool UP = false>
static int launch_rbt_(const CUtensorMap &tm, const RbtParams &p, unsigned grid, cudaStream_t st, const CUtensorMap *tm_up = nullptr) {
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    const int slot = EPI + (DBG ? 8 : 0) + (UP ? 16 : 0);
    if (dev < 64 && !g_rbt_attr[dev][slot]) {
        B2_CUDA_OK(cudaFuncSetAttribute(k_resblock_t<EPI, DBG, UP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTSmemBytes));
        g_rbt_attr[dev][slot] = true;
    }
    B2_CUDA_OK(launch_k(k_resblock_t<EPI, DBG, UP>, dim3(grid), dim3(192), kTSmemBytes, st, pdl_enabled(), tm, tm_up ? *tm_up : tm, p, g_rbt_dbg));
    B2_LAUNCH_OK("k_resblock_t");
    return 0;
}

int launch_resblock_t(const ResBlockArgs &a, cudaStream_t st) {
    const ResBlockPack &pk = *a.pack;
    if (!pk.tmap_t || !pk.wt) return set_error("resblock_t: weights were not packed");
    const bool post = a.audio != nullptr;
    RbtParams p;
    p.x = a.x; p.acc_src = a.acc_src; p.out32 = a.out32; p.outb = a.outb;
    p.post_w = a.post_w; p.post_b = a.post_b; p.audio = a.audio;
    p.slope = a.slope; p.outb_slope = a.outb_slope; p.div = a.div; p.rdiv = 1.0f / a.div;
    p.W = a.W; p.T = a.T; p.taps = pk.taps;
    for (int i = 0; i < 96; i++) { p.bias1[i] = pk.h_bias1[i]; p.cbias[i] = pk.h_cbias[i]; }
    for (int i = 0; i < 3; i++) { p.dil[i] = pk.dil[i]; p.mdiv[i] = (unsigned)(((1u << 20) + (unsigned)pk.dil[i] - 1u) / (unsigned)pk.dil[i]); }
    const bool up = a.up_in != nullptr;
    const CUtensorMap *tm_up = nullptr;
    p.up_in = a.up_in; p.up_T = a.T / 4;
    for (int i = 0; i < 32; i++) p.up_bias[i] = 0.0f;
    if (up) {
        const Layer *ul = a.up_layer;
        if (!ul || !ul->tmap_q || ul->Cin != 64 || ul->Cout != 128 || ul->taps != 3 || ul->h_bias.size() < 32 || (a.T & 3))
            return set_error("resblock_t: the fused upsampler needs a packed 64 -> 4 x 32 transposed conv and T = 0 (mod 4)");
        if (a.x) return set_error("resblock_t: x and up_in are exclusive");
        tm_up = reinterpret_cast<const CUtensorMap *>(ul->tmap_q);
        for (int i = 0; i < 32; i++) p.up_bias[i] = ul->h_bias[i];
    }
    if (resblock_t_plan(pk.taps, pk.dil, a.T, post, p.S, p.H, p.V, p.tiles_per_win, p.off, p.lim, up)) return 1;
    p.m_tpw = ((1ull << 40) + (unsigned long long)p.tiles_per_win - 1) / (unsigned long long)p.tiles_per_win;
    {
        // extended taps j' = k+2 .. 0: stacked outputs r' in [rlo, rhi] use tap j' - r' = slot k-1-j'+r' (taps are stored in reverse order), so
        // the B tile is the slot window [qlo, qhi]; it slides up by at most one slot per step at either end
        const int k = pk.taps, half = (k - 1) / 2;
        p.nsteps = k + 3;
        p.ngroups = (k + kTGrp - 1) / kTGrp;
        int prev_hi = -1;
        for (int s = 0; s < kTMaxTaps + 4; s++) {
            for (int c = 0; c < 6; c++) p.st[c][s] = make_uint4(0u, 0u, 0u, 0u);
            if (s >= p.nsteps) continue;
            const int jp = k + 2 - s;
            const int rlo = std::max(0, jp - (k - 1)), rhi = std::min(3, jp);
            const int qlo = k - 1 - jp + rlo, qhi = k - 1 - jp + rhi;
            const int e = jp - half, a = (e >= 0) ? e / 4 : -((-e + 3) / 4), bq = e - 4 * a;       // floor division
            const int nqlo = jp > 0 ? (k - jp + std::max(0, jp - k)) : k;      // first slot the next step still needs
            if (nqlo - qlo > 1 || qhi > prev_hi + 1 || qlo < 0 || qhi >= k) return set_error("resblock_t: slot window moves by more than one");
            // a group is waited for when the window first reaches its first slot, handed back when the window has left its last one
            const int wg = (qhi > prev_hi && qhi % kTGrp == 0) ? qhi / kTGrp + 1 : 0;
            const int fg = (nqlo > qlo && (nqlo % kTGrp == 0 || nqlo == k)) ? qlo / kTGrp + 1 : 0;
            prev_hi = std::max(prev_hi, qhi);
            // kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, M = 128, N = 32 * (rhi - rlo + 1)
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((128u >> 4) << 24) | ((uint32_t)((rhi - rlo + 1) * 4) << 17);
            for (int c = 0; c < 6; c++)
                p.st[c][s] = make_uint4((uint32_t)(bq * kTBR + kTG + a * ((c & 1) ? 1 : pk.dil[c >> 1])), (uint32_t)(qlo * (int)(kTTapBytes >> 4)),
                                        (uint32_t)(rlo * 32) | ((uint32_t)wg << 8) | ((uint32_t)fg << 12), idesc);
        }
    }
    const long long nct = (long long)a.W * p.tiles_per_win;
    if (nct >= (1ll << 24)) return set_error("resblock_t: too many tiles (%lld)", nct);
    const CUtensorMap &tm = *reinterpret_cast<const CUtensorMap *>(pk.tmap_t);
    static const bool dbg_on = getenv("B2_RB_DBG") != nullptr;
    const size_t dbg_n = (size_t)kRbtDbgCtas * kRbtDbgEvents;
    if (dbg_on) {
        if (!g_rbt_dbg) B2_CUDA_OK(cudaMalloc(&g_rbt_dbg, dbg_n * 8));
        B2_CUDA_OK(cudaMemsetAsync(g_rbt_dbg, 0, dbg_n * 8, st));
        int rc = up ? (post ? launch_rbt_<5, true, true>(tm, p, (unsigned)nct, st, tm_up) : launch_rbt_<4, true, true>(tm, p, (unsigned)nct, st, tm_up))
                    : (post ? launch_rbt_<5, true>(tm, p, (unsigned)nct, st) : launch_rbt_<4, true>(tm, p, (unsigned)nct, st));
        if (rc) return rc;
        // per-phase averages over the first CTAs of the launch (cycles of the SM clock)
        B2_CUDA_OK(cudaStreamSynchronize(st));
        static std::vector<unsigned long long> h;
        h.resize(dbg_n);
        B2_CUDA_OK(cudaMemcpy(h.data(), g_rbt_dbg, dbg_n * 8, cudaMemcpyDeviceToHost));
        const int n = (int)std::min<long long>(kRbtDbgCtas, nct);
        double ev[kRbtDbgEvents] = {0};
        int cnt = 0;
        for (int b = 0; b < n; b++) {
            const unsigned long long *r = &h[(size_t)b * kRbtDbgEvents];
            if (!r[0] || !r[15]) continue;
            cnt++;
            for (int q = 0; q < kRbtDbgEvents; q++) ev[q] += r[q] ? (double)(r[q] - r[0]) : 0.0;
        }
        if (cnt) {
            for (int q = 0; q < kRbtDbgEvents; q++) ev[q] /= cnt;
            fprintf(stderr, "[rbt dbg] k=%d T=%d S=%d H=%d V=%d ctas=%lld (avg of %d) cycles since CTA start: setup %.0f | load done %.0f | result ready %.0f | stored %.0f | end %.0f\n",
                    pk.taps, a.T, p.S, p.H, p.V, nct, cnt, ev[1], ev[2], ev[13], ev[14], ev[15]);
            if (post) fprintf(stderr, "[rbt dbg]   conv_post epilogue: pass A %.0f | pass B %.0f | pass C %.0f\n", ev[28] - ev[13], ev[29] - ev[28], ev[14] - ev[29]);
            else fprintf(stderr, "[rbt dbg]   final epilogue pieces done at +%.0f +%.0f +%.0f +%.0f\n", ev[24] - ev[13], ev[25] - ev[13], ev[26] - ev[13], ev[27] - ev[13]);
            for (int i = 0; i < 3; i++)
                fprintf(stderr, "[rbt dbg]   pair %d: conv1 issue %.0f..%.0f (%.0f) | epi1 %.0f..%.0f (%.0f) | conv2 issue %.0f..%.0f (%.0f) | epi2 %.0f..%.0f (%.0f)\n", i,
                        ev[16 + 4 * i], ev[17 + 4 * i], ev[17 + 4 * i] - ev[16 + 4 * i], ev[3 + 4 * i], ev[4 + 4 * i], ev[4 + 4 * i] - ev[3 + 4 * i],
                        ev[18 + 4 * i], ev[19 + 4 * i], ev[19 + 4 * i] - ev[18 + 4 * i], ev[5 + 4 * i], ev[6 + 4 * i], ev[6 + 4 * i] - ev[5 + 4 * i]);
        }
        return 0;
    }
    const bool acc = p.acc_src != nullptr, dv = p.div != 1.0f, o32 = p.out32 != nullptr, ob = p.outb != nullptr;
    if (up) {
        // the vocoder's three stage-3 launches: store / accumulate / accumulate-average-conv_post; anything else takes the run-time epilogue
        if (post) return launch_rbt_<5, false, true>(tm, p, (unsigned)nct, st, tm_up);
        if (!acc && !dv && o32 && !ob) return launch_rbt_<0, false, true>(tm, p, (unsigned)nct, st, tm_up);
        if (acc && !dv && o32 && !ob) return launch_rbt_<1, false, true>(tm, p, (unsigned)nct, st, tm_up);
        return launch_rbt_<4, false, true>(tm, p, (unsigned)nct, st, tm_up);
    }
    if (post) return launch_rbt_<5, false>(tm, p, (unsigned)nct, st);
    if (!acc && !dv && o32 && !ob) return launch_rbt_<0, false>(tm, p, (unsigned)nct, st);
    if (acc && !dv && o32 && !ob) return launch_rbt_<1, false>(tm, p, (unsigned)nct, st);
    if (acc && dv && !o32 && ob) return launch_rbt_<2, false>(tm, p, (unsigned)nct, st);
    if (acc && dv && o32 && !ob) return launch_rbt_<3, false>(tm, p, (unsigned)nct, st);
    return launch_rbt_<4, false>(tm, p, (unsigned)nct, st);
}

}  // namespace b2
