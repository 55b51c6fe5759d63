// One whole HiFiGAN ResBlock per launch on tcgen05 (modeling_speecht5.py:2903-2962):
//
//     for d in (d0, d1, d2):   x = x + conv2_d( lrelu( conv1_d( lrelu(x) ) ) )            six convolutions, k taps each
//
// The un-fused path (conv_umma.cu) moves ~16 bytes per element per conv pair through HBM (bf16 operands, fp32 residual
// stream in and out) and at 1,024 sessions the thin stages (C = 32, 64) are bound by exactly that traffic.  Here a CTA
// keeps a 512-row slab of one window on chip for all six convolutions:
//
//   X  (TMEM, fp32, kS x C columns)  the residual stream.  It is initialised with x by tcgen05.st, and every conv2 simply
//                                    ACCUMULATES into it (the residual add is the accumulator's own "+="); conv2's biases
//                                    are not written back but carried as a running per-channel offset added on read.
//   T1 (TMEM, fp32, kS x C columns)  conv1's accumulator.
//   A1, A2 (shared, bf16)            the operands lrelu(x) and lrelu(conv1(..)+b1) in the un-swizzled K-major interleaved UMMA
//                                    layout [channel/8][row][8 ch] (rows 16 bytes apart), so a filter tap is the same buffer
//                                    read through a descriptor advanced by j*dil rows (as in conv_umma.cu).  Each epilogue
//                                    writes the NEXT convolution's operand straight from TMEM: nothing goes back to HBM.
//   weights                          streamed by TMA in groups of `tps` taps through an mbarrier ring (they live in L2).
//
// The slab carries a halo: with buffer rows r <-> time t_base + r, every conv invalidates `pad` more rows at each end, so
// after the six convs rows [H, 512 - H) are exact, H = (k-1)/2 * (d0 + d1 + d2 + 3); tiles advance by V <= 512 - 2H rows.
// Rows outside the window are forced to zero in every operand (the reference pads each conv with zeros at the window edge).
//
// Pipelining inside a CTA is by 128-row sub-tile: the MMA warp issues   for tap group: for sub-tile: taps x K-steps   and
// commits a sub-tile's accumulator in the last group, so the epilogue of sub-tile s overlaps the MMAs of s+1..; the next
// conv starts as soon as the operand rows of its first two sub-tiles exist.  Two CTAs share an SM at C = 32.
//
// Warp roles (192 threads): 0-3 slab load + all epilogues (TMEM lanes 32*warp..), 4 TMA weight ring, 5 TMEM alloc + MMA issue.
#include "conv_umma.cuh"
#include "umma_ptx.cuh"

#include <cuda.h>
#include <stdlib.h>
#include <algorithm>
#include <vector>

namespace b2 {

static constexpr int kGuard = 26;                          // zero rows either side of the slab (>= largest pad, 5*5)
static constexpr int kRbStageLd = 36;                      // floats per staged row of the output transpose (32 + 4 pad)
static constexpr int kRbMaxC = 128;

// per-width geometry: TMEM holds X and T1 (2 * kS * C fp32 columns <= 512), so a CTA owns 4 sub-tiles up to C = 64 and 2 at C = 128
template <int C> struct RbGeom {
    static constexpr int kS = (C <= 64) ? 4 : 2;               // 128-row sub-tiles per CTA
    static constexpr int kRows = 128 * kS;                     // slab rows
    static constexpr int kRtot = kGuard + kRows + kGuard + 1;  // rows of an operand buffer (odd: K-chunks land on different banks)
    static constexpr int KB = (C >= 64) ? 64 : 32;             // K block of a weight tile (one swizzle span)
    static constexpr int NKB = C / KB;
    static constexpr uint32_t kABytes = ((uint32_t)kRtot * C * 2 + 1023u) & ~1023u;
};

struct RbParams {
    const float *x;          // [W][T][C] fp32
    const float *acc_src;    // optional fp32 [W][T][C] added to the result (MRF sum); may alias out32
    float *out32;            // optional
    __nv_bfloat16 *outb;     // optional: bf16(lrelu(result, outb_slope))
    const float *post_w;     // EPI 5: conv_post weights [7][32] fp32 and bias [1] (device), output audio [W][T] fp32
    const float *post_b;
    float *audio;
    float slope, outb_slope, div, rdiv;
    int W, T, taps, H, V, tiles_per_win, tps, ngroups, nslots;
    int dil0, dil1, dil2;
    unsigned long long m_tpw;
    unsigned long long *dbg;   // optional per-CTA phase timestamps (B2_RB_DBG analysis runs)
    float bias1[3 * kRbMaxC];  // conv1 biases                                         (constant bank: uniform loads)
    float cbias[3 * kRbMaxC];  // running sum of conv2 biases: cbias[i] = b2[0] + .. + b2[i]
};

__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&v)[32]) {
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

// 32 consecutive fp32 of one row (128 bytes) -> registers; zeros when the row is not wanted
__device__ __forceinline__ void ld_row32(const float *src, bool ok, uint32_t (&v)[32]) {
    if (ok) {
#pragma unroll
        for (int i = 0; i < 8; i++) {
            const uint4 q = __ldg(reinterpret_cast<const uint4 *>(src) + i);
            v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
        }
    } else {
#pragma unroll
        for (int i = 0; i < 32; i++) v[i] = 0u;
    }
}

// 32 consecutive channels [c0, c0+32) of buffer row r -> bf16(lrelu(v + bias)) (zeros when !keep) in the interleaved operand
// layout (RT rows per 8-channel chunk).  slope is in (0, 1), so leaky_relu(v) == max(v, slope * v).
// The bias add and the slope multiply run on packed pairs (add.rn.f32x2 / mul.rn.f32x2: the same IEEE results, half the instructions), and the
// zeroing select is skipped when every lane's row lies inside the window (warp-uniform): the conv epilogues were ~4.4 instructions per element and
// about half issue-bound with two CTAs per SM (ncu source page, round 2).
__device__ __forceinline__ unsigned long long rb_pack2(float lo, float hi) {
    unsigned long long r;
    asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
    return r;
}
template <int RT>
__device__ __forceinline__ void write_operand_row(uint32_t sA_u32, int r, int c0, const uint32_t (&v)[32], const float *bias, float slope, bool keep) {
    const unsigned long long slope2 = rb_pack2(slope, slope);
    const bool all_keep = __all_sync(0xffffffffu, keep);
#pragma unroll
    for (int i = 0; i < 4; i++) {
        uint32_t pk[4];
#pragma unroll
        for (int e = 0; e < 4; e++) {
            const int c = 8 * i + 2 * e;
            unsigned long long x2 = rb_pack2(__uint_as_float(v[c]), __uint_as_float(v[c + 1]));
            if (bias) asm("add.rn.f32x2 %0, %1, %2;" : "=l"(x2) : "l"(x2), "l"(rb_pack2(bias[c], bias[c + 1])));
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
        const uint32_t dst = sA_u32 + (uint32_t)(((((c0 >> 3) + i) * RT) + kGuard + r) * 16);
        asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(pk[0]), "r"(pk[1]), "r"(pk[2]), "r"(pk[3]) : "memory");
    }
}

// this thread's shared-memory operand writes and TMEM reads/writes are done: publish them to the MMA warps (one arrival per warp)
__device__ __forceinline__ void publish_rows(uint32_t bar, int lane) {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");          // generic-proxy writes -> UMMA (async proxy) reads
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncwarp();
    if (lane == 0) mbar_arrive(bar);
}

static constexpr int kRbDbgEvents = 48, kRbDbgCtas = 4096;
#define RB_DBG(k) do { if (DBG && p.dbg && blockIdx.x < kRbDbgCtas) p.dbg[(size_t)blockIdx.x * kRbDbgEvents + (k)] = clock64(); } while (0)

// Warp roles: [0, NEW) slab load + all epilogues (warp e: TMEM lane quadrant e % 4, column slice e / 4), warp NEW = TMEM alloc +
// TMA weight ring, then NMW MMA-issuing warps, each owning kS / NMW sub-tiles (a sub-tile's accumulator is only ever touched by
// one issuing thread, so the summation order is fixed).
// EPI selects the final epilogue at compile time (its code is a third of the kernel, and the kernel has to fit the instruction
// cache): 0 out32 = r;  1 out32 = acc + r;  2 outb = bf16(lrelu((acc + r) / div));  3 out32 = (acc + r) / div;  4 everything decided at run time;
// 5 (C = 32 only) the vocoder's last step fused in: audio = tanh(conv_post(lrelu((acc + r) / div, 0.01))), nothing else written.
template <int C, int NEW, int NMW, int EPI, bool DBG>
__global__ void __launch_bounds__((NEW + 1 + NMW) * 32) __maxnreg__((C == 32) ? 128 : 168) k_resblock(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ RbParams p) {
    extern __shared__ __align__(1024) uint8_t smem[];
    pdl_trigger();
    using G = RbGeom<C>;
    constexpr int kS = G::kS, kRows = G::kRows, kRtot = G::kRtot, KB = G::KB, NKB = G::NKB;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    constexpr int kThreads = (NEW + 1 + NMW) * 32;
    constexpr int CH = C / 32;                                  // 32-column chunks per row
    constexpr int CHW = CH / (NEW / 4);                         // ... of which one epilogue warp handles CHW
    constexpr int NCHW = kS * CHW;                              // 32x32 pieces per epilogue warp
    constexpr uint32_t kStgBytes = 8192u;                       // per-warp staging of the slab load (A2 holds NEW of them)
    constexpr int SPW = kS / NMW;                               // sub-tiles per MMA warp
    constexpr uint32_t kTapKbBytes = (uint32_t)C * KB * 2;      // one tap, one K block
    constexpr uint32_t kABytes = G::kABytes;
    static_assert(CH % (NEW / 4) == 0 && kS % NMW == 0 && 2 * kS * C <= 512 && NEW * kStgBytes <= G::kABytes, "unsupported geometry");
    const uint32_t slot_bytes = (uint32_t)p.tps * kTapKbBytes;
    uint8_t *sW = smem;
    uint8_t *sA1 = smem + (size_t)p.nslots * slot_bytes;
    uint8_t *sA2 = sA1 + kABytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sA2 + kABytes);
    // barriers: [0,4) w_full  [4,8) w_empty  [8,12) a1_ready[s]  [12,16) t1_full[s]  [16,20) a2_ready[s]  [20,24) x_full[s]
    const uint32_t bar0 = smem_u32(bars);
#define W_FULL(s) (bar0 + 8u * (uint32_t)(s))
#define W_EMPTY(s) (bar0 + 8u * (uint32_t)(4 + (s)))
#define A1_READY(s) (bar0 + 8u * (uint32_t)(8 + (s)))
#define T1_FULL(s) (bar0 + 8u * (uint32_t)(12 + (s)))
#define A2_READY(s) (bar0 + 8u * (uint32_t)(16 + (s)))
#define X_FULL(s) (bar0 + 8u * (uint32_t)(20 + (s)))
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 24);

    const int w = fdiv(blockIdx.x, p.m_tpw);
    const int tile = blockIdx.x - w * p.tiles_per_win;
    const int t_base = tile * p.V - p.H;               // time of slab row 0

    if (threadIdx.x == 0) RB_DBG(0);
    // The slab's x rows (and, for the final epilogue, the MRF partial sum's) start their way from HBM into L2 before anything else:
    // the load phase below keeps only two 4 KB pieces per warp in flight, so at HBM latency it was ~13k cycles of a 34-114k-cycle CTA
    // (phase timestamps, profiles/); out of L2 it is a few thousand.  One 128-byte line per lane per 32-channel piece.
    if (warp < NEW) {
        const int rq0 = (warp & 3) * 32 + lane, cb0 = (warp >> 2) * (CHW * 32);
#pragma unroll
        for (int s = 0; s < kS; s++) {
            const int r = s * 128 + rq0, t = t_base + r;
            if (t >= 0 && t < p.T) {
                const size_t off = ((size_t)w * p.T + t) * C + cb0;
#pragma unroll
                for (int cc = 0; cc < CHW; cc++) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.x + off + cc * 32));
                if (p.acc_src && r >= p.H && r < p.H + p.V) {
#pragma unroll
                    for (int cc = 0; cc < CHW; cc++) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.acc_src + off + cc * 32));
                }
            }
        }
    }
    // ---- prologue
    if (warp == NEW) {
        if (lane == 0) {
            if (smem_u32(smem) & 1023u) __trap();
            asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w) : "memory");
            for (int s = 0; s < 4; s++) { mbar_init(W_FULL(s), 1); mbar_init(W_EMPTY(s), NMW); }
            for (int s = 0; s < kS; s++) { mbar_init(A1_READY(s), NEW); mbar_init(T1_FULL(s), 1); mbar_init(A2_READY(s), NEW); mbar_init(X_FULL(s), 1); }
            asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        }
        __syncwarp();
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)(2 * kS * C)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    {
        // guard rows [0, kGuard) and [kGuard + kRows, kRtot) of both operand buffers
        constexpr int kGuardRows = kRtot - kRows;
        const uint32_t a1 = smem_u32(sA1), a2 = smem_u32(sA2);
        for (int q = threadIdx.x; q < kGuardRows * (C / 8); q += kThreads) {
            const int ch = q / kGuardRows, g = q - ch * kGuardRows;
            const int row = (g < kGuard) ? g : (kRows + g);
            const uint32_t off = (uint32_t)((ch * kRtot + row) * 16);
            asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(a1 + off), "r"(0u) : "memory");
            asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(a2 + off), "r"(0u) : "memory");
        }
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_X = *tmem_slot;
    const uint32_t tmem_T1 = tmem_X + (uint32_t)(kS * C);
    if (threadIdx.x == 0) RB_DBG(1);
    // PDL: barrier setup, TMEM allocation, guard rows and the L2 prefetches above ran while the previous kernel drained; its output (x, the MRF
    // partial sum) is only touched by the epilogue warps, from here on.  The weight ring (warp NEW) reads nothing a kernel writes.
    if (warp < NEW) pdl_wait();

    if (warp < NEW) {
        // ======================================================================================= slab load + epilogues
        const int quad = warp & 3;                             // TMEM lane quadrant this warp may touch
        const int cbase = (warp >> 2) * (CHW * 32);            // first column of this warp's slice
        const int rq = quad * 32 + lane;                       // row inside a sub-tile == TMEM lane
        const uint32_t tm_lane = (uint32_t)(quad * 32) << 16;
        const uint32_t a1_u32 = smem_u32(sA1), a2_u32 = smem_u32(sA2);
        uint32_t inside_mask = 0, out_mask = 0;                 // bit s: this lane's row of sub-tile s is inside the window / is an output row
#pragma unroll
        for (int s = 0; s < kS; s++) {
            const int r = s * 128 + rq, t = t_base + r;
            inside_mask |= ((t >= 0) && (t < p.T)) ? (1u << s) : 0u;
            out_mask |= (r >= p.H && r < p.H + p.V && t < p.T) ? (1u << s) : 0u;
        }
#define inside(s) (((inside_mask >> (s)) & 1u) != 0u)
#define is_out(s) (((out_mask >> (s)) & 1u) != 0u)

        // ---- x -> X (TMEM) and lrelu(x) -> A1.  Global memory is read coalesced (8 lanes per 128 contiguous bytes of a row, one
        // 32x32 piece ahead) and turned into the lane-owns-a-row order TMEM wants by a per-warp transpose through shared memory
        // (A2 is free until the first epilogue).  Row-per-lane loads cost 8x the LSU wavefronts and made this phase ~10k cycles.
        const int sub_r = lane >> 3, c4 = lane & 7;
        uint32_t inside_t[8];                                  // inside_mask of the rows this lane touches in the transposed order
#pragma unroll
        for (int j = 0; j < 8; j++) inside_t[j] = __shfl_sync(0xffffffffu, inside_mask, j * 4 + sub_r);
        {
            // two 4 KB staging buffers per warp, 128-byte rows with the 16-byte piece index XOR-ed with (row & 7): conflict-free
            // for the 8-lanes-per-row writes of cp.async and for the row-per-lane reads
            const uint32_t stg_u32 = a2_u32 + (uint32_t)warp * kStgBytes;
            const float *xq = p.x + ((size_t)w * p.T + (t_base + quad * 32 + sub_r)) * C + cbase + c4 * 4;   // row sub_r of this warp's rows in sub-tile 0
            auto issue_piece = [&](int q) {
                const int s1 = q / CHW, c1 = (q % CHW) * 32;
                const uint32_t dst0 = stg_u32 + (uint32_t)((q & 1) * 4096);
#pragma unroll
                for (int j = 0; j < 8; j++) {
                    const int row = j * 4 + sub_r;
                    const bool ok = ((inside_t[j] >> s1) & 1u) != 0u;
                    const float *src = ok ? xq + ((size_t)s1 * 128 + j * 4) * C + c1 : p.x;
                    cp_async16(dst0 + (uint32_t)(row * 128 + ((c4 ^ (row & 7)) << 4)), src, ok ? 16u : 0u);     // zero-fill outside the window
                }
                asm volatile("cp.async.commit_group;" ::: "memory");
            };
            issue_piece(0);
#pragma unroll 1
            for (int q = 0; q < NCHW; q++) {
                const int s = q / CHW, c0 = cbase + (q % CHW) * 32;
                if (q + 1 < NCHW) {
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
                tmem_st32(tmem_X + tm_lane + (uint32_t)(s * C + c0), v);
                write_operand_row<kRtot>(a1_u32, s * 128 + rq, c0, v, nullptr, p.slope, true);
                if ((q % CHW) == CHW - 1) {
                    asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
                    publish_rows(A1_READY(s), lane);
                    if (threadIdx.x == 0) RB_DBG(44 + s);
                }
            }
            // the staging area lay over guard rows of A2: zero them again (only this warp wrote there; the first conv2 reads
            // A2 after this warp's epilogue-1 publication, which comes later in program order)
            {
                constexpr int kGuardRows = kRtot - kRows;
                const uint32_t lo = (uint32_t)warp * kStgBytes, hi = lo + kStgBytes;
                for (int q = lane; q < kGuardRows * (C / 8); q += 32) {
                    const int ch = q / kGuardRows, g = q - ch * kGuardRows;
                    const int row = (g < kGuard) ? g : (kRows + g);
                    const uint32_t off = (uint32_t)((ch * kRtot + row) * 16);
                    if (off + 16 > lo && off < hi) asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(a2_u32 + off), "r"(0u) : "memory");
                }
            }
        }
        // every warp's staging area lies in rows of A2 that OTHER warps write in epilogue 1: nobody starts it before all are done
        asm volatile("bar.sync 1, %0;" ::"n"(NEW * 32) : "memory");
        if (threadIdx.x == 0) RB_DBG(2);

#pragma unroll 1
        for (int i = 0; i < 3; i++) {
            const uint32_t par = (uint32_t)(i & 1);
            // ---- epilogue 1: T1 -> lrelu(. + b1) -> A2, then (pairs 0, 1) epilogue 2: X (+ running conv2 bias) -> lrelu -> A1 of the
            // next pair.  ONE body serves both (source accumulator, bias row, destination buffer and barriers are run-time
            // values): the epilogue code is most of the kernel and has to stay small (instruction cache).
#pragma unroll 1
            for (int e = 0; e < ((i < 2) ? 2 : 1); e++) {
                const uint32_t src = (e ? tmem_X : tmem_T1) + tm_lane;
                const uint32_t dst = e ? a1_u32 : a2_u32;
                const float *bias = (e ? p.cbias : p.bias1) + i * C + cbase;
                const uint32_t full0 = e ? X_FULL(0) : T1_FULL(0), ready0 = e ? A1_READY(0) : A2_READY(0);
#pragma unroll 1
                for (int s = 0; s < kS; s++) {
                    const bool probe = DBG && threadIdx.x == 0 && i == 1 && e == 0 && s == 1;     // micro-phases of ONE sub-tile's epilogue (analysis build)
                    if (probe) RB_DBG(15);
                    mbar_wait(full0 + 8u * (uint32_t)s, par);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    if (threadIdx.x == 0 && s == 0) RB_DBG(3 + 4 * i + 2 * e);
                    if (probe) RB_DBG(29);
#pragma unroll 1
                    for (int cc = 0; cc < CHW; cc++) {
                        uint32_t acc[32];
                        tmem_ld32(src + (uint32_t)(s * C + cbase + cc * 32), acc);
                        if (probe && cc == 0) RB_DBG(30);
                        write_operand_row<kRtot>(dst, s * 128 + rq, cbase + cc * 32, acc, bias + cc * 32, p.slope, inside(s));
                    }
                    if (probe) RB_DBG(31);
                    if constexpr (DBG) {
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                        if (probe) RB_DBG(41);
                        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) mbar_arrive(ready0 + 8u * (uint32_t)s);
                        if (probe) RB_DBG(42);
                    } else {
                        publish_rows(ready0 + 8u * (uint32_t)s, lane);
                    }
                }
                if (threadIdx.x == 0) RB_DBG(4 + 4 * i + 2 * e);
            }
            if (i == 2) {
                if constexpr (EPI == 5) {
                    // ---- last ResBlock of the vocoder: MRF mean -> lrelu(0.01) -> conv_post (32 -> 1, 7 taps) -> tanh, in place of
                    // writing the fp32 mean and reading it back in k_conv_post (modeling_speecht5.py:3074-3078).  Every MMA of the
                    // CTA has to be complete first, because the whole 512 x 32 fp32 slab V is laid over the weight ring and A1
                    // (rows of 128 bytes, 16-byte pieces XOR-ed with row & 7) and the conv_post weights over A2.
                    static_assert(EPI != 5 || C == 32, "conv_post is fused into the C = 32 stage only");
#pragma unroll 1
                    for (int s = 0; s < kS; s++) mbar_wait(X_FULL(s), par);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    if (threadIdx.x == 0) RB_DBG(5 + 4 * i);
                    const uint32_t v_u32 = smem_u32(smem);
                    float *wp = reinterpret_cast<float *>(sA2);
                    for (int q = threadIdx.x; q < 7 * 32; q += NEW * 32) wp[q] = __ldg(p.post_w + q);
                    // pass A (lane owns a row): X + running bias -> V
#pragma unroll 1
                    for (int s = 0; s < kS; s++) {
                        uint32_t a32[32];
                        tmem_ld32(tmem_X + tm_lane + (uint32_t)(s * C), a32);
                        const float *cb = p.cbias + 2 * C;
                        const int r = s * 128 + rq;
#pragma unroll
                        for (int j = 0; j < 8; j++) {
                            const uint32_t dst = v_u32 + (uint32_t)(r * 128 + ((j ^ (r & 7)) << 4));
                            asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "f"(__uint_as_float(a32[4 * j]) + cb[4 * j]),
                                         "f"(__uint_as_float(a32[4 * j + 1]) + cb[4 * j + 1]), "f"(__uint_as_float(a32[4 * j + 2]) + cb[4 * j + 2]),
                                         "f"(__uint_as_float(a32[4 * j + 3]) + cb[4 * j + 3]) : "memory");
                        }
                    }
                    asm volatile("bar.sync 1, %0;" ::"n"(NEW * 32) : "memory");
                    // pass B (8 lanes per row, coalesced): + MRF partial sum, mean, lrelu(0.01), zero outside the window
                    {
                        const float rcp = p.rdiv, nd = -p.div;
                        const float *aq = p.acc_src + ((size_t)w * p.T + (t_base + quad * 32 + sub_r)) * C + c4 * 4;
#pragma unroll 1
                        for (int s = 0; s < kS; s++) {
                            float4 acc4[8];
#pragma unroll
                            for (int j = 0; j < 8; j++)
                                acc4[j] = ((inside_t[j] >> s) & 1u) ? *reinterpret_cast<const float4 *>(aq + ((size_t)s * 128 + j * 4) * C) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                            for (int j = 0; j < 8; j++) {
                                const int r = s * 128 + quad * 32 + j * 4 + sub_r;
                                const uint32_t a = v_u32 + (uint32_t)(r * 128 + ((c4 ^ (r & 7)) << 4));
                                float4 v;
                                asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a) : "memory");
                                const bool in = ((inside_t[j] >> s) & 1u) != 0u;
                                float o[4] = {acc4[j].x + v.x, acc4[j].y + v.y, acc4[j].z + v.z, acc4[j].w + v.w};
#pragma unroll
                                for (int e = 0; e < 4; e++) {
                                    const float q0 = o[e] * rcp;
                                    const float m = fmaf(fmaf(nd, q0, o[e]), rcp, q0);       // (acc + r) / 3, see the generic epilogue
                                    o[e] = in ? fmaxf(m, 0.01f * m) : 0.0f;
                                }
                                asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(o[0]), "f"(o[1]), "f"(o[2]), "f"(o[3]) : "memory");
                            }
                        }
                    }
                    asm volatile("bar.sync 1, %0;" ::"n"(NEW * 32) : "memory");
                    // pass C (one output sample per thread and trip): 7 taps x 32 channels, weights broadcast from shared memory
                    {
                        const float pb = __ldg(p.post_b);
                        const int tid = threadIdx.x;             // 0 .. 127 (epilogue warps are warps 0 .. 3)
#pragma unroll 1
                        for (int r = p.H + tid; r < p.H + p.V; r += NEW * 32) {
                            const int t = t_base + r;
                            if (t >= p.T) break;
                            float acc = pb;
#pragma unroll
                            for (int j = 0; j < 7; j++) {
                                const int rr = r - 3 + j;
                                if ((unsigned)rr >= (unsigned)kRows) continue;          // outside the slab == outside the window here
#pragma unroll
                                for (int ch = 0; ch < 8; ch++) {
                                    float4 x, wv;
                                    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(x.x), "=f"(x.y), "=f"(x.z), "=f"(x.w)
                                                 : "r"(v_u32 + (uint32_t)(rr * 128 + ((ch ^ (rr & 7)) << 4))) : "memory");
                                    wv = *reinterpret_cast<const float4 *>(wp + j * 32 + ch * 4);
                                    acc = fmaf(wv.x, x.x, acc); acc = fmaf(wv.y, x.y, acc); acc = fmaf(wv.z, x.z, acc); acc = fmaf(wv.w, x.w, acc);
                                }
                            }
                            p.audio[(size_t)w * p.T + t] = tanhf(acc);
                        }
                    }
                    if (threadIdx.x == 0) RB_DBG(6 + 4 * i);
                } else {
                // ---- final epilogue: rows [H, H+V) of the slab leave through a per-warp transpose (A1 is dead: every conv1
                // has retired), 8 lanes per 128 contiguous bytes of an output row.  The MRF partial sum (acc_src) is read in that
                // same coalesced order, one 32x32 piece ahead, starting before the last conv2 has finished.
                float *stg = reinterpret_cast<float *>(sA1) + warp * 32 * kRbStageLd;
                uint32_t out_t[8];
#pragma unroll
                for (int j = 0; j < 8; j++) out_t[j] = __shfl_sync(0xffffffffu, out_mask, j * 4 + sub_r);
                const size_t row0 = (size_t)w * p.T + (t_base + quad * 32 + sub_r);        // global row of (sub-tile 0, j = 0)
                const float *aq = p.acc_src + row0 * C + cbase + c4 * 4;            // only dereferenced when the epilogue has an acc_src
                auto ld_acc = [&](int q, float4 (&b)[8]) {
                    const int s1 = q / CHW, c1 = (q % CHW) * 32;
#pragma unroll
                    for (int j = 0; j < 8; j++)
                        b[j] = ((out_t[j] >> s1) & 1u) ? *reinterpret_cast<const float4 *>(aq + ((size_t)s1 * 128 + j * 4) * C + c1) : make_float4(0.f, 0.f, 0.f, 0.f);
                };
                const bool has_acc = (EPI == 4) ? (p.acc_src != nullptr) : (EPI >= 1);
                const bool has_div = (EPI == 4) ? (p.div != 1.0f) : (EPI >= 2);
                const bool has_o32 = (EPI == 4) ? (p.out32 != nullptr) : (EPI != 2);
                const bool has_ob = (EPI == 4) ? (p.outb != nullptr) : (EPI == 2);
                // register prefetch of the NEXT piece's partial sums
                float4 accA[8], accB[8];
                if (has_acc) ld_acc(0, accA);
                if (threadIdx.x == 0) RB_DBG(40);
                const float rcp = p.rdiv, nd = -p.div;
                // One 32x32 piece.  `cur` holds its partial sums; the next piece's are requested into `nxt` while this one is worked on, and the two
                // buffers swap roles from piece to piece (moving one into the other made every piece wait for its loads).  The row loop is
                // branch-free: four staged rows are read back at a time and the stores are predicated -- with `if (row is an output) { load; add;
                // store; }` the compiler emitted a divergent branch and a load -> store round trip per row, one after the other (round 2: ~1.4k
                // cycles per piece in the stacked-output kernel, whose final epilogue had the same shape).
                auto piece = [&](int q, float4 (&cur)[8], float4 (&nxt)[8]) {
                    const int s = q / CHW, c0 = cbase + (q % CHW) * 32;
                    if ((q % CHW) == 0) {
                        mbar_wait(X_FULL(s), par);
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        if (threadIdx.x == 0 && s == 0) RB_DBG(5 + 4 * i);
                        if (threadIdx.x == 0) RB_DBG(32 + s);
                    }
                    {
                        uint32_t a32[32];
                        tmem_ld32(tmem_X + tm_lane + (uint32_t)(s * C + c0), a32);
                        const float *cb = p.cbias + 2 * C + c0;
#pragma unroll
                        for (int j = 0; j < 32; j++) a32[j] = __float_as_uint(__uint_as_float(a32[j]) + cb[j]);
#pragma unroll
                        for (int j = 0; j < 8; j++)
                            *reinterpret_cast<uint4 *>(stg + lane * kRbStageLd + j * 4) = make_uint4(a32[4 * j], a32[4 * j + 1], a32[4 * j + 2], a32[4 * j + 3]);
                    }
                    __syncwarp();
                    if (has_acc && q + 1 < NCHW) ld_acc(q + 1, nxt);
#pragma unroll
                    for (int jh = 0; jh < 8; jh += 4) {
                        float4 v[4];
#pragma unroll
                        for (int jj = 0; jj < 4; jj++) v[jj] = *reinterpret_cast<const float4 *>(stg + ((jh + jj) * 4 + sub_r) * kRbStageLd + c4 * 4);
#pragma unroll
                        for (int jj = 0; jj < 4; jj++) {
                            const int j = jh + jj;
                            if (has_acc) { v[jj].x = cur[j].x + v[jj].x; v[jj].y = cur[j].y + v[jj].y; v[jj].z = cur[j].z + v[jj].z; v[jj].w = cur[j].w + v[jj].w; }
                            if (has_div) {
                                // v / div as a reciprocal multiply plus one Newton correction (correctly rounded away from denormals;
                                // __fdiv_rn was 9 % of this kernel's stall samples)
                                float q0;
                                q0 = v[jj].x * rcp; v[jj].x = fmaf(fmaf(nd, q0, v[jj].x), rcp, q0);
                                q0 = v[jj].y * rcp; v[jj].y = fmaf(fmaf(nd, q0, v[jj].y), rcp, q0);
                                q0 = v[jj].z * rcp; v[jj].z = fmaf(fmaf(nd, q0, v[jj].z), rcp, q0);
                                q0 = v[jj].w * rcp; v[jj].w = fmaf(fmaf(nd, q0, v[jj].w), rcp, q0);
                            }
                            const bool out = ((out_t[j] >> s) & 1u) != 0u;
                            const size_t o = out ? (row0 + (size_t)s * 128 + j * 4) * C + (size_t)(c0 + c4 * 4) : 0;
                            if (has_o32)
                                asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %5, 0;\n\t@p st.global.v4.f32 [%0], {%1, %2, %3, %4};\n\t}"
                                             ::"l"(p.out32 + o), "f"(v[jj].x), "f"(v[jj].y), "f"(v[jj].z), "f"(v[jj].w), "r"((int)out) : "memory");
                            if (has_ob) {
                                __nv_bfloat162 h0 = __floats2bfloat162_rn(lrelu_f(v[jj].x, p.outb_slope), lrelu_f(v[jj].y, p.outb_slope));
                                __nv_bfloat162 h1 = __floats2bfloat162_rn(lrelu_f(v[jj].z, p.outb_slope), lrelu_f(v[jj].w, p.outb_slope));
                                asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %3, 0;\n\t@p st.global.v2.b32 [%0], {%1, %2};\n\t}"
                                             ::"l"(p.outb + o), "r"(*reinterpret_cast<uint32_t *>(&h0)), "r"(*reinterpret_cast<uint32_t *>(&h1)), "r"((int)out) : "memory");
                            }
                        }
                    }
                    __syncwarp();
                    if ((q % CHW) == CHW - 1 && threadIdx.x == 0) RB_DBG(36 + s);
                };
                static_assert(NCHW % 2 == 0, "the final epilogue walks the pieces in pairs");
#pragma unroll 1
                for (int q = 0; q < NCHW; q += 2) {
                    piece(q, accA, accB);
                    piece(q + 1, accB, accA);
                }
                }
                if (threadIdx.x == 0) RB_DBG(6 + 4 * i);
            }
        }
    } else if (warp == NEW) {
        // ======================================================================================= weight ring (TMA)
        if (lane == 0) {
            int slot = 0; uint32_t phase = 0;
            for (int c = 0; c < 6; c++)
                for (int g = 0; g < p.ngroups; g++)
                    for (int kb = 0; kb < NKB; kb++) {
                        mbar_wait(W_EMPTY(slot), phase ^ 1);
                        mbar_expect_tx(W_FULL(slot), slot_bytes);
                        tma_load_3d(smem_u32(sW + (size_t)slot * slot_bytes), &tmap_w, W_FULL(slot), kb * KB, 0, c * p.taps + g * p.tps);
                        if (++slot == p.nslots) { slot = 0; phase ^= 1; }
                    }
        }
        __syncwarp();
    } else {
        // ======================================================================================= MMA issuers
        // Everything that feeds tcgen05.mma has to live in UNIFORM registers.  The warp index and the TMEM base are therefore
        // taken through a lane-0 broadcast (which the compiler knows to be warp-uniform) and the whole issue loop runs inside
        // one elected thread: descriptors are then computed on the uniform datapath, with no per-MMA R2UR traffic.
        const int mw = __shfl_sync(0xffffffffu, warp, 0) - (NEW + 1);
        const uint32_t tX = __shfl_sync(0xffffffffu, tmem_X, 0);
        if (elect_one()) {
            const int s_first = mw * SPW;
            // kind::f16 instruction descriptor: D = f32, A = B = bf16, both K-major, N = C, M = 128
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(C >> 3) << 17) | ((128u >> 4) << 24);
            const uint32_t b_layout = (KB == 64) ? 2u : 4u;                // SWIZZLE_128B : SWIZZLE_64B (a weight row is KB bf16)
            const uint64_t adesc_1 = smem_desc(smem_u32(sA1), (uint32_t)kRtot * 16, 128u, 0u);
            const uint64_t adesc_2 = smem_desc(smem_u32(sA2), (uint32_t)kRtot * 16, 128u, 0u);
            const uint64_t bdesc0 = smem_desc(smem_u32(sW), 0u, 8u * (uint32_t)KB * 2, b_layout);
            const uint32_t slot_16 = slot_bytes >> 4, tap_16 = kTapKbBytes >> 4;
            constexpr int ksteps = KB / 16;
            int slot = 0; uint32_t phase = 0;
#pragma unroll 1
            for (int i = 0; i < 3; i++) {
                const uint32_t par = (uint32_t)(i & 1);
#pragma unroll 1
                for (int cv = 0; cv < 2; cv++) {
                    const int dil = cv ? 1 : (i == 0 ? p.dil0 : (i == 1 ? p.dil1 : p.dil2));
                    const int pad = ((p.taps - 1) >> 1) * dil;
                    const uint64_t adesc_c = (cv ? adesc_2 : adesc_1) + (uint64_t)(uint32_t)(kGuard - pad);
                    const uint32_t acc_base = cv ? tX : tX + (uint32_t)(kS * C);
                    const uint32_t ready0 = cv ? A2_READY(0) : A1_READY(0);
                    const uint32_t done0 = cv ? X_FULL(0) : T1_FULL(0);
#pragma unroll 1
                    for (int g = 0; g < p.ngroups; g++) {
                        const int j0 = g * p.tps;
                        const int ntap = min(p.tps, p.taps - j0);
#pragma unroll 1
                        for (int kb = 0; kb < NKB; kb++) {
                            mbar_wait(W_FULL(slot), phase);
                            const uint64_t bdesc_g = bdesc0 + (uint64_t)((uint32_t)slot * slot_16);
                            const bool first = (g == 0) && (kb == 0), last = (g == p.ngroups - 1) && (kb == NKB - 1);
#pragma unroll 1
                            for (int ss = 0; ss < SPW; ss++) {
                                const int s = s_first + ss;
                                if (first) {
                                    // operand rows of sub-tiles s-1 .. s+1 (the taps reach at most 25 rows out)
                                    if (ss == 0) {
                                        if (s > 0) mbar_wait(ready0 + 8u * (uint32_t)(s - 1), par);
                                        mbar_wait(ready0 + 8u * (uint32_t)s, par);
                                    }
                                    if (s + 1 < kS) mbar_wait(ready0 + 8u * (uint32_t)(s + 1), par);
                                }
                                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                                if (mw == 0 && first && ss == 0) RB_DBG(16 + 2 * (2 * i + cv));
                                const uint32_t tacc = acc_base + (uint32_t)(s * C);
                                uint64_t ad = adesc_c + (uint64_t)(uint32_t)(s * 128 + j0 * dil + kb * (KB / 8) * kRtot);
                                uint64_t bd = bdesc_g;
#pragma unroll 1
                                for (int tt = 0; tt < ntap; tt++) {
#pragma unroll
                                    for (int ks = 0; ks < ksteps; ks++)
                                        umma_f16(tacc, ad + (uint64_t)(uint32_t)(ks * 2 * kRtot), bd + (uint64_t)(uint32_t)(ks * 2), idesc,
                                                 (ks || cv || !first || tt) ? 1u : 0u);      // conv2 always adds to the residual stream
                                    ad += (uint64_t)(uint32_t)dil;
                                    bd += (uint64_t)tap_16;
                                }
                                if (last) umma_commit(done0 + 8u * (uint32_t)s);
                            }
                            umma_commit(W_EMPTY(slot));
                            if (++slot == p.nslots) { slot = 0; phase ^= 1; }
                        }
                    }
                    if (mw == 0) RB_DBG(17 + 2 * (2 * i + cv));
                }
            }
        }
        __syncwarp();
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) RB_DBG(28);
    if (warp == NEW) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_X), "r"((uint32_t)(2 * kS * C)) : "memory");
    }
}

#undef W_FULL
#undef W_EMPTY
#undef A1_READY
#undef T1_FULL
#undef A2_READY
#undef X_FULL
#undef inside
#undef is_out
#undef RB_DBG

// ---------------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int tps_for(int C) { return C <= 64 ? 4 : 1; }           // taps per weight slot
static int nslots_for(int C) { return C == 64 ? 2 : 4; }          // slots of 8 KB (C=32), 32 KB (C=64), 16 KB (C=128: one tap, one K block)
static int kb_for(int C) { return C >= 64 ? 64 : 32; }
static int rows_for(int C) { return C <= 64 ? 512 : 256; }

bool resblock_supported(int C, int taps) { return (C == 32 || C == 64 || C == 128) && (taps & 1) && taps >= 3 && taps <= 11; }

int resblock_pack(const Layer *const conv1[3], const Layer *const conv2[3], ResBlockPack &out, std::vector<void *> &allocs, size_t &bytes) {
    const int C = conv1[0]->Cin, k = conv1[0]->taps;
    if (!resblock_supported(C, k)) return set_error("resblock: unsupported C=%d k=%d", C, k);
    for (int i = 0; i < 3; i++) {
        const Layer *ls[2] = {conv1[i], conv2[i]};
        for (const Layer *l : ls)
            if (l->Cin != C || l->Cout != C || l->taps != k || !l->wbf || l->pad * 2 != (k - 1) * l->dil)
                return set_error("resblock: the six convolutions must share C and k and have bf16 weights");
        if (conv2[i]->dil != 1) return set_error("resblock: conv2 must have dilation 1");
        if (((k - 1) / 2) * conv1[i]->dil >= kGuard) return set_error("resblock: dilation %d too large", conv1[i]->dil);
        out.dil[i] = conv1[i]->dil;
    }
    out.C = C; out.taps = k;
    const int tps = tps_for(C);
    const size_t per_conv = (size_t)k * C * C;
    const size_t total = (6 * (size_t)k + tps) * C * C;              // + tps zero taps: the last TMA box stays in bounds
    void *q = nullptr;
    B2_CUDA_OK(cudaMalloc(&q, total * sizeof(__nv_bfloat16)));
    allocs.push_back(q); bytes += total * sizeof(__nv_bfloat16);
    out.w = reinterpret_cast<__nv_bfloat16 *>(q);
    B2_CUDA_OK(cudaMemset(q, 0, total * sizeof(__nv_bfloat16)));
    std::vector<float> hb((size_t)6 * C), b1((size_t)3 * C), cb((size_t)3 * C);
    for (int i = 0; i < 3; i++) {
        B2_CUDA_OK(cudaMemcpy(out.w + (size_t)(2 * i) * per_conv, conv1[i]->wbf, per_conv * sizeof(__nv_bfloat16), cudaMemcpyDeviceToDevice));
        B2_CUDA_OK(cudaMemcpy(out.w + (size_t)(2 * i + 1) * per_conv, conv2[i]->wbf, per_conv * sizeof(__nv_bfloat16), cudaMemcpyDeviceToDevice));
        B2_CUDA_OK(cudaMemcpy(hb.data() + (size_t)(2 * i) * C, conv1[i]->bias, C * sizeof(float), cudaMemcpyDeviceToHost));
        B2_CUDA_OK(cudaMemcpy(hb.data() + (size_t)(2 * i + 1) * C, conv2[i]->bias, C * sizeof(float), cudaMemcpyDeviceToHost));
    }
    for (int i = 0; i < 3; i++)
        for (int c = 0; c < C; c++) {
            b1[(size_t)i * C + c] = hb[(size_t)(2 * i) * C + c];
            cb[(size_t)i * C + c] = hb[(size_t)(2 * i + 1) * C + c] + (i ? cb[(size_t)(i - 1) * C + c] : 0.0f);
        }
    out.h_bias1 = b1;          // the biases travel as kernel parameters (constant bank)
    out.h_cbias = cb;

    if (umma_init()) return 1;
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) return set_error("cuTensorMapEncodeTiled is not available from the driver");
    CUtensorMap *tm = new CUtensorMap();
    cuuint64_t gdim[3] = {(cuuint64_t)C, (cuuint64_t)C, (cuuint64_t)(6 * k + tps)};
    cuuint64_t gstr[2] = {(cuuint64_t)C * 2, (cuuint64_t)C * C * 2};
    cuuint32_t box[3] = {(cuuint32_t)kb_for(C), (cuuint32_t)C, (cuuint32_t)tps};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = reinterpret_cast<EncodeTiledFn>(fn)(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void *)out.w, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                                                     C >= 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                                                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { delete tm; return set_error("resblock: cuTensorMapEncodeTiled failed with CUresult %d (C %d k %d)", (int)r, C, k); }
    out.tmap = tm;
    return resblock_t_pack(out, allocs, bytes);          // C = 32: the stacked-output kernel's copy of the weights (no-op otherwise)
}

void resblock_free(ResBlockPack &p) {
    if (p.tmap) { delete reinterpret_cast<CUtensorMap *>(p.tmap); p.tmap = nullptr; }
    resblock_t_free(p);
}


static bool g_rb_attr[64][3][7] = {};

// launches the instantiation whose compile-time epilogue matches the request (the vocoder's three launches per stage are EPI 0, 1 and 2
// or 3); anything else, and the timestamped analysis build, runs the generic kernel
template <int C, int NEW, int NMW>
static int launch_rb(const CUtensorMap &tm, const RbParams &p, unsigned grid, size_t smem, cudaStream_t st, int wslot) {
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    auto go = [&](void (*kern)(CUtensorMap, RbParams), int eslot) -> int {
        if (dev < 64 && !g_rb_attr[dev][wslot][eslot]) {
            B2_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
            g_rb_attr[dev][wslot][eslot] = true;
        }
        B2_CUDA_OK(launch_k(kern, dim3(grid), dim3((NEW + 1 + NMW) * 32), smem, st, pdl_enabled(), tm, p));
        B2_LAUNCH_OK("k_resblock");
        return 0;
    };
    if (p.dbg) return go(k_resblock<C, NEW, NMW, 4, true>, 6);
    if constexpr (C == 32) {
        if (p.audio) return go(k_resblock<C, NEW, NMW, 5, false>, 5);
    }
    const bool acc = p.acc_src != nullptr, dv = p.div != 1.0f, o32 = p.out32 != nullptr, ob = p.outb != nullptr;
    if (!acc && !dv && o32 && !ob) return go(k_resblock<C, NEW, NMW, 0, false>, 0);
    if (acc && !dv && o32 && !ob) return go(k_resblock<C, NEW, NMW, 1, false>, 1);
    if (acc && dv && !o32 && ob) return go(k_resblock<C, NEW, NMW, 2, false>, 2);
    if (acc && dv && o32 && !ob) return go(k_resblock<C, NEW, NMW, 3, false>, 3);
    return go(k_resblock<C, NEW, NMW, 4, false>, 4);
}

int g_rbt_min_taps = 0;

int launch_resblock(const ResBlockArgs &a, cudaStream_t st) {
    const ResBlockPack &pk = *a.pack;
    if (!pk.tmap || !pk.w) return set_error("resblock: weights were not packed");
    const bool post = a.audio != nullptr;
    if (post && (pk.C != 32 || !a.post_w || !a.post_b || !a.acc_src)) return set_error("resblock: the conv_post epilogue needs C = 32, weights and the MRF partial sum");
    if ((!a.x && !a.up_in) || (!a.out32 && !a.outb && !post)) return set_error("resblock: null input or no output");
    if (a.W <= 0 || a.T <= 0) return 0;
    if (a.up_in) {                  // x = upsampler(up_in) computed in the kernel: the stacked-output kernel only
        if (!pk.tmap_t) return set_error("resblock: the fused upsampler needs the stacked-output kernel (C = 32)");
        return launch_resblock_t(a, st);
    }
    // C = 32, five taps and more: the stacked-output kernel (conv_resblock_t.cu).  Measured (ncu, 4,096 windows, same run):
    // k = 11 2.73 vs 3.57 ms, k = 7 1.85 vs 2.01 ms, but k = 3 1.44 vs 1.34 ms -- with three taps half of the stacked MMAs' N range is
    // structural zeros and the conv epilogues, not the MMAs, set the pace in both kernels.
    const int rbt_mink = g_rbt_min_taps > 0 ? g_rbt_min_taps : 5;          // b2_debug_set_stacked_min_taps: the tests run both C = 32 kernels
    if (pk.tmap_t && pk.taps >= rbt_mink) return launch_resblock_t(a, st);
    RbParams p;
    p.x = a.x; p.acc_src = a.acc_src; p.out32 = a.out32; p.outb = a.outb;
    p.post_w = a.post_w; p.post_b = a.post_b; p.audio = a.audio;
    p.slope = a.slope; p.outb_slope = a.outb_slope; p.div = a.div; p.rdiv = 1.0f / a.div;
    p.W = a.W; p.T = a.T; p.taps = pk.taps;
    for (int i = 0; i < 3 * kRbMaxC; i++) { p.bias1[i] = 0.0f; p.cbias[i] = 0.0f; }
    for (int i = 0; i < 3 * pk.C; i++) { p.bias1[i] = pk.h_bias1[i]; p.cbias[i] = pk.h_cbias[i]; }
    int dsum = 0;
    for (int i = 0; i < 3; i++) dsum += pk.dil[i] + 1;
    p.dil0 = pk.dil[0]; p.dil1 = pk.dil[1]; p.dil2 = pk.dil[2];
    const int rows = rows_for(pk.C);
    if (a.T <= rows) {
        // the whole window fits in one slab: its edges are the reference's own zero padding, no halo is needed
        p.H = 0; p.tiles_per_win = 1; p.V = a.T;
    } else {
        p.H = ((pk.taps - 1) / 2) * dsum + (post ? 3 : 0);      // conv_post reaches three more rows either side
        const int vmax = rows - 2 * p.H;
        if (vmax < 64) return set_error("resblock: halo %d leaves no room in a %d-row slab", p.H, rows);
        p.tiles_per_win = cdiv(a.T, vmax);
        p.V = cdiv(a.T, p.tiles_per_win);
    }
    p.m_tpw = ((1ull << 40) + (unsigned long long)p.tiles_per_win - 1) / (unsigned long long)p.tiles_per_win;
    p.tps = tps_for(pk.C);
    p.ngroups = cdiv(pk.taps, p.tps);
    p.nslots = nslots_for(pk.C);
    const long long nct = (long long)a.W * p.tiles_per_win;
    if (nct >= (1ll << 24)) return set_error("resblock: too many tiles (%lld)", nct);
    const size_t a_bytes = ((size_t)(rows + 2 * kGuard + 1) * pk.C * 2 + 1023) & ~(size_t)1023;
    const size_t smem = (size_t)p.nslots * p.tps * pk.C * kb_for(pk.C) * 2 + 2 * a_bytes + 24 * 8 + 16;
    if (smem > 227 * 1024) return set_error("resblock: needs %zu bytes of shared memory", smem);
    const CUtensorMap &tm = *reinterpret_cast<const CUtensorMap *>(pk.tmap);
    static const bool dbg_on = getenv("B2_RB_DBG") != nullptr;
    static unsigned long long *dbg_buf = nullptr;
    const size_t dbg_n = (size_t)kRbDbgCtas * kRbDbgEvents;
    if (dbg_on && !dbg_buf) B2_CUDA_OK(cudaMalloc(&dbg_buf, dbg_n * 8));
    p.dbg = dbg_on ? dbg_buf : nullptr;
    if (dbg_on) B2_CUDA_OK(cudaMemsetAsync(dbg_buf, 0, dbg_n * 8, st));
    // C = 32: four epilogue warps (two CTAs share an SM); C = 64 / 128: eight, each with half of a row's columns
    const int rc = (pk.C == 32) ? launch_rb<32, 4, 2>(tm, p, (unsigned)nct, smem, st, 0)
                   : (pk.C == 64) ? launch_rb<64, 8, 2>(tm, p, (unsigned)nct, smem, st, 1)
                   : launch_rb<128, 8, 2>(tm, p, (unsigned)nct, smem, st, 2);
    if (dbg_on && !rc) {
        // per-phase averages over the first CTAs of the launch (cycles of the SM clock)
        B2_CUDA_OK(cudaStreamSynchronize(st));
        static std::vector<unsigned long long> h;
        h.resize(dbg_n);
        B2_CUDA_OK(cudaMemcpy(h.data(), dbg_buf, dbg_n * 8, cudaMemcpyDeviceToHost));
        const int n = (int)std::min<long long>(kRbDbgCtas, nct);
        double ev[kRbDbgEvents] = {0};
        int cnt = 0;
        for (int b = 0; b < n; b++) {
            const unsigned long long *r = &h[(size_t)b * kRbDbgEvents];
            if (!r[0] || !r[28]) continue;
            cnt++;
            for (int k = 0; k < kRbDbgEvents; k++) ev[k] += r[k] ? (double)(r[k] - r[0]) : 0.0;
        }
        if (cnt) {
            for (int k = 0; k < kRbDbgEvents; k++) ev[k] /= cnt;
            fprintf(stderr, "[rb dbg] C=%d k=%d T=%d ctas=%lld (avg of %d) cycles since CTA start: setup %.0f | load done %.0f | end %.0f\n", pk.C, pk.taps, a.T, nct, cnt, ev[1], ev[2], ev[28]);
            fprintf(stderr, "[rb dbg]   load done per sub-tile %.0f %.0f %.0f %.0f | acc parked %.0f | final: ready/done per sub-tile %.0f/%.0f %.0f/%.0f %.0f/%.0f %.0f/%.0f\n",
                    ev[44], ev[45], ev[46], ev[47], ev[40], ev[32], ev[36], ev[33], ev[37], ev[34], ev[38], ev[35], ev[39]);
            fprintf(stderr, "[rb dbg]   conv-epilogue micro-phases (warp 0, pair 1 epilogue 1, sub-tile 1): barrier wait %.0f | TMEM load %.0f | math + st.shared %.0f | proxy fence %.0f | arrive %.0f\n",
                    ev[29] - ev[15], ev[30] - ev[29], ev[31] - ev[30], ev[41] - ev[31], ev[42] - ev[41]);
            for (int i = 0; i < 3; i++)
                fprintf(stderr, "[rb dbg]   pair %d: conv1 issue %.0f..%.0f (%.0f) | epi1 first-ready %.0f done %.0f | conv2 issue %.0f..%.0f (%.0f) | epi2 first-ready %.0f done %.0f\n", i,
                        ev[16 + 4 * i], ev[17 + 4 * i], ev[17 + 4 * i] - ev[16 + 4 * i], ev[3 + 4 * i], ev[4 + 4 * i],
                        ev[18 + 4 * i], ev[19 + 4 * i], ev[19 + 4 * i] - ev[18 + 4 * i], ev[5 + 4 * i], ev[6 + 4 * i]);
        }
    }
    return rc;
}

}  // namespace b2
