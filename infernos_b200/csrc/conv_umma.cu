// tcgen05 (UMMA) implicit-GEMM conv1d, hand-written for sm_100a.
//
// One CTA computes a 128-row x N_TILE tile of   out[w][t][n] = bias[n] + sum_j sum_ci Wb[j][n][ci] * in[w][t + j*dil - pad][ci]
// for the HiFiGAN upsamplers (ConvTranspose1d restated as a 3-tap conv, see tail.cu:pack_convT) and ResBlock convs
// (modeling_speecht5.py:2954-2962, 3066-3067), with bias / residual / MRF-accumulate / leaky-ReLU fused in the epilogue.
//
//   A operand (activations, M = time)  : the tile's rows PLUS the conv halo are brought into shared memory ONCE with
//       cp.async (zero-filled outside the window: every window is padded on its own, HelloSippyRTPipe.py:234-236),
//       in the un-swizzled K-major "interleaved" UMMA layout [channel/8][row][8 channels].  In that layout consecutive
//       rows are exactly 16 bytes apart, so filter tap j is the SAME buffer read through a descriptor whose start
//       address is advanced by j*dil rows: the k taps cost no extra global or L2 traffic.
//   B operand (weights, N = out chans) : streamed per (K-block, tap) by TMA into a 128B/64B-swizzled ring, mbarrier pipelined.
//   D accumulator                      : fp32 in TMEM (N_TILE columns), read back with tcgen05.ld by four epilogue warps.
//
// Warp roles (192 threads): warps 0-3 = A producers, then epilogue (TMEM lanes 32*warp..); warp 4 = TMA producer for B;
// warp 5 = TMEM allocator + single-thread tcgen05.mma issuer.
#include "conv_umma.cuh"
#include "umma_ptx.cuh"

#include <cuda.h>
#include <stdlib.h>
#include <algorithm>
#include <mutex>
#include <vector>

namespace b2 {

static constexpr int kThreads = 192;
static constexpr int kMaxKB = 8;      // Cin <= 512 in blocks of 64
static constexpr int kStageLd = 36;                       // floats per staged row (32 + 4 pad: conflict-free 128-bit access)
static constexpr int kStageBytes = 4 * 32 * kStageLd * 4; // epilogue transpose staging, four warps

struct UmmaParams {
    const __nv_bfloat16 *in;
    const float *bias;
    const float *residual;
    const float *acc_src;
    float *out32;
    __nv_bfloat16 *outb;
    float outb_slope, div;
    int W, T, Cin, N, taps, dil, pad;
    int R;            // rows of the A buffer (128 + (taps-1)*dil, made odd)
    int KB;           // K block: 64 (128B swizzle) or 32 (64B swizzle)
    int nkb;          // Cin / KB
    int nseg;         // windows per tile (short windows), else 1
    int period;       // row period between the windows of a tile (T + pad), or 1<<30
    int tiles_per_win;// ceil(T / 128) when nseg == 1
    int stages;       // B ring depth
    unsigned long long *dbg;   // optional per-CTA phase timestamps (analysis builds)
    unsigned long long m_period, m_tpw, m_ntiles;   // ceil(2^40 / d) for period, tiles_per_win, ntiles (see fdiv)
};

// ---------------------------------------------------------------------------------------------------- kernel
__device__ __forceinline__ unsigned long long gtime() { unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t; }
#define DBG(k) do { if (p.dbg && blockIdx.x < 8192 && blockIdx.y == 0) p.dbg[(size_t)blockIdx.x * 8 + (k)] = gtime(); } while (0)
template <int N_TILE>
__global__ void __launch_bounds__(kThreads, (N_TILE <= 64) ? 4 : ((N_TILE <= 128) ? 2 : 1)) k_conv_umma(const __grid_constant__ CUtensorMap tmap_w, const UmmaParams p) {
    pdl_trigger();
    extern __shared__ __align__(1024) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int KB = p.KB;
    const uint32_t b_stage_bytes = (uint32_t)N_TILE * KB * 2;
    const uint32_t a_raw = (uint32_t)p.R * p.Cin * 2;
    const uint32_t a_bytes = a_raw > (uint32_t)kStageBytes ? a_raw : (uint32_t)kStageBytes;   // doubles as the epilogue staging area
    uint8_t *sB = smem;
    uint8_t *sA = smem + (size_t)p.stages * b_stage_bytes;
    uint64_t *bars = reinterpret_cast<uint64_t *>(sA + ((a_bytes + 15) & ~15u));
    // bars: [0..stages) b_full, [stages..2*stages) b_empty, [2*stages .. +kMaxKB) a_full, then acc_full
    const uint32_t bar_b_full = smem_u32(bars);
    const uint32_t bar_b_empty = smem_u32(bars + p.stages);
    const uint32_t bar_a_full = smem_u32(bars + 2 * p.stages);
    const uint32_t bar_acc = smem_u32(bars + 2 * p.stages + kMaxKB);
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * p.stages + kMaxKB + 1);

    // ---- tile coordinates
    int w0, t0;
    if (p.nseg > 1) { w0 = blockIdx.x * p.nseg; t0 = 0; }
    else { w0 = fdiv(blockIdx.x, p.m_tpw); t0 = (blockIdx.x - w0 * p.tiles_per_win) * 128; }
    const int n0 = blockIdx.y * N_TILE;

    // Prologue, arranged so that nothing waits for anything it does not need: the TMA thread initialises the barriers and
    // starts streaming weights at once, the producer warps start the first K block of the A tile, warp 5 allocates TMEM;
    // only then does the CTA synchronise.  (what-if runs: this fixed per-CTA cost was 43 % of the thin layers' time.)
    if (threadIdx.x == 0) DBG(0);
    const int total_b = p.nkb * p.taps;
    int b_issued = 0;
    if (warp == 4 && lane == 0) {
        if (smem_u32(smem) & 1023u) __trap();
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_w) : "memory");
        for (int s = 0; s < p.stages; s++) { mbar_init(bar_b_full + 8 * s, 1); mbar_init(bar_b_empty + 8 * s, 1); }
        for (int k = 0; k < kMaxKB; k++) mbar_init(bar_a_full + 8 * k, 128);
        mbar_init(bar_acc, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        for (; b_issued < p.stages && b_issued < total_b; b_issued++) {        // first round of the ring: every slot is free
            const int kb = b_issued / p.taps, j = b_issued - kb * p.taps;
            mbar_expect_tx(bar_b_full + 8 * b_issued, b_stage_bytes);
            tma_load_3d(smem_u32(sB + (size_t)b_issued * b_stage_bytes), &tmap_w, bar_b_full + 8 * b_issued, kb * KB, n0, j);
        }
    }
    if (warp == 5) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)N_TILE) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    const int cshift = (KB == 64) ? 3 : 2;        // 16-byte pieces per row per K block = 1 << cshift
    const int cpr = 1 << cshift;
    const int pieces = p.R * cpr;
    auto load_a_block = [&](int kb) {
        const uint32_t sA_u32 = smem_u32(sA);
        for (int q = threadIdx.x; q < pieces; q += 128) {
            const int r = q >> cshift, c = q & (cpr - 1);
            const int u = r - p.pad;
            const int s = (u >= 0 && p.nseg > 1) ? fdiv(u, p.m_period) : 0;
            const int t = t0 + (u - s * p.period);
            const int w = w0 + s;
            const bool ok = (t >= 0) && (t < p.T) && (s < p.nseg) && (w < p.W);
            const __nv_bfloat16 *src = ok ? p.in + ((size_t)w * p.T + t) * p.Cin + kb * KB + c * 8 : p.in;
            cp_async16(sA_u32 + (uint32_t)(((kb * cpr + c) * p.R + r) * 16), src, ok ? 16u : 0u);
        }
    };
    if (warp < 4) {
        pdl_wait();                 // the activations are the previous kernel's output (the weight ring above overlapped its tail)
        load_a_block(0);
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    if (threadIdx.x == 0) DBG(1);

    if (warp < 4) {
        // =========================== A producer: tile rows + halo, once ===========================
        cp_async_arrive_noinc(bar_a_full);
        for (int kb = 1; kb < p.nkb; kb++) {
            load_a_block(kb);
            cp_async_arrive_noinc(bar_a_full + 8 * kb);
        }
        if (threadIdx.x == 0) DBG(2);
        // =========================== epilogue ===========================
        mbar_wait(bar_acc, 0);
        if (threadIdx.x == 0) DBG(3);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        // The A buffer is dead once the accumulator barrier has fired (every MMA that read it has retired): it becomes the
        // staging area of a per-warp transpose, so that global memory is touched with 8 lanes per 128 contiguous bytes of one
        // output row (4 whole rows per warp instruction) instead of one 16-byte piece per row per lane.  The what-if runs in
        // profiles/ put 54 % of the round-1 step time on the un-coalesced version of these accesses.
        if (!p.residual && !p.acc_src && !p.out32) {
            // bf16-only output (conv1 of a pair): a lane already owns 64 contiguous bytes of its row, written as four
            // 128-bit stores; the transpose would only add work (measured 1.16x slower at C=32)
            const int m = warp * 32 + lane;
            const int s = (p.nseg > 1) ? fdiv(m, p.m_period) : 0;
            const int t = t0 + (m - s * p.period);
            const int w = w0 + s;
            const bool ok = (t < p.T) && (s < p.nseg) && (w < p.W);
            const size_t row_off = ((size_t)w * p.T + t) * p.N + n0;
#pragma unroll 1
            for (int c0 = 0; c0 < N_TILE; c0 += 32) {
                uint32_t acc[32];
                tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, acc);
                if (!ok) continue;
                uint4 *op = reinterpret_cast<uint4 *>(p.outb + row_off + c0);
#pragma unroll
                for (int i = 0; i < 4; i++) {
                    uint32_t pk[4];
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        const float2 b = __ldg(reinterpret_cast<const float2 *>(p.bias + n0 + c0 + 8 * i + 2 * e));
                        __nv_bfloat162 h2 = __floats2bfloat162_rn(lrelu_f(__uint_as_float(acc[8 * i + 2 * e]) + b.x, p.outb_slope),
                                                                  lrelu_f(__uint_as_float(acc[8 * i + 2 * e + 1]) + b.y, p.outb_slope));
                        pk[e] = *reinterpret_cast<uint32_t *>(&h2);
                    }
                    op[i] = make_uint4(pk[0], pk[1], pk[2], pk[3]);
                }
            }
        } else {
            float *stg = reinterpret_cast<float *>(sA) + warp * 32 * kStageLd;
            const int sub_r = lane >> 3, c4 = lane & 7;
            const int m = warp * 32 + lane;
            const int s = (p.nseg > 1) ? fdiv(m, p.m_period) : 0;
            const int t = t0 + (m - s * p.period);
            const int w = w0 + s;
            const int grow_own = ((t < p.T) && (s < p.nseg) && (w < p.W)) ? (w * p.T + t) : -1;
            int grow[8];
#pragma unroll
            for (int i = 0; i < 8; i++) grow[i] = __shfl_sync(0xffffffffu, grow_own, i * 4 + sub_r);
#pragma unroll 1
            for (int c0 = 0; c0 < N_TILE; c0 += 32) {
                const int col = n0 + c0 + c4 * 4;
                const float4 bias = __ldg(reinterpret_cast<const float4 *>(p.bias + col));
                {
                    uint32_t a32[32];
                    tmem_ld32(tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)c0, a32);
#pragma unroll
                    for (int i = 0; i < 8; i++)
                        *reinterpret_cast<uint4 *>(stg + lane * kStageLd + i * 4) = make_uint4(a32[4 * i], a32[4 * i + 1], a32[4 * i + 2], a32[4 * i + 3]);
                }
                __syncwarp();
#pragma unroll
                for (int h = 0; h < 2; h++) {
                    float4 res[4], accs[4];
                    if (p.residual) {
#pragma unroll
                        for (int i = 0; i < 4; i++)
                            res[i] = grow[h * 4 + i] >= 0 ? *reinterpret_cast<const float4 *>(p.residual + (size_t)grow[h * 4 + i] * p.N + col) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
                    if (p.acc_src) {
#pragma unroll
                        for (int i = 0; i < 4; i++)
                            accs[i] = grow[h * 4 + i] >= 0 ? *reinterpret_cast<const float4 *>(p.acc_src + (size_t)grow[h * 4 + i] * p.N + col) : make_float4(0.f, 0.f, 0.f, 0.f);
                    }
#pragma unroll
                    for (int i = 0; i < 4; i++) {
                        const int g = grow[h * 4 + i];
                        if (g < 0) continue;
                        float4 v = *reinterpret_cast<const float4 *>(stg + ((h * 4 + i) * 4 + sub_r) * kStageLd + c4 * 4);
                        v.x += bias.x; v.y += bias.y; v.z += bias.z; v.w += bias.w;
                        if (p.residual) { v.x += res[i].x; v.y += res[i].y; v.z += res[i].z; v.w += res[i].w; }
                        if (p.acc_src) { v.x = accs[i].x + v.x; v.y = accs[i].y + v.y; v.z = accs[i].z + v.z; v.w = accs[i].w + v.w; }
                        if (p.div != 1.0f) { v.x = __fdiv_rn(v.x, p.div); v.y = __fdiv_rn(v.y, p.div); v.z = __fdiv_rn(v.z, p.div); v.w = __fdiv_rn(v.w, p.div); }
                        const size_t o = (size_t)g * p.N + col;
                        if (p.out32) *reinterpret_cast<float4 *>(p.out32 + o) = v;
                        if (p.outb) {
                            __nv_bfloat162 h0 = __floats2bfloat162_rn(lrelu_f(v.x, p.outb_slope), lrelu_f(v.y, p.outb_slope));
                            __nv_bfloat162 h1 = __floats2bfloat162_rn(lrelu_f(v.z, p.outb_slope), lrelu_f(v.w, p.outb_slope));
                            *reinterpret_cast<uint2 *>(p.outb + o) = make_uint2(*reinterpret_cast<uint32_t *>(&h0), *reinterpret_cast<uint32_t *>(&h1));
                        }
                    }
                }
                __syncwarp();
            }
        }
        if (threadIdx.x == 0) DBG(4);
    } else if (warp == 4) {
        // =========================== B producer (TMA) ===========================
        if (lane == 0) {
            // the first p.stages loads were issued in the prologue; the ring wraps from here on
            int stage = (b_issued == p.stages) ? 0 : b_issued;
            uint32_t phase = (b_issued == p.stages) ? 1 : 0;
            for (int i = b_issued; i < total_b; i++) {
                const int kb = i / p.taps, j = i - kb * p.taps;
                mbar_wait(bar_b_empty + 8 * stage, phase ^ 1);
                mbar_expect_tx(bar_b_full + 8 * stage, b_stage_bytes);
                tma_load_3d(smem_u32(sB + (size_t)stage * b_stage_bytes), &tmap_w, bar_b_full + 8 * stage, kb * KB, n0, j);
                if (++stage == p.stages) { stage = 0; phase ^= 1; }
            }
        }
    } else {
        // =========================== MMA issuer ===========================
        // Everything that feeds tcgen05.mma has to live in UNIFORM registers: the TMEM base goes through a lane-0 broadcast
        // (which the compiler knows to be warp-uniform) and the whole issue loop runs inside one elected thread, so that the
        // descriptors are computed on the uniform datapath.  (With per-lane values every MMA cost ~9 R2UR moves and ~130
        // cycles of issue time against 40-128 cycles of tensor-pipe time.)
        const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
        if (elect_one()) {
            // kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, N = N_TILE, M = 128
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N_TILE >> 3) << 17) | ((128u >> 4) << 24);
            const uint32_t sA_u32 = smem_u32(sA);
            const uint32_t b_layout = (KB == 64) ? 2u : 4u;             // SWIZZLE_128B : SWIZZLE_64B
            // descriptors differ only in the 14-bit start-address field (units of 16 bytes): build them once, then add
            const uint64_t adesc0 = smem_desc(sA_u32, (uint32_t)p.R * 16, 128u, 0u);
            const uint64_t bdesc0 = smem_desc(smem_u32(sB), 0u, 8u * (uint32_t)KB * 2, b_layout);
            const uint32_t b_stage_16 = b_stage_bytes >> 4;
            const int ksteps = KB / 16;
            int stage = 0; uint32_t phase = 0; uint32_t accum = 0;
            for (int kb = 0; kb < p.nkb; kb++) {
                mbar_wait(bar_a_full + 8 * kb, 0);
                if (kb == 0) DBG(6);
                asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // cp.async (generic proxy) writes -> UMMA (async proxy) reads
                for (int j = 0; j < p.taps; j++) {
                    mbar_wait(bar_b_full + 8 * stage, phase);
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    const uint64_t bdesc_s = bdesc0 + (uint64_t)((uint32_t)stage * b_stage_16);
                    const uint32_t a_row = (uint32_t)(kb * (KB / 8) * p.R + j * p.dil);     // in rows (= 16-byte units)
                    for (int ks = 0; ks < ksteps; ks++) {
                        const uint64_t adesc = adesc0 + (uint64_t)(a_row + (uint32_t)(ks * 2 * p.R));
                        const uint64_t bdesc = bdesc_s + (uint64_t)(ks * 2);
                        umma_f16(tb, adesc, bdesc, idesc, (accum | (uint32_t)ks) ? 1u : 0u);
                    }
                    accum = 1;
                    umma_commit(bar_b_empty + 8 * stage);   // frees the B slot when these MMAs retire
                    if (++stage == p.stages) { stage = 0; phase ^= 1; }
                }
            }
            umma_commit(bar_acc);
            DBG(5);
        }
        __syncwarp();
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x == 0) DBG(7);
    if (warp == 5) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)N_TILE) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------- kernel v2
// Persistent, fully pipelined variant (the default).  One CTA per SM (up to three for the thin layers) loops over tiles;
// four roles run concurrently on different tiles, connected by mbarrier pipelines:
//   warps 6-9  A producers : cp.async the next tile's rows+halo into a double-buffered A region (per-K-block full/empty
//                            barriers, so a K block is refilled as soon as the MMAs that read it have retired)
//   warp  4    B producer  : TMA weight ring, or -- when all taps of the layer fit -- weights loaded ONCE and kept resident
//   warp  5    MMA issuer  : tcgen05.mma into one of TWO TMEM accumulators
//   warps 0-3  epilogue    : tcgen05.ld -> shared-memory transpose -> coalesced 128-bit residual loads / stores
//                            (8 lanes cover 128 contiguous bytes of one output row), overlapping the next tile's MMAs
struct UmmaParams2 {
    UmmaParams b;
    int mtiles, ntiles, total_tiles;
    int nA;            // A buffers: 2, or 1 when two do not fit (per-K-block recycling still overlaps the refill)
    int resident;      // all (K-block, tap) weight tiles stay in shared memory
    int rows_per_thr;  // A rows handled by one producer thread per K block
    int iters;         // tiles per CTA, ceil(total_tiles / grid)
};

static constexpr int kThreads2 = 320;
// B2_UMMA_PDBG=1: clock64 per CTA (first 160) x tile iteration (first 16) x event -- 0 producer past A_EMPTY(kb 0), 1 producer issued the
// tile's last load, 2 MMA thread past ACC_EMPTY, 3 ... past A_FULL(kb 0), 4 ... committed the tile, 5 epilogue past ACC_FULL, 6 epilogue done
#define PDBG(ev) do { if (p.dbg && blockIdx.x < 160 && it < 16) p.dbg[((size_t)blockIdx.x * 16 + it) * 8 + (ev)] = (unsigned long long)clock64(); } while (0)

// PAIR (N_TILE = 256 only, clusters of two CTAs = the two SMs of a TPC): `tcgen05.mma.cta_group::2`.  The CTAs of a pair work on two consecutive
// 128-row tiles as ONE M = 256 MMA stream issued by the leader (cluster rank 0): each CTA keeps only ITS half of every weight tile (N rows
// [128 * rank, +128): 16 KB per stage, so the ring is 7-8 deep in the shared memory that held 4 stages, and each SM fetches half the weight bytes
// from L2), the tensor core of each SM reads A (4 KB) and half of B (4 KB) per K16 step instead of A + all of B (12 KB) from its own shared memory,
// and each CTA's 128 accumulator rows land in its own TMEM, so the A producers and the epilogue are untouched.  Hand-offs that cross the pair:
//   B_FULL   lives in the leader; both CTAs' TMA loads (`.cta_group::2`) count their bytes there
//   A_FULL   of the leader takes one extra arrival per K block, sent by the peer's (otherwise idle) warp 5 once the peer's rows have landed
//   B_EMPTY / A_EMPTY / ACC_FULL are signalled in both CTAs by the leader's multicast commits
//   ACC_EMPTY of the leader counts the epilogue warps of both CTAs
template <int N_TILE, int MINB, bool PAIR = false>
__global__ void __launch_bounds__(kThreads2, MINB) k_conv_umma_p(const __grid_constant__ CUtensorMap tmap_w, const __grid_constant__ CUtensorMap tmap_h,
                                                                  const UmmaParams2 pp) {
    extern __shared__ __align__(1024) uint8_t smem[];
    pdl_trigger();
    const UmmaParams &p = pp.b;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int KB = p.KB;
    constexpr int NBS = PAIR ? 8 : 4;        // barrier slots of the weight ring
    const uint32_t b_tile_bytes = (uint32_t)(PAIR ? N_TILE / 2 : N_TILE) * KB * 2;
    const uint32_t a_bytes = ((uint32_t)p.R * p.Cin * 2 + 15) & ~15u;
    const int nB = pp.resident ? p.nkb * p.taps : p.stages;
    uint8_t *sB = smem;
    uint8_t *sA = smem + (size_t)nB * b_tile_bytes;
    float *sStage = reinterpret_cast<float *>(sA + (size_t)pp.nA * a_bytes);
    uint64_t *bars = reinterpret_cast<uint64_t *>(reinterpret_cast<uint8_t *>(sStage) + kStageBytes);
    // barrier map: [0,4) b_full  [4,8) b_empty  [8,24) a_full[2][8]  [24,40) a_empty[2][8]  [40,42) acc_full  [42,44) acc_empty
    const uint32_t bar0 = smem_u32(bars);
    auto B_FULL = [&](int s) { return bar0 + 8u * (uint32_t)s; };
    auto B_EMPTY = [&](int s) { return bar0 + 8u * (uint32_t)(NBS + s); };
    auto A_FULL = [&](int buf, int kb) { return bar0 + 8u * (uint32_t)(2 * NBS + buf * 8 + kb); };
    auto A_EMPTY = [&](int buf, int kb) { return bar0 + 8u * (uint32_t)(2 * NBS + 16 + buf * 8 + kb); };
    auto ACC_FULL = [&](int a) { return bar0 + 8u * (uint32_t)(2 * NBS + 32 + a); };
    auto ACC_EMPTY = [&](int a) { return bar0 + 8u * (uint32_t)(2 * NBS + 34 + a); };
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(bars + 2 * NBS + 36);
    const uint32_t crank = PAIR ? cluster_ctarank() : 0u;

    if (threadIdx.x == 0) {
        if (smem_u32(smem) & 1023u) __trap();
        for (int s = 0; s < NBS; s++) { mbar_init(B_FULL(s), 1); mbar_init(B_EMPTY(s), 1); }
        for (int b = 0; b < 2; b++)
            for (int k = 0; k < 8; k++) { mbar_init(A_FULL(b, k), (PAIR && crank == 0) ? 129 : 128); mbar_init(A_EMPTY(b, k), 1); }
        for (int a = 0; a < 2; a++) { mbar_init(ACC_FULL(a), 1); mbar_init(ACC_EMPTY(a), PAIR ? 8 : 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 5) {
        if constexpr (PAIR) {
            asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)(2 * N_TILE)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
        } else {
            asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)(2 * N_TILE)) : "memory");
            asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
        }
    }
    if (warp == 4 && lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(PAIR ? &tmap_h : &tmap_w) : "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();  // the peer's barriers exist before anything is multicast to them
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem_base = *tmem_slot;
    // everything above overlapped the previous kernel (PDL); the weight producer (warp 4) reads nothing a kernel writes and goes straight on
    if (warp != 4) pdl_wait();

    auto tile_coords = [&](int tile, int &w0, int &t0, int &n0) {
        const int mt = (pp.ntiles > 1) ? fdiv(tile, p.m_ntiles) : tile;
        n0 = (tile - mt * pp.ntiles) * N_TILE;
        if (p.nseg > 1) { w0 = mt * p.nseg; t0 = 0; }
        else { w0 = fdiv(mt, p.m_tpw); t0 = (mt - w0 * p.tiles_per_win) * 128; }
    };

    if (warp < 4) {
        // =========================== epilogue ===========================
        float *stg = sStage + warp * 32 * kStageLd;
        const int sub_r = lane >> 3, c4 = lane & 7;
        // both CTAs of a pair run the same number of tiles (the MMAs are shared): tiles past the end are dummies whose rows are
        // all masked (w >= W)
        // The fp32 residual / MRF-sum rows a tile's epilogue will add come from HBM (the tensors are larger than L2): they are pulled
        // into L2 one TILE ahead (lane = row, one 128-byte line per 32-column piece), so that the register prefetch one PIECE ahead
        // only has to cover an L2 hit.  No registers are held across the wait.
        auto l2_prefetch_tile = [&](int tile_n) {
            if (!(p.residual || p.acc_src) || tile_n >= pp.total_tiles) return;
            int w0n, t0n, n0n;
            tile_coords(tile_n, w0n, t0n, n0n);
            const int mn = warp * 32 + lane;
            const int sn = (p.nseg > 1) ? fdiv(mn, p.m_period) : 0;
            const int tn = t0n + (mn - sn * p.period);
            const int wn = w0n + sn;
            if ((tn < p.T) && (sn < p.nseg) && (wn < p.W)) {
                const size_t off = (size_t)(wn * p.T + tn) * p.N + n0n;
                for (int c = 0; c < N_TILE; c += 32) {
                    if (p.residual) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.residual + off + c));
                    if (p.acc_src) asm volatile("prefetch.global.L2 [%0];" ::"l"(p.acc_src + off + c));
                }
            }
        };
        l2_prefetch_tile((int)blockIdx.x);
        for (int it = 0; it < pp.iters; ++it) {
            const int tile = (int)blockIdx.x + it * (int)gridDim.x;
            if (!PAIR && tile >= pp.total_tiles) break;
            l2_prefetch_tile(tile + (int)gridDim.x);
            int w0, t0, n0;
            tile_coords(tile, w0, t0, n0);
            const int acc = it & 1, use = it >> 1;
            const int m = warp * 32 + lane;
            const int s = (p.nseg > 1) ? fdiv(m, p.m_period) : 0;
            const int t = t0 + (m - s * p.period);
            const int w = w0 + s;
            const int grow_own = ((t < p.T) && (s < p.nseg) && (w < p.W)) ? (w * p.T + t) : -1;
            int grow[8];
#pragma unroll
            for (int i = 0; i < 8; i++) grow[i] = __shfl_sync(0xffffffffu, grow_own, i * 4 + sub_r);
            const uint32_t tmem_acc = tmem_base + (uint32_t)(acc * N_TILE) + ((uint32_t)(warp * 32) << 16);
            // The fp32 residual (and the MRF running sum) of a 32-column piece are fetched ONE PIECE AHEAD, the first one before the
            // accumulator barrier is even waited on: loaded right before use they cost a full memory latency per half piece, which made
            // the conv2 launches of stage 0 epilogue-bound (what-if runs: epilogue memory = 2.9 of the 8.1 ms of this kernel family).
            // (the MRF sum, present in one conv out of six, is fetched at the top of its own piece instead: registers)
            float4 res_n[8];
            auto fetch = [&](int c0n) {
                const int coln = n0 + c0n + c4 * 4;
#pragma unroll
                for (int i = 0; i < 8; i++)
                    res_n[i] = (grow[i] >= 0) ? *reinterpret_cast<const float4 *>(p.residual + (size_t)grow[i] * p.N + coln) : make_float4(0.f, 0.f, 0.f, 0.f);
            };
            if (p.residual) fetch(0);
#pragma unroll 1
            for (int c0 = 0; c0 < N_TILE; c0 += 32) {
                const int col = n0 + c0 + c4 * 4;
                const float4 bias = __ldg(reinterpret_cast<const float4 *>(p.bias + col));
                float4 accs[8];
                if (p.acc_src) {
#pragma unroll
                    for (int i = 0; i < 8; i++)
                        accs[i] = (grow[i] >= 0) ? *reinterpret_cast<const float4 *>(p.acc_src + (size_t)grow[i] * p.N + col) : make_float4(0.f, 0.f, 0.f, 0.f);
                }
                if (c0 == 0) {
                    mbar_wait(ACC_FULL(acc), (uint32_t)(use & 1));
                    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                    if (threadIdx.x == 0) PDBG(5);
                }
                {
                    uint32_t a32[32];
                    tmem_ld32(tmem_acc + (uint32_t)c0, a32);
                    if (c0 + 32 >= N_TILE) {
                        // last read of this accumulator: hand it back to the MMA warp
                        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
                        __syncwarp();
                        if (lane == 0) {
                            if constexpr (PAIR) mbar_arrive_cluster(mapa_u32(ACC_EMPTY(acc), 0u));    // the leader's MMA thread waits for both CTAs' epilogues
                            else mbar_arrive(ACC_EMPTY(acc));
                        }
                    }
#pragma unroll
                    for (int i = 0; i < 8; i++)
                        *reinterpret_cast<uint4 *>(stg + lane * kStageLd + i * 4) = make_uint4(a32[4 * i], a32[4 * i + 1], a32[4 * i + 2], a32[4 * i + 3]);
                }
                __syncwarp();
                // Branch-free blocks over the eight row groups (each block guarded by ONE warp-uniform condition): with a branch per row
                // the single epilogue warp of a scheduler ran the rows as one dependent chain, ~2.3k cycles per 32-column piece
                // (B2_UMMA_PDBG: the epilogue, not the MMAs, set the tile period of almost every launch of this kernel).
                float4 v[8];
#pragma unroll
                for (int i = 0; i < 8; i++) v[i] = *reinterpret_cast<const float4 *>(stg + (i * 4 + sub_r) * kStageLd + c4 * 4);
                if (p.residual) {
#pragma unroll
                    for (int i = 0; i < 8; i++) { v[i].x = (v[i].x + bias.x) + res_n[i].x; v[i].y = (v[i].y + bias.y) + res_n[i].y; v[i].z = (v[i].z + bias.z) + res_n[i].z; v[i].w = (v[i].w + bias.w) + res_n[i].w; }
                    if (c0 + 32 < N_TILE) fetch(c0 + 32);
                } else {
#pragma unroll
                    for (int i = 0; i < 8; i++) { v[i].x += bias.x; v[i].y += bias.y; v[i].z += bias.z; v[i].w += bias.w; }
                }
                if (p.acc_src) {
#pragma unroll
                    for (int i = 0; i < 8; i++) { v[i].x = accs[i].x + v[i].x; v[i].y = accs[i].y + v[i].y; v[i].z = accs[i].z + v[i].z; v[i].w = accs[i].w + v[i].w; }
                }
                if (p.div != 1.0f) {
                    // v / div as a reciprocal multiply and one Newton step (q = v * r; q + r * (v - div * q)): no IEEE-division sequence per element
                    const float rcp = __frcp_rn(p.div), nd = -p.div;
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        float q;
                        q = v[i].x * rcp; v[i].x = fmaf(fmaf(nd, q, v[i].x), rcp, q);
                        q = v[i].y * rcp; v[i].y = fmaf(fmaf(nd, q, v[i].y), rcp, q);
                        q = v[i].z * rcp; v[i].z = fmaf(fmaf(nd, q, v[i].z), rcp, q);
                        q = v[i].w * rcp; v[i].w = fmaf(fmaf(nd, q, v[i].w), rcp, q);
                    }
                }
                if (p.out32) {
#pragma unroll
                    for (int i = 0; i < 8; i++)
                        if (grow[i] >= 0) *reinterpret_cast<float4 *>(p.out32 + (size_t)grow[i] * p.N + col) = v[i];
                }
                if (p.outb) {
#pragma unroll
                    for (int i = 0; i < 8; i++) {
                        __nv_bfloat162 h0 = __floats2bfloat162_rn(lrelu_f(v[i].x, p.outb_slope), lrelu_f(v[i].y, p.outb_slope));
                        __nv_bfloat162 h1 = __floats2bfloat162_rn(lrelu_f(v[i].z, p.outb_slope), lrelu_f(v[i].w, p.outb_slope));
                        if (grow[i] >= 0) *reinterpret_cast<uint2 *>(p.outb + (size_t)grow[i] * p.N + col) = make_uint2(*reinterpret_cast<uint32_t *>(&h0), *reinterpret_cast<uint32_t *>(&h1));
                    }
                }
                __syncwarp();
            }
            if (threadIdx.x == 0) PDBG(6);
        }
    } else if (warp == 4) {
        // =========================== B producer (TMA) ===========================
        if (lane == 0) {
            if (pp.resident) {
                mbar_expect_tx(B_FULL(0), (uint32_t)nB * b_tile_bytes);
                for (int kb = 0; kb < p.nkb; kb++)
                    for (int j = 0; j < p.taps; j++)
                        tma_load_3d(smem_u32(sB + (size_t)(kb * p.taps + j) * b_tile_bytes), &tmap_w, B_FULL(0), kb * KB, 0, j);
            } else {
                int stage = 0; uint32_t phase = 0;
                for (int it = 0; it < pp.iters; ++it) {
                    const int tile = (int)blockIdx.x + it * (int)gridDim.x;
                    if (!PAIR && tile >= pp.total_tiles) break;
                    int w0, t0, n0;
                    tile_coords(tile, w0, t0, n0);
                    for (int kb = 0; kb < p.nkb; kb++)
                        for (int j = 0; j < p.taps; j++) {
                            mbar_wait(B_EMPTY(stage), phase ^ 1);
                            if constexpr (PAIR) {
                                // my half of the tile into MY shared memory; the bytes of both halves are counted on the leader's barrier
                                if (crank == 0) mbar_expect_tx(B_FULL(stage), 2 * b_tile_bytes);
                                tma_load_3d_2sm(smem_u32(sB + (size_t)stage * b_tile_bytes), &tmap_h, mapa_u32(B_FULL(stage), 0u), kb * KB,
                                                n0 + (int)crank * (N_TILE / 2), j);
                            } else {
                                mbar_expect_tx(B_FULL(stage), b_tile_bytes);
                                tma_load_3d(smem_u32(sB + (size_t)stage * b_tile_bytes), &tmap_w, B_FULL(stage), kb * KB, n0, j);
                            }
                            if (++stage == p.stages) { stage = 0; phase ^= 1; }
                        }
                }
            }
        }
    } else if (warp == 5) {
        // =========================== MMA issuer ===========================
        // the issue loop runs in one elected thread on the uniform datapath: see k_conv_umma
        const uint32_t tb = __shfl_sync(0xffffffffu, tmem_base, 0);
        if (PAIR && crank != 0) {
            // the peer of a pair issues no MMAs: its warp 5 tells the leader when each K block of the PEER's rows has landed
            if (elect_one()) {
                for (int it = 0; it < pp.iters; ++it) {
                    const int abuf = (pp.nA == 2) ? (it & 1) : 0, ause = (pp.nA == 2) ? (it >> 1) : it;
                    for (int kb = 0; kb < p.nkb; kb++) {
                        mbar_wait(A_FULL(abuf, kb), (uint32_t)(ause & 1));
                        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // cp.async writes -> the tensor core's (async proxy) reads
                        mbar_arrive_cluster(mapa_u32(A_FULL(abuf, kb), 0u));
                    }
                }
            }
        } else if (elect_one()) {
            const uint32_t idesc = (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N_TILE >> 3) << 17) | (((PAIR ? 256u : 128u) >> 4) << 24);
            const uint32_t b_layout = (KB == 64) ? 2u : 4u;
            const uint64_t adesc0 = smem_desc(smem_u32(sA), (uint32_t)p.R * 16, 128u, 0u);
            const uint64_t bdesc0 = smem_desc(smem_u32(sB), 0u, 8u * (uint32_t)KB * 2, b_layout);
            const uint32_t b_tile_16 = b_tile_bytes >> 4, a_buf_16 = a_bytes >> 4;
            const int ksteps = KB / 16;
            int stage = 0; uint32_t phase = 0;
            if (pp.resident) { mbar_wait(B_FULL(0), 0); }
            for (int it = 0; it < pp.iters; ++it) {
                const int tile = (int)blockIdx.x + it * (int)gridDim.x;
                if (!PAIR && tile >= pp.total_tiles) break;
                const int acc = it & 1, use = it >> 1;
                const int abuf = (pp.nA == 2) ? (it & 1) : 0, ause = (pp.nA == 2) ? (it >> 1) : it;
                if constexpr (PAIR) mbar_wait_cluster(ACC_EMPTY(acc), (uint32_t)((use & 1) ^ 1));
                else mbar_wait(ACC_EMPTY(acc), (uint32_t)((use & 1) ^ 1));
                asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                PDBG(2);
                const uint64_t adesc_t = adesc0 + (uint64_t)((uint32_t)abuf * a_buf_16);
                const uint32_t tmem_acc = tb + (uint32_t)(acc * N_TILE);
                uint32_t accum = 0;
                for (int kb = 0; kb < p.nkb; kb++) {
                    if constexpr (PAIR) mbar_wait_cluster(A_FULL(abuf, kb), (uint32_t)(ause & 1));
                    else mbar_wait(A_FULL(abuf, kb), (uint32_t)(ause & 1));
                    if (kb == 0) PDBG(3);
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    for (int j = 0; j < p.taps; j++) {
                        uint64_t bdesc_s;
                        if (pp.resident) bdesc_s = bdesc0 + (uint64_t)((uint32_t)(kb * p.taps + j) * b_tile_16);
                        else {
                            mbar_wait(B_FULL(stage), phase);
                            bdesc_s = bdesc0 + (uint64_t)((uint32_t)stage * b_tile_16);
                        }
                        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
                        const uint32_t a_row = (uint32_t)(kb * (KB / 8) * p.R + j * p.dil);
                        for (int ks = 0; ks < ksteps; ks++) {
                            if constexpr (PAIR) umma_f16_2cta(tmem_acc, adesc_t + (uint64_t)(a_row + (uint32_t)(ks * 2 * p.R)), bdesc_s + (uint64_t)(ks * 2), idesc, accum);
                            else umma_f16(tmem_acc, adesc_t + (uint64_t)(a_row + (uint32_t)(ks * 2 * p.R)), bdesc_s + (uint64_t)(ks * 2), idesc, accum);
                            accum = 1;
                        }
                        if (!pp.resident) {
                            if constexpr (PAIR) umma_commit_2cta(B_EMPTY(stage), (uint16_t)3);
                            else umma_commit(B_EMPTY(stage));
                            if (++stage == p.stages) { stage = 0; phase ^= 1; }
                        }
                    }
                    // this K block of the A buffer may be refilled once these MMAs retire
                    if constexpr (PAIR) umma_commit_2cta(A_EMPTY(abuf, kb), (uint16_t)3);
                    else umma_commit(A_EMPTY(abuf, kb));
                }
                if constexpr (PAIR) umma_commit_2cta(ACC_FULL(acc), (uint16_t)3);
                else umma_commit(ACC_FULL(acc));
                PDBG(4);
            }
        }
        __syncwarp();
    } else {
        // =========================== A producers ===========================
        const int ptid = threadIdx.x - 192;
        const int cshift = (KB == 64) ? 3 : 2;
        const int cpr = 1 << cshift;
        const int rstep = 128 >> cshift;
        const int r_first = ptid >> cshift, c = ptid & (cpr - 1);
        for (int it = 0; it < pp.iters; ++it) {
            const int tile = (int)blockIdx.x + it * (int)gridDim.x;
            if (!PAIR && tile >= pp.total_tiles) break;
            int w0, t0, n0;
            tile_coords(tile, w0, t0, n0);
            const int abuf = (pp.nA == 2) ? (it & 1) : 0, ause = (pp.nA == 2) ? (it >> 1) : it;
            const uint32_t sA_u32 = smem_u32(sA + (size_t)abuf * a_bytes);
            int grow[12];
#pragma unroll
            for (int i = 0; i < 12; i++) {
                const int r = r_first + i * rstep;
                const int u = r - p.pad;
                const int s = (u >= 0 && p.nseg > 1) ? fdiv(u, p.m_period) : 0;
                const int t = t0 + (u - s * p.period);
                const int w = w0 + s;
                const bool ok = (r < p.R) && (t >= 0) && (t < p.T) && (s < p.nseg) && (w < p.W);
                grow[i] = ok ? (w * p.T + t) : -1;
            }
            for (int kb = 0; kb < p.nkb; kb++) {
                mbar_wait(A_EMPTY(abuf, kb), (uint32_t)((ause & 1) ^ 1));
                if (kb == 0 && ptid == 0) PDBG(0);
#pragma unroll
                for (int i = 0; i < 12; i++) {
                    const int r = r_first + i * rstep;
                    if (r < p.R) {
                        const __nv_bfloat16 *src = grow[i] >= 0 ? p.in + (size_t)grow[i] * p.Cin + kb * KB + c * 8 : p.in;
                        cp_async16(sA_u32 + (uint32_t)(((kb * cpr + c) * p.R + r) * 16), src, grow[i] >= 0 ? 16u : 0u);
                    }
                }
                cp_async_arrive_noinc(A_FULL(abuf, kb));
            }
            if (ptid == 0) PDBG(1);
        }
    }

    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if constexpr (PAIR) cluster_sync_all();  // nobody leaves while the peer may still arrive on this CTA's barriers
    if (warp == 5) {
        if constexpr (PAIR) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * N_TILE)) : "memory");
        else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)(2 * N_TILE)) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *, const cuuint64_t *,
                                  const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn g_encode = nullptr;
static std::mutex g_init_mu;
static bool g_attr_set[64][4] = {};

static int n_tile_for(const Layer &l) {
    if (l.Cout >= 256) return (l.Cin >= 512) ? 128 : 256;
    return l.Cout;     // 32, 64, 128
}

int umma_init() {
    std::lock_guard<std::mutex> g(g_init_mu);
    if (g_encode) return 0;
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
    if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn)
        return set_error("cuTensorMapEncodeTiled is not available from the driver: %s", cudaGetErrorString(e));
    g_encode = reinterpret_cast<EncodeTiledFn>(fn);
    return 0;
}

int umma_prepare_layer(Layer &l) {
    if (umma_init()) return 1;
    if (l.Cin % 32 || (l.Cin > 32 && l.Cin % 64) || l.Cin > 64 * kMaxKB) return set_error("conv_umma: unsupported Cin %d", l.Cin);
    const int nt = n_tile_for(l);
    if (l.Cout % nt || (nt != 32 && nt != 64 && nt != 128 && nt != 256)) return set_error("conv_umma: unsupported Cout %d", l.Cout);
    if (l.stride != 1) return set_error("conv_umma: stride must be 1");
    const int KB = l.Cin >= 64 ? 64 : 32;
    CUtensorMap *tm = new CUtensorMap();
    cuuint64_t gdim[3] = {(cuuint64_t)l.Cin, (cuuint64_t)l.Cout, (cuuint64_t)l.taps};
    cuuint64_t gstr[2] = {(cuuint64_t)l.Cin * 2, (cuuint64_t)l.Cin * l.Cout * 2};
    cuuint32_t box[3] = {(cuuint32_t)KB, (cuuint32_t)nt, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = g_encode(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void *)l.wbf, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                          KB == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { delete tm; return set_error("cuTensorMapEncodeTiled failed with CUresult %d (Cin %d Cout %d taps %d)", (int)r, l.Cin, l.Cout, l.taps); }
    l.tmap = tm;
    if (l.Cin == 64 && l.Cout == 128 && l.taps == 3) {
        // upsampler 3 (64 -> 4 x 32): 8 KB boxes of one tap and 32 input channels for the stacked-output ResBlock kernel's weight ring
        CUtensorMap *tq = new CUtensorMap();
        cuuint32_t boxq[3] = {32u, 128u, 1u};
        r = g_encode(tq, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void *)l.wbf, gdim, gstr, boxq, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { delete tq; return set_error("cuTensorMapEncodeTiled (upsampler box) failed with CUresult %d", (int)r); }
        l.tmap_q = tq;
    }
    if (nt == 256 && l.Cout == 256) {
        // the CTA pair of the persistent kernel: the same tensor with a box of half the tile's rows (each CTA loads its half)
        CUtensorMap *th = new CUtensorMap();
        cuuint32_t boxh[3] = {(cuuint32_t)KB, (cuuint32_t)(nt / 2), 1};
        r = g_encode(th, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 3, (void *)l.wbf, gdim, gstr, boxh, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     KB == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { delete th; return set_error("cuTensorMapEncodeTiled (half box) failed with CUresult %d", (int)r); }
        l.tmap_half = th;
    }
    return 0;
}

void umma_free_layer(Layer &l) {
    if (l.tmap) { delete reinterpret_cast<CUtensorMap *>(l.tmap); l.tmap = nullptr; }
    if (l.tmap_half) { delete reinterpret_cast<CUtensorMap *>(l.tmap_half); l.tmap_half = nullptr; }
    if (l.tmap_q) { delete reinterpret_cast<CUtensorMap *>(l.tmap_q); l.tmap_q = nullptr; }
}

template <int NT>
static int launch_nt(const CUtensorMap &tm, const UmmaParams &p, dim3 grid, size_t smem, cudaStream_t st, int slot) {
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    if (dev < 64 && !g_attr_set[dev][slot]) {
        B2_CUDA_OK(cudaFuncSetAttribute(k_conv_umma<NT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        g_attr_set[dev][slot] = true;
    }
    B2_CUDA_OK(launch_k(k_conv_umma<NT>, dim3(grid), dim3(kThreads), smem, st, pdl_enabled(), tm, p));
    B2_LAUNCH_OK("k_conv_umma");
    return 0;
}

// the thin layers (Cout <= 128): one 128-row tile per CTA, many CTAs per SM
static int launch_conv_umma_v1(const UmmaConvArgs &a, cudaStream_t st) {
    const Layer &l = *a.layer;
    if (!l.tmap || !l.wbf) return set_error("conv_umma: layer has no tensor-core weights (context not in B2_MODE_BF16?)");
    if (a.W <= 0 || a.T <= 0) return 0;
    if ((l.taps - 1) * l.dil != 2 * l.pad) return set_error("conv_umma: only 'same' convolutions are supported");
    UmmaParams p;
    p.in = a.in; p.bias = l.bias; p.residual = a.residual; p.acc_src = a.acc_src; p.out32 = a.out32; p.outb = a.outb;
    p.outb_slope = a.outb_slope; p.div = a.div;
    static const bool dbg_on = getenv("B2_UMMA_DBG") != nullptr;
    static unsigned long long *dbg_buf = nullptr;
    if (dbg_on && !dbg_buf) cudaMalloc(&dbg_buf, 8192 * 8 * 8);
    p.dbg = dbg_on ? dbg_buf : nullptr;
    if (dbg_on) cudaMemsetAsync(dbg_buf, 0, 8192 * 8 * 8, st);
    p.W = a.W; p.T = a.T; p.Cin = l.Cin; p.N = l.Cout; p.taps = l.taps; p.dil = l.dil; p.pad = l.pad;
    p.KB = l.Cin >= 64 ? 64 : 32;
    p.nkb = l.Cin / p.KB;
    const int nt = n_tile_for(l);
    p.R = (128 + (l.taps - 1) * l.dil) | 1;
    unsigned mtiles;
    if (a.T < 128) {
        // short windows: several per tile, `pad` zero rows apart
        const int G = l.pad;
        p.nseg = std::max(1, (128 + G) / (a.T + G));
        p.period = a.T + G;
        p.tiles_per_win = 1;
        mtiles = (unsigned)cdiv(a.W, p.nseg);
    } else {
        p.nseg = 1; p.period = 1 << 30; p.tiles_per_win = cdiv(a.T, 128);
        mtiles = (unsigned)((long long)a.W * p.tiles_per_win);
    }
    p.m_period = ((1ull << 40) + (unsigned long long)p.period - 1) / (unsigned long long)p.period;
    p.m_tpw = ((1ull << 40) + (unsigned long long)p.tiles_per_win - 1) / (unsigned long long)p.tiles_per_win;
    p.m_ntiles = 0;
    const size_t a_bytes = (std::max<size_t>((size_t)p.R * l.Cin * 2, (size_t)kStageBytes) + 15) & ~(size_t)15;
    const size_t b_stage = (size_t)nt * p.KB * 2;
    const size_t tail_bytes = (2 * 16 + kMaxKB + 1) * 8 + 16;
    // weight ring: four stages, fewer where shared memory runs out or the layer has fewer (K block, tap) tiles
    int stages = 4;
    while (stages > 2 && stages * b_stage + a_bytes + tail_bytes > 200 * 1024) stages--;
    const int total_b = p.nkb * l.taps;
    if (stages > total_b) stages = std::max(1, total_b);
    p.stages = stages;
    const size_t smem = stages * b_stage + a_bytes + tail_bytes;
    if (smem > 227 * 1024) return set_error("conv_umma: tile needs %zu bytes of shared memory", smem);
    dim3 grid(mtiles, (unsigned)(l.Cout / nt));
    const CUtensorMap &tm = *reinterpret_cast<const CUtensorMap *>(l.tmap);
    int rc;
    switch (nt) {
        case 32: rc = launch_nt<32>(tm, p, grid, smem, st, 0); break;
        case 64: rc = launch_nt<64>(tm, p, grid, smem, st, 1); break;
        default: rc = launch_nt<128>(tm, p, grid, smem, st, 2); break;
    }
    if (dbg_on && !rc) {
        cudaStreamSynchronize(st);
        static std::vector<unsigned long long> h(8192 * 8);
        cudaMemcpy(h.data(), dbg_buf, h.size() * 8, cudaMemcpyDeviceToHost);
        const int n = std::min<int>(8192, (int)grid.x);
        double d[8] = {0}; int cnt = 0;
        unsigned long long tmin = ~0ull, tmax = 0;
        for (int i = 0; i < n; i++) {
            const unsigned long long *r = &h[(size_t)i * 8];
            if (!r[0] || !r[7]) continue;
            cnt++;
            tmin = std::min(tmin, r[0]); tmax = std::max(tmax, r[7]);
            d[0] += (double)(r[1] - r[0]);   // setup: start -> after sync
            d[1] += (double)(r[2] - r[1]);   // A issue
            d[2] += (double)(r[6] - r[1]);   // sync -> A(kb0) landed (seen by MMA thread)
            d[3] += (double)(r[5] - r[6]);   // MMA issue loop (incl. waiting for weights)
            d[4] += (double)(r[3] - r[5]);   // last commit -> accumulator barrier seen by epilogue
            d[5] += (double)(r[4] - r[3]);   // epilogue
            d[6] += (double)(r[7] - r[4]);   // teardown sync
            d[7] += (double)(r[7] - r[0]);   // CTA lifetime
        }
        if (cnt) fprintf(stderr, "[umma dbg] N=%d Cin=%d taps=%d dil=%d grid=%u res=%d out32=%d | ns: setup %.0f, A-issue %.0f, A-landed %.0f, mma-loop %.0f, commit->epi %.0f, epilogue %.0f, teardown %.0f, lifetime %.0f | span %.1f us for %d CTAs\n",
                         nt, l.Cin, l.taps, l.dil, grid.x, a.residual != nullptr, a.out32 != nullptr, d[0] / cnt, d[1] / cnt, d[2] / cnt, d[3] / cnt, d[4] / cnt, d[5] / cnt, d[6] / cnt, d[7] / cnt,
                         (double)(tmax - tmin) / 1e3, cnt);
    }
    return rc;
}


static int g_occ2[64][5] = {};

template <int NT, int MINB, bool PAIR = false>
static int launch_nt2(const CUtensorMap &tm, const CUtensorMap *tm_half, UmmaParams2 &p, size_t smem, cudaStream_t st, int slot) {
    int dev = 0;
    B2_CUDA_OK(cudaGetDevice(&dev));
    if (dev >= 64) return set_error("conv_umma: device index too large");
    if (!g_occ2[dev][slot]) {
        B2_CUDA_OK(cudaFuncSetAttribute(k_conv_umma_p<NT, MINB, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
        g_occ2[dev][slot] = 1;
    }
    int occ = 0;
    B2_CUDA_OK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_conv_umma_p<NT, MINB, PAIR>, kThreads2, smem));
    occ = std::max(1, std::min(occ, std::min(MINB, 512 / (2 * NT))));
    int grid = std::min(p.total_tiles, sm_count() * occ);
    if (PAIR) grid = std::min((p.total_tiles + 1) & ~1, (sm_count() * occ) & ~1);      // whole pairs; a tile past the end is a dummy (all rows masked)
    p.iters = cdiv(p.total_tiles, grid);
    static const bool pdbg_on = getenv("B2_UMMA_PDBG") != nullptr;
    static unsigned long long *pdbg_buf = nullptr;
    constexpr size_t kPdbgWords = 160 * 16 * 8;
    if (pdbg_on) {
        if (!pdbg_buf) cudaMalloc(&pdbg_buf, kPdbgWords * 8);
        cudaMemsetAsync(pdbg_buf, 0, kPdbgWords * 8, st);
        p.b.dbg = pdbg_buf;
    }
    auto report = [&]() {
        if (pdbg_on) {
            cudaStreamSynchronize(st);
            static std::vector<unsigned long long> h(kPdbgWords);
            cudaMemcpy(h.data(), pdbg_buf, kPdbgWords * 8, cudaMemcpyDeviceToHost);
            // steady state: tile iterations 3..min(iters,16)-2 of every CTA
            double d[8] = {0}; int cnt = 0;
            const int hi = std::min(p.iters, 16) - 1;
            for (int c = 0; c < std::min(grid, 160); c++)
                for (int it = 3; it < hi; it++) {
                    const unsigned long long *e = &h[((size_t)c * 16 + it) * 8], *pe = e - 8;
                    if (!e[0] || !e[6] || !pe[4]) continue;
                    cnt++;
                    d[0] += (double)(e[4] - pe[4]);     // tile period (MMA commit to MMA commit)
                    d[1] += (double)(e[4] - e[3]);      // MMA loop: A(kb 0) seen -> tile committed (incl. waiting for weights / later K blocks)
                    d[2] += (double)(e[3] - e[2]);      // MMA thread waiting for the tile's first A block
                    d[3] += (double)((long long)e[2] - (long long)pe[4]);   // MMA thread waiting for a free accumulator
                    d[4] += (double)(e[1] - e[0]);      // producer: issuing the tile's loads (incl. waiting for free K blocks)
                    d[5] += (double)(e[6] - e[5]);      // epilogue of the tile
                    d[6] += (double)((long long)e[5] - (long long)pe[6]);   // epilogue waiting for the next accumulator
                    d[7] += (double)((long long)e[3] - (long long)e[1]);    // last load issued -> first A block seen (negative: loads trail)
                }
            if (cnt) fprintf(stderr, "[umma_p dbg] N=%d Cin=%d taps=%d dil=%d T=%d res=%d out32=%d outb=%d nA=%d stages=%d resident=%d iters=%d | cycles per tile: period %.0f, "
                             "mma-loop %.0f, mma-wait-A %.0f, mma-wait-acc %.0f, producer %.0f, epilogue %.0f, epi-wait-acc %.0f, issue->A-seen %.0f (n=%d)\n",
                             p.b.N, p.b.Cin, p.b.taps, p.b.dil, p.b.T, p.b.residual != nullptr, p.b.out32 != nullptr, p.b.outb != nullptr, p.nA, p.b.stages, p.resident, p.iters,
                             d[0] / cnt, d[1] / cnt, d[2] / cnt, d[3] / cnt, d[4] / cnt, d[5] / cnt, d[6] / cnt, d[7] / cnt, cnt);
        }
    };
    if constexpr (!PAIR) {
        B2_CUDA_OK(launch_k(k_conv_umma_p<NT, MINB, PAIR>, dim3(grid), dim3(kThreads2), smem, st, pdl_enabled(), tm, tm, p));
        B2_LAUNCH_OK("k_conv_umma_p");
        report();
        return 0;
    }
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3(kThreads2); cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute at[2];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = pdl_enabled() ? 2 : 1;
    B2_CUDA_OK(cudaLaunchKernelEx(&cfg, k_conv_umma_p<NT, MINB, PAIR>, tm, *tm_half, (const UmmaParams2)p));
    B2_LAUNCH_OK("k_conv_umma_p (cta_group::2)");
    report();
    return 0;
}

int launch_conv_umma(const UmmaConvArgs &a, cudaStream_t st) {
    // Two kernels, chosen per layer from the round-1 launch lists (profiles/): the persistent pipelined kernel wins on the
    // wide layers (stage 0, the upsamplers); the one-tile-per-CTA kernel with many co-resident CTAs wins on the thin ones,
    // where a tile is too little work to amortise a pipeline hand-off.
    const Layer &l = *a.layer;
    const bool wide = l.Cin >= 256 || l.Cout > l.Cin;
    if (!wide) return launch_conv_umma_v1(a, st);
    if (!l.tmap || !l.wbf) return set_error("conv_umma: layer has no tensor-core weights (context not in B2_MODE_BF16?)");
    if (a.W <= 0 || a.T <= 0) return 0;
    if ((l.taps - 1) * l.dil != 2 * l.pad) return set_error("conv_umma: only 'same' convolutions are supported");
    UmmaParams2 pp;
    UmmaParams &p = pp.b;
    p.in = a.in; p.bias = l.bias; p.residual = a.residual; p.acc_src = a.acc_src; p.out32 = a.out32; p.outb = a.outb;
    p.outb_slope = a.outb_slope; p.div = a.div;
    p.W = a.W; p.T = a.T; p.Cin = l.Cin; p.N = l.Cout; p.taps = l.taps; p.dil = l.dil; p.pad = l.pad;
    p.dbg = nullptr;
    p.R = (128 + (l.taps - 1) * l.dil) | 1;
    p.KB = l.Cin >= 64 ? 64 : 32;
    p.nkb = l.Cin / p.KB;
    const int nt = n_tile_for(l);
    if (a.T < 128) {
        const int G = l.pad;
        p.nseg = std::max(1, (128 + G) / (a.T + G));
        p.period = a.T + G;
        p.tiles_per_win = 1;
        pp.mtiles = cdiv(a.W, p.nseg);
    } else {
        p.nseg = 1; p.period = 1 << 30; p.tiles_per_win = cdiv(a.T, 128);
        pp.mtiles = (int)((long long)a.W * p.tiles_per_win);
    }
    p.m_period = ((1ull << 40) + (unsigned long long)p.period - 1) / (unsigned long long)p.period;
    p.m_tpw = ((1ull << 40) + (unsigned long long)p.tiles_per_win - 1) / (unsigned long long)p.tiles_per_win;
    pp.ntiles = l.Cout / nt;
    p.m_ntiles = ((1ull << 40) + (unsigned long long)pp.ntiles - 1) / (unsigned long long)pp.ntiles;
    pp.total_tiles = pp.mtiles * pp.ntiles;
    const int cpr = p.KB / 8;
    pp.rows_per_thr = cdiv(p.R, 128 / cpr);
    if (pp.rows_per_thr > 12) return set_error("conv_umma: halo too large (%d rows)", p.R);
    const size_t a_bytes = ((size_t)p.R * l.Cin * 2 + 15) & ~(size_t)15;
    // The C = 256 layers (stage 0's 18 ResBlock convs, 4 ms of the step) run as CTA pairs on `tcgen05.mma.cta_group::2` (see k_conv_umma_p, PAIR):
    // the single-CTA launches ran at the SM's shared-memory bandwidth, not at the tensor pipe's pace -- per k = 11 tile 2.1 MB of operand reads
    // + 1.4 MB of TMA writes + 0.35 MB of A / epilogue traffic = 30k cycles at 128 B/cycle against 32.4k measured and 22.5k of tensor-pipe time.
    const bool pair = nt == 256 && pp.ntiles == 1 && l.tmap_half && pp.total_tiles >= 2 && p.KB == 64 && l.Cin >= 256;    // not upsampler 2 (128 -> 256: 0.38 vs 0.35 ms as a pair, launch list r3)
    const size_t b_tile = (size_t)(pair ? nt / 2 : nt) * p.KB * 2;
    const size_t fixed = kStageBytes + (pair ? 56 : 48) * 8 + 16;
    const size_t budget = 225 * 1024;
    const size_t all_w = (size_t)p.nkb * l.taps * b_tile;
    // weights stay resident when the whole CTA then still fits three to an SM; otherwise they stream through a TMA ring
    pp.resident = (!pair && pp.ntiles == 1 && all_w + 2 * a_bytes + fixed <= 72 * 1024) ? 1 : 0;
    size_t b_bytes;
    if (pp.resident) { b_bytes = all_w; p.stages = 0; pp.nA = 2; }
    else {
        // Streamed weights need a DEEP ring before a second A buffer: an N=256 tile consumes 64 B of weights per cycle, i.e. 4 x 32 KB
        // in flight at ~1 us of L2 latency.  (B2_UMMA_PDBG: with two A buffers and a 2-deep ring the MMA loop of the C=256 layers ran
        // at 1.8x its tensor-pipe time, with one A buffer -- K blocks recycled as their MMAs retire -- and 3-4 stages at 1.4x.)
        // So: two A buffers where four stages still fit beside them, else one; then as deep a ring as fits, at most 4 stages
        // (8 for a pair, whose stages are half a tile: 16 KB per CTA).
        int stages = pair ? 8 : 4;
        pp.nA = (4 * b_tile + 2 * a_bytes + fixed > budget) ? 1 : 2;
        while (stages > 2 && stages * b_tile + pp.nA * a_bytes + fixed > budget) stages--;
        p.stages = std::min(stages, std::max(1, p.nkb * l.taps));
        b_bytes = p.stages * b_tile;
    }
    const size_t smem = b_bytes + pp.nA * a_bytes + fixed;
    if (smem > 227 * 1024) return set_error("conv_umma: tile needs %zu bytes of shared memory", smem);
    const CUtensorMap &tm = *reinterpret_cast<const CUtensorMap *>(l.tmap);
    const CUtensorMap *th = reinterpret_cast<const CUtensorMap *>(l.tmap_half);
    switch (nt) {
        case 32: return launch_nt2<32, 3>(tm, nullptr, pp, smem, st, 0);
        case 64: return launch_nt2<64, 2>(tm, nullptr, pp, smem, st, 1);
        case 128: return launch_nt2<128, 1>(tm, nullptr, pp, smem, st, 2);
        default:
            if (pair) return launch_nt2<256, 1, true>(tm, th, pp, smem, st, 4);
            return launch_nt2<256, 1>(tm, nullptr, pp, smem, st, 3);
    }
}

}  // namespace b2
