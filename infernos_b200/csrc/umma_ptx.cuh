// Inline-PTX wrappers for sm_100a: mbarrier, TMA, cp.async, tcgen05 (alloc / mma / commit / ld) and the UMMA
// shared-memory descriptor.  Shared by the tcgen05 convolution kernels.
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace b2 {

// ---------------------------------------------------------------------------------------------------- PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
// try_wait carries a suspend-time hint: without one the hardware's default time limit is a few tens of cycles, and the waiting warps (TMA producer,
// MMA issuers, epilogue warps between sub-tiles) re-issue the try_wait + branch pair all the time -- in k_resblock<32> a quarter of all executed
// warp instructions were this polling (ncu source page, round 2), on the same schedulers the epilogue math needs.  With the hint the warp is parked
// until the phase completes (or the limit passes).
#ifndef B2_MBAR_HINT_NS
#define B2_MBAR_HINT_NS 0x989680
#endif
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n\t"
        "@P1 bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(bar), "r"(parity), "r"((uint32_t)B2_MBAR_HINT_NS) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const void *tmap, uint32_t bar, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(dst), "l"(tmap), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// ---- cta_group::2: the two CTAs of a cluster (one TPC) drive ONE M = 256 MMA.  The leader (cluster rank 0) issues it; each CTA supplies its 128 rows of A
// and its half of B's N rows from its own shared memory (same offsets in both) and receives its 128 accumulator rows in its own TMEM.
__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t cta_rank) {
    uint32_t r;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(cta_rank));
    return r;
}
// arrive on a barrier of another CTA of the cluster (address from mapa_u32)
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// wait on an own barrier that the peer CTA also arrives on
__device__ __forceinline__ void mbar_wait_cluster(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 P1, [%0], %1, %2;\n\t"
        "@P1 bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(bar), "r"(parity), "r"((uint32_t)B2_MBAR_HINT_NS) : "memory");
}
// TMA load into OWN shared memory whose completion bytes are counted on a barrier of the pair's leader (cluster address)
__device__ __forceinline__ void tma_load_3d_2sm(uint32_t dst, const void *tmap, uint32_t bar_cluster, int c0, int c1, int c2) {
    asm volatile("cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(dst), "l"(tmap), "r"(bar_cluster), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
// arrives on the barrier at this offset in every CTA of cta_mask once the pair's MMAs issued so far have retired
__device__ __forceinline__ void umma_commit_2cta(uint32_t bar, uint16_t cta_mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar), "h"(cta_mask) : "memory");
}
__device__ __forceinline__ void umma_f16_2cta(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void cp_async16(uint32_t dst, const void *src, uint32_t src_bytes) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) {
    asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&v)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
          "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
          "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
          "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
        : "r"(taddr));
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// shared memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout, version 1 = sm_100)
__device__ __forceinline__ uint64_t smem_desc(uint32_t addr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout_type) {
    uint64_t d = 0;
    d |= (uint64_t)((addr >> 4) & 0x3FFF);
    d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)(layout_type & 7) << 61;
    return d;
}

// n / d for 0 <= n < 2^24, d < 2^16, with m = ceil(2^40 / d): a multiply and a shift instead of a ~40-instruction division
__device__ __forceinline__ int fdiv(int n, unsigned long long m) { return (int)(((unsigned long long)(unsigned)n * m) >> 40); }

__device__ __forceinline__ float lrelu_f(float v, float slope) { return v > 0.0f ? v : v * slope; }


// one lane of a fully active warp (the same lane every time): the thread that issues tcgen05.mma / tcgen05.commit
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

}  // namespace b2
