// tma.cuh -- minimal TMA (cp.async.bulk.tensor) + mbarrier helpers for sm_100a.
// SASS evidence: UTMALDG (tensor load), SYNCS.* (mbarrier).  No CUTLASS dependency.
#pragma once

#include <cuda.h>   // CUtensorMap (types only; the encoder is fetched through cudaGetDriverEntryPoint)
#include <cuda_runtime.h>
#include <stdint.h>

namespace cc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_fence_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
// one lane of a converged warp (ELECT: no S2R of the lane id, which the compiler otherwise
// rematerialises per frame in the register-bound consumers)
__device__ __forceinline__ bool elect_one() {
    uint32_t p;
    asm volatile("{ .reg .pred q; elect.sync _|q, 0xffffffff; selp.u32 %0, 1, 0, q; }" : "=r"(p));
    return p != 0;
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;"
                 :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return done != 0;
}
// try_wait with a suspend-time hint: the hardware parks the warp for up to `ns` (no instructions
// issued meanwhile) and wakes it when the phase completes.
__device__ __forceinline__ bool mbar_try_wait_hint(uint64_t* bar, uint32_t parity, uint32_t ns) {
    uint32_t done;
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t"
        "}"
        : "=r"(done) : "r"(smem_u32(bar)), "r"(parity), "r"(ns) : "memory");
    return done != 0;
}
// producer side: long parked waits (a free stage appears once per item, microseconds apart)
template <int HINT_NS>
__device__ __forceinline__ void mbar_wait_parked(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait_hint(bar, parity, HINT_NS)) {}
}
// Polling costs issue slots that other CTAs on the SM could use: back off between probes.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    if (mbar_try_wait(bar, parity)) return;
    while (!mbar_try_wait(bar, parity)) __nanosleep(256);
}

// L2 eviction-priority policy for the staged boxes (createpolicy): the source lines of a box are
// wanted again by the neighbouring tiles (halo) within microseconds, the output never is
__device__ __forceinline__ uint64_t l2_evict_last() {
    uint64_t pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
// 3-D tiled tensor load global -> shared with an L2 cache policy, completion signalled on an mbarrier
__device__ __forceinline__ void tma_load_3d_hint(void* smem_dst, const CUtensorMap* map, uint64_t* bar,
                                                 int c0, int c1, int c2, uint64_t policy) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes.L2::cache_hint"
        " [%0], [%1, {%3, %4, %5}], [%2], %6;"
        :: "r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)),
           "r"(c0), "r"(c1), "r"(c2), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

}  // namespace cc
