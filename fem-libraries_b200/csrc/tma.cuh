// tma.cuh -- mbarrier, 1-D bulk copy (cp.async.bulk -> UBLKCP) and cp.async helpers (sm_100a).
#pragma once
#include "common.cuh"

namespace femb {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
   asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
   asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// raises the phase's transaction count without an arrival (the arrival follows once the thread's own stores are done)
__device__ __forceinline__ void mbar_expect_tx_only(uint64_t *bar, uint32_t bytes)
{
   asm volatile("mbarrier.expect_tx.relaxed.cta.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
   asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// The try_wait carries a suspend-time hint: the waiting warp is parked by the hardware until the phase completes (or
// the hint expires) instead of re-issuing the probe -- without it 17 % of the SpMV's executed instructions were the
// spin loop (SYNCS + BRA + YIELD; ncu, n = 5792), issue slots and power the working warps of the SM pay for.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
   const uint32_t ticks = 0x989680u;  // arbitrarily large: the wait ends with the phase, not with the timer
   asm volatile(
       "{\n"
       ".reg .pred P1;\n"
       "LAB_WAIT:\n"
       "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1, %2;\n"
       "@P1 bra DONE;\n"
       "bra LAB_WAIT;\n"
       "DONE:\n"
       "}" ::"r"(smem_u32(bar)),
       "r"(parity), "r"(ticks)
       : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
   asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                    smem_u32(dst)),
                "l"(src), "r"(bytes), "r"(smem_u32(bar))
                : "memory");
}

// 16-byte asynchronous gather global -> shared (LDGSTS), L2 only
__device__ __forceinline__ void cp_async16(void *dst, const void *src)
{
   asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait()
{
   asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}
// barrier over a subset of the CTA's warps (id 1..15, nthreads a multiple of 32)
__device__ __forceinline__ void named_bar_sync(int id, int nthreads)
{
   asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

}  // namespace femb
