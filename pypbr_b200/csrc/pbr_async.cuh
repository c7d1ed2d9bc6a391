// pbr_async.cuh — sm_100a asynchronous-copy primitives used by the streamed Cook-Torrance kernels:
// mbarrier (transaction-count completion) + cp.async.bulk (the TMA engine's 1-D bulk copy,
// global -> shared).  A row segment of one channel plane is one contiguous run of bytes, so no
// tensor map is needed; every copy is >= 16 B, 16-byte aligned on both sides.
// (A shared -> global bulk-store epilogue was measured and dropped: profiles/r1_ncu_summary.md.)
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>

namespace pbr {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(arrivals) : "memory");
}
// makes the initialised barriers visible to the async proxy (the copy engine completes on them)
__device__ __forceinline__ void mbar_init_fence() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }

// one arrival + the number of bytes the copies of this phase will deliver
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}

// try_wait suspends the warp in hardware until the phase completes or a time limit expires; with the default limit a warp
// whose tile is late came back ~18 times per tile (YIELD + TRYWAIT + BRA: 4.6 % of the streamed backward's instructions,
// issued in competition with the warps that have work).  So the wait passes a time hint that raises the limit.
constexpr uint32_t kWaitHintNs = 20000;
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "PBR_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
      "@p bra PBR_DONE_%=;\n"
      "bra PBR_WAIT_%=;\n"
      "PBR_DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity), "r"(kWaitHintNs)
      : "memory");
}

// L2 policy for data that is read exactly once
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t pol;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}

// global -> shared bulk copy, completion signalled on `bar` as `bytes` transaction bytes
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar, uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}

}  // namespace pbr
