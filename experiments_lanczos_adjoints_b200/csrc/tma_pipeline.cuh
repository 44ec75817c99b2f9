// TMA bulk-copy + mbarrier pipeline helpers (sm_100a).
//
// The basis-streaming kernels stage rows of the Krylov basis in shared memory with the TMA
// engine (`cp.async.bulk.shared::cluster.global`, SASS `UBLKCP`): one elected producer thread
// issues 1-D bulk copies of contiguous row segments, completion is signalled on an mbarrier
// (`complete_tx::bytes`), consumer warps wait on the "full" barrier, read the stage with
// LDS.128 and release it through an "empty" barrier.  No registers are spent on loads in
// flight, so a block keeps tens of KB outstanding regardless of occupancy.
#pragma once

#include <cstdint>

namespace bl {
namespace tma {

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}

// make barrier initialisation visible to the async proxy before the first bulk copy
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}

__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred P1;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
      "@P1 bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}

// 1-D bulk copy global -> shared; `bytes` multiple of 16, both addresses 16-byte aligned.
__device__ __forceinline__ void bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
          smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
      : "memory");
}

// same, with an L2 eviction-priority hint (createpolicy result)
__device__ __forceinline__ void bulk_g2s_hint(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar,
                                              uint64_t policy) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;" ::
          "r"(smem_u32(dst_smem)),
      "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
      : "memory");
}

__device__ __forceinline__ uint64_t policy_evict_first() {
  uint64_t p;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
  return p;
}

// 2-D tiled TMA load through a tensor map (`cp.async.bulk.tensor`, SASS UTMALDG): one
// instruction moves a [box_rows x box_cols] box; elements outside the tensor are zero-filled
// and the mbarrier always receives the full box size.
__device__ __forceinline__ void tensor_g2s_2d(void* dst_smem, const void* tensor_map, int col, int row,
                                              uint64_t* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];" ::
          "r"(smem_u32(dst_smem)),
      "l"(reinterpret_cast<uint64_t>(tensor_map)), "r"(col), "r"(row), "r"(smem_u32(bar))
      : "memory");
}
__device__ __forceinline__ void prefetch_tensormap(const void* tensor_map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tensor_map)) : "memory");
}

// named barrier among `nthreads` threads (ids 1..15; 0 is __syncthreads)
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}

// Programmatic dependent launch (PDL): a kernel launched with the programmatic-stream-
// serialization attribute may start while its predecessor is still draining; it must execute
// `griddep_wait` before touching anything the predecessor wrote.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;"); }

}  // namespace tma
}  // namespace bl
