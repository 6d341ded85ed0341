// tma.cuh -- 1-D bulk asynchronous copies global -> shared memory (TMA engine, cp.async.bulk) with
// mbarrier completion, as raw PTX for sm_100a.  One elected lane issues a copy of a whole contiguous
// (stage, group) record; consumers spin on the barrier's phase parity.  Used to stream the serial,
// latency-bound recursions (k_riccati) so that the next stage's record lands in shared memory
// while the current stage is being factorised.
//
// Rules the callers follow: destination / source 16-byte aligned, size a multiple of 16; a buffer
// is re-armed only after every lane has finished reading it (a __syncwarp() between the last read
// and the issuing lane's next copy); barriers are initialised by one lane, then made visible with
// fence.mbarrier_init + __syncwarp().
#pragma once
#ifndef IDOCP_B200_EMU
#include <cuda_runtime.h>
#include <cstdint>
#else
#include <cstdint>
#include <cstring>
#include "cuda_emu.h"
#endif

namespace idocp_b200 {

#ifndef IDOCP_B200_EMU
// a shared-memory address in the form the async-copy instructions take; a loop that re-issues copies into
// the same buffers converts its destinations and barriers once (smem_addr) and passes these
using smem_t = uint32_t;
__device__ __forceinline__ smem_t smem_addr(const void* p) {
  return static_cast<smem_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void tma_bar_init(uint64_t* bar, int arrivals) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(arrivals));
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
// arm the barrier with the number of bytes the following copies will deliver (one arrival)
__device__ __forceinline__ void tma_bar_expect(smem_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bar_expect(uint64_t* bar, uint32_t bytes) { tma_bar_expect(smem_addr(bar), bytes); }
__device__ __forceinline__ void tma_load_1d(smem_t dst_smem, const void* src_gmem, uint32_t bytes, smem_t bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst_smem),
               "l"(src_gmem), "r"(bytes), "r"(bar)
               : "memory");
}
__device__ __forceinline__ void tma_load_1d(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  tma_load_1d(smem_addr(dst_smem), src_gmem, bytes, smem_addr(bar));
}
// orders this thread's earlier generic-proxy global writes before later async-proxy (TMA) reads;
// every writer executes it, then the warp synchronises, then the elected lane issues the copy
__device__ __forceinline__ void tma_fence_global_writes() { asm volatile("fence.proxy.async.global;" ::: "memory"); }
__device__ __forceinline__ void tma_bar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "TMA_WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra TMA_DONE_%=;\n"
      "bra TMA_WAIT_%=;\n"
      "TMA_DONE_%=:\n"
      "}\n" ::"r"(smem_addr(bar)),
      "r"(parity)
      : "memory");
}
#else
// SIMT-emulator build (tests only): the copy itself happens at issue time, but the barrier keeps real
// phase semantics (low word = completed phases, high word = bytes still expected), so a consumer
// that runs ahead of the issuing lane blocks exactly as on the GPU, and a missing __syncwarp()
// before a re-arm corrupts the buffer under the lanes that still read it (caught by the parity tests).
// shared memory is host memory here: an "address" is the pointer itself, with byte arithmetic as on the GPU
using smem_t = uintptr_t;
inline smem_t smem_addr(const void* p) { return reinterpret_cast<smem_t>(p); }
inline void tma_bar_init(uint64_t* bar, int) { *bar = 0; }
inline void tma_bar_expect(uint64_t* bar, uint32_t bytes) { *bar += static_cast<uint64_t>(bytes) << 32; }
inline void tma_bar_expect(smem_t bar, uint32_t bytes) { tma_bar_expect(reinterpret_cast<uint64_t*>(bar), bytes); }
inline void tma_load_1d(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
  std::memcpy(dst, src, bytes);
  *bar -= static_cast<uint64_t>(bytes) << 32;
  if ((*bar >> 32) == 0) *bar += 1;   // all expected bytes landed: phase complete
}
inline void tma_load_1d(smem_t dst, const void* src, uint32_t bytes, smem_t bar) {
  tma_load_1d(reinterpret_cast<void*>(dst), src, bytes, reinterpret_cast<uint64_t*>(bar));
}
inline void tma_bar_wait(uint64_t* bar, uint32_t parity) {
  while ((static_cast<uint32_t>(*bar) & 1u) == parity) emu::yield();
}
inline void tma_fence_global_writes() {}
#endif

}  // namespace idocp_b200
