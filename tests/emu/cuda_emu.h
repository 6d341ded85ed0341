// cuda_emu.h -- TEST INFRASTRUCTURE ONLY: a tiny SIMT emulator so the CUDA sources of
// idocp_b200/csrc can be compiled with g++ and stepped on the CPU-only build container
// (no GPU there; every real-GPU run costs a gpurun call).
//
// It is NOT a fallback: the product package (idocp_b200/) only ever loads the nvcc-built
// libidocp_b200.so and fails loudly without it.  The emulator library is built by
// tests/emu/Makefile into tests/emu/libidocp_b200_emu.so and is loaded explicitly, by path,
// from `-m "not gpu"` tests that check the lane-parallel algorithms against the oracle.
//
// Model: every CUDA thread of a block is a ucontext fiber; warp/block barriers and shuffles
// are cooperative round-robin rendezvous.  Blocks run one after another.
#pragma once
#include <ucontext.h>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <vector>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline __attribute__((always_inline))
#define __noinline__ inline
#define __restrict__ __restrict
#define __launch_bounds__(...)
#define __constant__ static
#define __shared__ static

struct dim3 {
  unsigned x, y, z;
  dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
struct uint3_emu {
  unsigned x, y, z;
};

namespace emu {
struct Fiber {
  ucontext_t ctx;
  char* stack = nullptr;
  bool done = false;
};
struct Block {
  int nthreads = 0;
  int cur = 0;
  ucontext_t main;
  std::vector<Fiber> fibers;
  // barriers
  int block_arrived = 0, block_gen = 0;
  int warp_arrived[64] = {0}, warp_gen[64] = {0};
  double xbuf[2048];
  std::function<void()> body;
  std::vector<char> smem;
};
extern Block* g_block;
extern thread_local int t_dummy;
// cudaEventCreate hands out distinct non-null tokens; events created and not yet destroyed (idocp_b200_emu_live_events)
extern long long g_event_serial, g_live_events;
void yield();
void warp_barrier();
void block_barrier();
void launch(dim3 grid, dim3 block, size_t smem_bytes, const std::function<void()>& body);
extern uint3_emu threadIdx_, blockIdx_, blockDim_, gridDim_;
inline int warp_nthreads(int w) {
  const int n = g_block->nthreads - w * 32;
  return n > 32 ? 32 : n;
}
}  // namespace emu

#define threadIdx (emu::threadIdx_)
#define blockIdx (emu::blockIdx_)
#define blockDim (emu::blockDim_)
#define gridDim (emu::gridDim_)

inline void __syncwarp(unsigned = 0xffffffffu) { emu::warp_barrier(); }
inline void __syncthreads() { emu::block_barrier(); }

template <typename T>
inline T emu_exchange(T x, int src_lane_in_warp) {
  static_assert(sizeof(T) <= 8, "emu shuffle supports <= 8 byte types");
  const int tid = threadIdx.x;
  double slot = 0;
  std::memcpy(&slot, &x, sizeof(T));
  emu::g_block->xbuf[tid] = slot;
  emu::warp_barrier();
  const int w = tid / 32;
  double got = emu::g_block->xbuf[w * 32 + src_lane_in_warp];
  emu::warp_barrier();
  T r;
  std::memcpy(&r, &got, sizeof(T));
  return r;
}
template <typename T>
inline T __shfl_sync(unsigned, T x, int src, int width = 32) {
  const int lane = threadIdx.x & 31;
  const int base = lane & ~(width - 1);
  return emu_exchange(x, base + (src & (width - 1)));
}
template <typename T>
inline T __shfl_up_sync(unsigned, T x, unsigned d, int width = 32) {
  const int lane = threadIdx.x & 31;
  const int base = lane & ~(width - 1);
  const int src = lane - (int)d;
  return emu_exchange(x, src < base ? lane : src);
}
template <typename T>
inline T __shfl_down_sync(unsigned, T x, unsigned d, int width = 32) {
  const int lane = threadIdx.x & 31;
  const int base = lane & ~(width - 1);
  const int src = lane + (int)d;
  return emu_exchange(x, src >= base + width ? lane : src);
}
template <typename T>
inline T __shfl_xor_sync(unsigned, T x, int m, int width = 32) {
  const int lane = threadIdx.x & 31;
  const int base = lane & ~(width - 1);
  const int src = lane ^ m;
  return emu_exchange(x, (src >= base + width || src < base) ? lane : src);
}
// mma.sync.aligned.m8n8k4.row.col.f64 as the ascending fma chain the B200 was measured to execute (tools/dmma_probe.cu):
// a = A[g][t], b = B[t][g], d = C[g][2 t + {0, 1}], g = lane / 4, t = lane % 4; one rendezvous for both operand fragments
inline void emu_dmma_m8n8k4(double& d0, double& d1, double a, double b) {
  const int tid = threadIdx.x, w = tid / 32, lane = tid & 31, g = lane >> 2, t = lane & 3;
  emu::g_block->xbuf[tid] = a;
  emu::g_block->xbuf[1024 + tid] = b;
  emu::warp_barrier();
  const double* xa = emu::g_block->xbuf + w * 32;
  const double* xb = emu::g_block->xbuf + 1024 + w * 32;
  for (int k = 0; k < 4; ++k) {
    d0 = std::fma(xa[g * 4 + k], xb[(2 * t) * 4 + k], d0);
    d1 = std::fma(xa[g * 4 + k], xb[(2 * t + 1) * 4 + k], d1);
  }
  emu::warp_barrier();
}
inline int __any_sync(unsigned, int pred) {
  const int tid = threadIdx.x;
  emu::g_block->xbuf[tid] = pred ? 1.0 : 0.0;
  emu::warp_barrier();
  const int w = tid / 32;
  int any = 0;
  for (int l = 0; l < emu::warp_nthreads(w); ++l) any |= (emu::g_block->xbuf[w * 32 + l] != 0.0);
  emu::warp_barrier();
  return any;
}
template <typename T>
inline T __ldg(const T* p) { return *p; }
template <typename T>
inline T __ldcg(const T* p) { return *p; }
inline double __drcp_rn(double x) { return 1.0 / x; }
inline double __dsqrt_rn(double x) { return std::sqrt(x); }
inline double __ddiv_rn(double a, double b) { return a / b; }
inline double __fma_rn(double a, double b, double c) { return std::fma(a, b, c); }

// runtime API shim ---------------------------------------------------------------------------
typedef int cudaError_t;
typedef void* cudaStream_t;
typedef void* cudaEvent_t;
enum { cudaSuccess = 0 };
enum cudaMemcpyKind { cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice, cudaMemcpyDefault };
inline cudaError_t cudaMalloc(void** p, size_t n) { *p = std::calloc(n ? n : 1, 1); return *p ? 0 : 2; }
template <typename T>
inline cudaError_t cudaMalloc(T** p, size_t n) { return cudaMalloc((void**)p, n); }
inline cudaError_t cudaFree(void* p) { std::free(p); return 0; }
inline cudaError_t cudaMallocHost(void** p, size_t n) { return cudaMalloc(p, n); }
template <typename T>
inline cudaError_t cudaMallocHost(T** p, size_t n) { return cudaMalloc((void**)p, n); }
inline cudaError_t cudaFreeHost(void* p) { std::free(p); return 0; }
inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind) { std::memcpy(d, s, n); return 0; }
inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind, cudaStream_t = nullptr) {
  std::memcpy(d, s, n);
  return 0;
}
inline cudaError_t cudaMemset(void* d, int v, size_t n) { std::memset(d, v, n); return 0; }
inline cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t = nullptr) { std::memset(d, v, n); return 0; }
inline cudaError_t cudaSetDevice(int) { return 0; }
inline cudaError_t cudaGetDevice(int* d) { *d = 0; return 0; }
inline cudaError_t cudaGetDeviceCount(int* n) { *n = 1; return 0; }
inline cudaError_t cudaStreamCreate(cudaStream_t* s) { *s = nullptr; return 0; }
inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = nullptr; return 0; }
inline cudaError_t cudaStreamDestroy(cudaStream_t) { return 0; }
inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return 0; }
inline cudaError_t cudaDeviceSynchronize() { return 0; }
inline cudaError_t cudaGetLastError() { return 0; }
inline cudaError_t cudaPeekAtLastError() { return 0; }
inline const char* cudaGetErrorString(cudaError_t) { return "emu"; }
inline cudaError_t cudaEventCreate(cudaEvent_t* e) {
  *e = reinterpret_cast<cudaEvent_t>(++emu::g_event_serial);
  ++emu::g_live_events;
  return 0;
}
inline cudaError_t cudaEventDestroy(cudaEvent_t e) {
  if (e) --emu::g_live_events;
  return 0;
}
inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t = nullptr) { return 0; }
inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return 0; }
inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t) { *ms = 0.f; return 0; }
#define cudaStreamNonBlocking 1
template <typename F>
inline cudaError_t cudaFuncSetAttribute(F, int, int) { return 0; }
#define cudaFuncAttributeMaxDynamicSharedMemorySize 8
// one emulated SM: persistent kernels launch 2 CTAs and loop over their tasks (the multi-task path is what the tests exercise)
#define cudaDevAttrMultiProcessorCount 16
inline cudaError_t cudaDeviceGetAttribute(int* v, int, int) { *v = 1; return 0; }

inline void sincos_emu(double x, double* s, double* c) { *s = std::sin(x); *c = std::cos(x); }
