// devmath.cu -- TEST INFRASTRUCTURE ONLY: the device math building blocks of the kernels (canonical arithmetic of
// octet.cuh, SE(3) of fb_math.cuh, the task-space pose error of task_space_cost.cuh, the warp Cholesky of warp_llt.cuh
// and the interior-point fraction rule of pdipm.cuh), called directly on arrays of inputs.  The product headers are
// included unchanged.  The same file builds with nvcc and the product's flags (-fmad=false) for the B200, and with g++
// against the SIMT emulator of tests/emu for the CPU-only machines; tests/test_device_math.py compares both builds
// with high-precision references and with each other.
//
// Every entry point takes host arrays, copies them to the device, runs one thin kernel, synchronises and copies the
// results back; it returns 0 or the CUDA error code.
#ifdef IDOCP_B200_EMU
#include "cuda_emu.h"
#define DM_LAUNCH(kern, grid, block, ...) emu::launch(dim3(grid), dim3(block), 0, [&]() { kern(__VA_ARGS__); })
#else
#include <cuda_runtime.h>
#define DM_LAUNCH(kern, grid, block, ...) kern<<<(grid), (block)>>>(__VA_ARGS__)
#endif

#include "fb_math.cuh"
#include "pdipm.cuh"
#include "task_space_cost.cuh"
#include "warp_llt.cuh"

using namespace idocp_b200;

// one thread per input: the scalar / SE(3) function `fn` reads DM_IN doubles of its row and writes DM_OUT doubles
constexpr int DM_IN = 40, DM_OUT = 40;
enum DmFn {
  DM_SINCOS, DM_LOG, DM_RSQRT, DM_PIVOT_OK, DM_ACOS, DM_LOG3_CANON, DM_JLOG3_CANON, DM_FB_LOG3, DM_FB_JLOG3, DM_FB_LOG6,
  DM_FB_JLOG6, DM_FB_EXP6, DM_FB_JEXP6, DM_FB_JEXP3, DM_FB_R_TO_QUAT, DM_FB_QUAT_TO_R, DM_FB_INV33, DM_FB_INTEGRATE,
  DM_FB_SUBTRACT, DM_FB_DSUBTRACT_DPLUS, DM_FB_DSUBTRACT_DMINUS, DM_FB_DSUBTRACT_INVERSE, DM_FB_DINTEGRATE_DQ,
  DM_FB_DINTEGRATE_DV, DM_FRACTION_ROW, DM_NUM_FN
};

__global__ void k_dm_scalar(int fn, const double* in_all, double* out_all, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const double* in = in_all + static_cast<size_t>(i) * DM_IN;
  double* out = out_all + static_cast<size_t>(i) * DM_OUT;
  switch (fn) {
    case DM_SINCOS: canon_sincos(in[0], out, out + 1); break;
    case DM_LOG: out[0] = canon_log(in[0]); break;
    case DM_RSQRT: out[0] = canon_rsqrt(in[0]); break;
    case DM_PIVOT_OK: out[0] = canon_pivot_ok(in[0]) ? 1.0 : 0.0; break;
    case DM_ACOS: out[0] = canon_acos(in[0]); break;
    case DM_LOG3_CANON: {
      const V3 w = log3_canon(in, out[0]);
      out[1] = w.x; out[2] = w.y; out[3] = w.z;
      break;
    }
    case DM_JLOG3_CANON: jlog3_canon(in[0], V3{in[1], in[2], in[3]}, out); break;
    case DM_FB_LOG3: fb_log3(in, out, out + 1); break;
    case DM_FB_JLOG3: fb_Jlog3(in[0], in + 1, out); break;
    case DM_FB_LOG6: fb_log6(in, in + 9, out); break;
    case DM_FB_JLOG6: fb_Jlog6(in, in + 9, out); break;
    case DM_FB_EXP6: fb_exp6(in, out, out + 9); break;
    case DM_FB_JEXP6: fb_Jexp6(in, out); break;
    case DM_FB_JEXP3: fb_Jexp3(in, out); break;
    case DM_FB_R_TO_QUAT: fb_R_to_quat(in, out); break;
    case DM_FB_QUAT_TO_R: fb_quat_to_R(in, out); break;
    case DM_FB_INV33: fb_inv33(in, out); break;
    case DM_FB_INTEGRATE: fb_integrate(in, in + FB_NQ, in[FB_NQ + FB_NV], out); break;
    case DM_FB_SUBTRACT: fb_subtract(in, in + FB_NQ, out); break;
    case DM_FB_DSUBTRACT_DPLUS: fb_dsubtract_dplus(in, in + FB_NQ, out); break;
    case DM_FB_DSUBTRACT_DMINUS: fb_dsubtract_dminus(in, in + FB_NQ, out); break;
    case DM_FB_DSUBTRACT_INVERSE: fb_dsubtract_inverse(in, out); break;
    case DM_FB_DINTEGRATE_DQ: fb_dintegrate_dq(in, out); break;
    case DM_FB_DINTEGRATE_DV: fb_dintegrate_dv(in, out); break;
    case DM_FRACTION_ROW: out[0] = pdipm_fraction_row(in[0], in[1], in[2], in[3]); break;
    default: break;
  }
}

// one octet per input: lane l of the octet gets the world placement (R, p) of "its joint" from in[12 l .. 12 l + 11]
// (lane 6 carries the end-effector pose), the end-effector placement is the identity and the reference is
// in[96 .. 107]; the output is the pose error diff (6) followed by the JJ column of every lane (8 x 6).
constexpr int DM_TASK_IN = 8 * 12 + 12, DM_TASK_OUT = 6 + 8 * 6;
__global__ void k_dm_task(const double* in_all, double* out_all, int n) {
  const int lane = threadIdx.x & 7;
  const int i = (blockIdx.x * blockDim.x + threadIdx.x) >> 3;
  const int src = i < n ? i : n - 1;   // octets past the end shadow the last input (never stored); shuffles need them
  const double* in = in_all + static_cast<size_t>(src) * DM_TASK_IN;
  double R[9];
  for (int k = 0; k < 9; ++k) R[k] = in[12 * lane + k];
  const V3 p = V3{in[12 * lane + 9], in[12 * lane + 10], in[12 * lane + 11]};
  const double ee[12] = {1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0, 1.0, 0.0, 0.0, 0.0};
  TaskEval te;
  task_evaluate<true>(R, p, ee, in + 96, te, 1);
  if (i >= n) return;
  double* out = out_all + static_cast<size_t>(i) * DM_TASK_OUT;
  if (lane == 0)
    for (int k = 0; k < 6; ++k) out[k] = te.diff[k];
  for (int k = 0; k < 6; ++k) out[6 + 6 * lane + k] = te.JJ[k];
}

// one warp per matrix: warp_llt of the column-major n x n input (only its lower triangle is meant to be read), then
// lane c < n solves column c of (L L^T)^-1.  Output per matrix: the factor as left in A (n x n column-major), the
// pivot reciprocals rd (n), the return value of warp_llt, and the inverse (n x n column-major).
template <int n>
__global__ void k_dm_llt(const double* in_all, double* out_all) {
  alignas(16) __shared__ double A[n * n];
  alignas(16) __shared__ double LT[n * n];
  alignas(16) __shared__ double rd[n];
  const int wl = threadIdx.x & 31;
  const double* in = in_all + static_cast<size_t>(blockIdx.x) * n * n;
  double* out = out_all + static_cast<size_t>(blockIdx.x) * (2 * n * n + n + 1);
  for (int e = wl; e < n * n; e += 32) { A[e] = in[e]; LT[e] = 0.0; }
  __syncwarp();
  const int fail = warp_llt<n, n>(A, LT, rd, wl);
  double y[n];
  warp_llt_solve_unit<n, n>(A, LT, rd, wl < n ? wl : 0, y);
  __syncwarp();
  for (int e = wl; e < n * n; e += 32) out[e] = A[e];
  for (int e = wl; e < n; e += 32) out[n * n + e] = rd[e];
  if (wl == 0) out[n * n + n] = static_cast<double>(fail);
  if (wl < n)
    for (int r = 0; r < n; ++r) out[n * n + n + 1 + wl * n + r] = y[r];
}

namespace {
struct DevBuf {
  double* p = nullptr;
  ~DevBuf() { if (p) cudaFree(p); }
};
int dm_run(size_t in_count, size_t out_count, const double* in, double* out, void (*launch)(const double*, double*)) {
  DevBuf din, dout;
  cudaError_t e = cudaMalloc(&din.p, in_count * sizeof(double));
  if (e == cudaSuccess) e = cudaMalloc(&dout.p, out_count * sizeof(double));
  if (e == cudaSuccess) e = cudaMemcpy(din.p, in, in_count * sizeof(double), cudaMemcpyHostToDevice);
  if (e == cudaSuccess) e = cudaMemset(dout.p, 0, out_count * sizeof(double));
  if (e != cudaSuccess) return static_cast<int>(e);
  launch(din.p, dout.p);
  e = cudaGetLastError();
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  if (e == cudaSuccess) e = cudaMemcpy(out, dout.p, out_count * sizeof(double), cudaMemcpyDeviceToHost);
  return static_cast<int>(e);
}
int g_fn, g_n;
template <int n>
void launch_llt(const double* in, double* out) { DM_LAUNCH(k_dm_llt<n>, g_n, 32, in, out); }
}  // namespace

extern "C" {
int dm_num_fn(void) { return DM_NUM_FN; }

// rows of DM_IN doubles in, rows of DM_OUT doubles out
int dm_scalar(int fn, const double* in, double* out, int n) {
  if (fn < 0 || fn >= DM_NUM_FN || n <= 0) return -1;
  g_fn = fn;
  g_n = n;
  return dm_run(static_cast<size_t>(n) * DM_IN, static_cast<size_t>(n) * DM_OUT, in, out, [](const double* i, double* o) {
    DM_LAUNCH(k_dm_scalar, (g_n + 127) / 128, 128, g_fn, i, o, g_n);
  });
}

int dm_task(const double* in, double* out, int n) {
  if (n <= 0) return -1;
  g_n = n;
  return dm_run(static_cast<size_t>(n) * DM_TASK_IN, static_cast<size_t>(n) * DM_TASK_OUT, in, out,
                [](const double* i, double* o) { DM_LAUNCH(k_dm_task, (g_n + 15) / 16, 128, i, o, g_n); });
}

// the sizes the solvers instantiate: contact-space S (3 .. 12), UnParNMPC (14, 21), joint-space inertia (18)
int dm_llt(int dim, const double* in, double* out, int n) {
  if (n <= 0) return -1;
  g_n = n;
  void (*launch)(const double*, double*) = nullptr;
  switch (dim) {
    case 3: launch = launch_llt<3>; break;
    case 6: launch = launch_llt<6>; break;
    case 12: launch = launch_llt<12>; break;
    case 14: launch = launch_llt<14>; break;
    case 18: launch = launch_llt<18>; break;
    case 21: launch = launch_llt<21>; break;
    default: return -1;
  }
  const size_t d = static_cast<size_t>(dim);
  return dm_run(n * d * d, n * (2 * d * d + d + 1), in, out, launch);
}
}
