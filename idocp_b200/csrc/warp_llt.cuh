// warp_llt.cuh -- one WARP factorises a small dense symmetric positive definite matrix (n <= 32) and inverts it:
// right-looking Cholesky with lane = row, column-oriented substitutions with lane = right-hand side.  Shared by the
// 35 x 35 KKT inversion of UnParNMPC (unparnmpc_kernels.cuh: n = 21, 14) and by the contact-dynamics condensing of the
// floating-base path (fb_kernels.cuh: joint-space inertia n = 18, contact-space S n = 3 .. 12).  The arithmetic is the
// canonical one of the oracle: llt_lower / fb_llt (ascending chains, pivots by canon_rsqrt) and llt_solve_desc / fb_llt_solve.
#pragma once
#include "octet.cuh"

namespace idocp_b200 {

// The products and substitutions below take one operand from shared memory as a warp-wide BROADCAST (every lane reads the
// same address) and one from registers: one shared-memory wavefront per fma, which is what bounds the kernel (one wavefront
// per clock and SM against two FP64 warp instructions).  All indices are compile-time constants, so consecutive operands
// are fetched as one 16-byte load wherever the element index is even: half the wavefronts.
struct alignas(16) InvD2 {
  double x, y;
};
__device__ __forceinline__ InvD2 inv_ld2(const double* p) { return *reinterpret_cast<const InvD2*>(p); }

// y[i] (-)+= M[BASE + i] * x for i = I .. END-1 (each y[i] is a separate chain; one fma per element)
template <bool NEG, int I, int END, int BASE, int N>
__device__ __forceinline__ void inv_axpy(const double* M, double x, double (&y)[N]) {
  if constexpr (I < END) {
    if constexpr (((BASE + I) & 1) == 0 && I + 1 < END) {
      const InvD2 v = inv_ld2(M + BASE + I);
      y[I] = fma(NEG ? -v.x : v.x, x, y[I]);
      y[I + 1] = fma(NEG ? -v.y : v.y, x, y[I + 1]);
      inv_axpy<NEG, I + 2, END, BASE, N>(M, x, y);
    } else {
      const double v = M[BASE + I];
      y[I] = fma(NEG ? -v : v, x, y[I]);
      inv_axpy<NEG, I + 1, END, BASE, N>(M, x, y);
    }
  }
}

// Right-looking Cholesky of the lower triangle of the n x n matrix at A (column stride ld), in place; lane = row.
// The lane keeps its row of the trailing matrix in registers.  Step k: the pivot comes from lane k by shuffle, every
// lane scales its entry of column k (L_ik = a_ik r_k, r_k = canon_rsqrt(pivot)), publishes it (column-major in A, row-major
// in LT for the backward substitution), and applies the n - 1 - k INDEPENDENT updates a_ic -= L_ik L_ck of its row (L_ck:
// shared-memory broadcast).  Every element receives its updates in ascending k, i.e. exactly the fma chain of the
// left-looking oracle (llt_lower), but the dependent chain of the factorisation is one fma per column instead of k (the
// left-looking form of round 1 was bound by those chains).  Eigen::LLT<Lower> semantics (SURVEY A.7).  Returns non-zero
// on a bad pivot.
template <int n, int ld, int K>
__device__ __forceinline__ void warp_llt_step(double* A, double* LT, double* rd, int wl, double (&a)[n], int& fail) {
  if constexpr (K < n) {
    const double piv = __shfl_sync(FULL, a[K], K);
    if (!canon_pivot_ok(piv) && fail == 0) fail = K + 1;
    const double r = canon_rsqrt(piv);
    const double lk = a[K] * r;          // lane K: L_KK = pivot * r
    if (wl >= K && wl < n) {
      A[K * ld + wl] = lk;
      if (LT) LT[wl * ld + K] = lk;    // callers that only need the factor pass LT = nullptr
    }
    if (wl == K) rd[K] = r;
    __syncwarp();
    inv_axpy<true, K + 1, n, K * ld, n>(A, lk, a);
    warp_llt_step<n, ld, K + 1>(A, LT, rd, wl, a, fail);
  }
}
// a[c] = element (row of this lane, c) of the matrix, c <= row (the other entries are never used); returns 0 or the index
// of the first bad pivot + 1
template <int n, int ld>
__device__ __forceinline__ int warp_llt_rows(double (&a)[n], double* L, double* LT, double* rd, int wl) {
  int fail = 0;
  warp_llt_step<n, ld, 0>(L, LT, rd, wl, a, fail);
  return fail;
}
// in place on a column-major matrix (column stride ld)
template <int n, int ld>
__device__ __forceinline__ int warp_llt(double* A, double* LT, double* rd, int wl) {
  double a[n];
  const int row = wl < n ? wl : n - 1;   // idle lanes shadow the last row (never stored)
#pragma unroll
  for (int c = 0; c < n; ++c) a[c] = A[c * ld + row];   // entries c > row are never used
  __syncwarp();
  return warp_llt_rows<n, ld>(a, A, LT, rd, wl);
}

// column `c` of (L L^T)^-1: forward + backward substitution of the unit vector e_c, column-oriented: as soon as y_j is
// final it is subtracted from every later row (forward, column j of L) / every earlier row (backward, row j of L = column j
// of LT), so the rows advance together and the dependent chain is two operations per row.  Forward: row i receives its
// terms in ascending j; backward: in descending j -- the operation order of the oracle's llt_solve_desc.
// The warp barrier after every step keeps the (address-independent) shared-memory loads of L from being hoisted above the
// whole unrolled substitution (the pointers are deliberately not __restrict__: 1 KB of spills per thread in round 1).
template <int n, int ld, int J>
__device__ __forceinline__ void warp_llt_forward(const double* Lm, const double* rd, double (&y)[n]) {
  if constexpr (J < n) {
    y[J] *= rd[J];
    inv_axpy<true, J + 1, n, J * ld, n>(Lm, y[J], y);
    __syncwarp();
    warp_llt_forward<n, ld, J + 1>(Lm, rd, y);
  }
}
template <int n, int ld, int J>
__device__ __forceinline__ void warp_llt_backward(const double* LT, const double* rd, double (&y)[n]) {
  if constexpr (J >= 0) {
    y[J] *= rd[J];
    inv_axpy<true, 0, J, J * ld, n>(LT, y[J], y);
    __syncwarp();
    warp_llt_backward<n, ld, J - 1>(LT, rd, y);
  }
}
template <int n, int ld>
__device__ __forceinline__ void warp_llt_solve_unit(const double* Lm, const double* LT, const double* rd, int c, double (&y)[n]) {
#pragma unroll
  for (int i = 0; i < n; ++i) y[i] = (i == c) ? 1.0 : 0.0;
  warp_llt_forward<n, ld, 0>(Lm, rd, y);
  warp_llt_backward<n, ld, n - 1>(LT, rd, y);
}

}  // namespace idocp_b200
