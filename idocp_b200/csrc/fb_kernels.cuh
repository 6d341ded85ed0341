// fb_kernels.cuh -- batched OCPSolver Newton step for the floating-base robot (ANYmal), SURVEY.md §8 row a12.
//
// Reference path (file:line):
//   OCPSolver::updateSolution / computeKKTResidual / KKTError       src/ocp/ocp_solver.cpp:67-92,202-213
//   OCPLinearizer::runParallel, integrateSolution                   include/idocp/ocp/ocp_linearizer.hxx:113-228, src/ocp/ocp_linearizer.cpp:140-221
//   SplitOCP / ImpulseSplitOCP / TerminalOCP ::linearizeOCP         ocp/split_ocp.hxx:58-134, impulse/impulse_split_ocp.hxx:47-72, ocp/terminal_ocp.hxx:50-66
//   ContactDynamics, ImpulseDynamicsForwardEuler                    ocp/contact_dynamics.hxx:48-200, impulse/impulse_dynamics_forward_euler.hxx:25-150
//   stateequation::linearize/condenseForwardEuler (SE(3) blocks)    ocp/state_equation.hxx:11-110
//   ForwardSwitchingConstraint                                      ocp/forward_switching_constraint.hxx:27-68
//   RiccatiRecursionSolver, SplitRiccatiFactorizer (+ constrained)  src/ocp/riccati_recursion_solver.cpp:48-251, ocp/split_riccati_factorizer.hxx:36-148
//   Robot::RNEA/RNEADerivatives/computeMJtJinv/Baumgarte*           robot/robot.hxx:246-350,444-615, robot/point_contact.hxx:67-205
//
// Mapping: one CTA per (instance, stage of the hybrid chain) for the stage-parallel kernels, one CTA per instance
// for the serial Riccati sweeps.  Every working matrix of a stage lives in shared memory; every output element of a
// dense product is one ascending-index fma chain owned by one thread (fb_mm), so the result does not depend on the
// thread mapping and is bit-identical to the serial oracle.  Records in HBM are arrays of structs indexed
// [slot][instance]: a CTA reads and writes contiguous, aligned runs.
#pragma once
#include "fb_math.cuh"
#include "warp_llt.cuh"
#include "line_search_filter.cuh"
#include "pdipm.cuh"

namespace idocp_b200 {

enum { FB_GRID = 0, FB_IMPULSE = 1, FB_AUX = 2, FB_LIFT = 3, FB_TERMINAL = 4 };
enum { FBC_POS_LO = 0, FBC_POS_UP, FBC_VEL_LO, FBC_VEL_UP, FBC_TRQ_LO, FBC_TRQ_UP, FBC_FRICTION, FBC_IMPULSE_FRICTION, FBC_ACC_LO,
       FBC_ACC_UP, FBC_DISTANCE, FBC_NCOMP };
#define FB_NCON 140   /* 6 x 12 joint limits, 20 + 20 friction-cone rows (stage / impulse), 2 x 12 acceleration limits, 4 contact distances */
__host__ __device__ inline int fbc_offset(int c) {
  return c < FBC_FRICTION ? 12 * c
                          : (c == FBC_FRICTION ? 72 : (c == FBC_IMPULSE_FRICTION ? 92 : (c == FBC_DISTANCE ? 136 : 112 + 12 * (c - FBC_ACC_LO))));
}
__host__ __device__ inline int fbc_dim(int c) {   // storage
  return (c == FBC_FRICTION || c == FBC_IMPULSE_FRICTION) ? 20 : (c == FBC_DISTANCE ? 4 : 12);
}
__host__ __device__ inline int fbc_comp(int idx) {   // component of row idx
  return idx < 72 ? idx / 12
                  : (idx < 92 ? FBC_FRICTION : (idx < 112 ? FBC_IMPULSE_FRICTION : (idx < 124 ? FBC_ACC_LO : (idx < 136 ? FBC_ACC_UP : FBC_DISTANCE))));
}
__host__ __device__ inline bool fbc_is_cone(int c) { return c == FBC_FRICTION || c == FBC_IMPULSE_FRICTION; }
// rows a stage has to walk over: the acceleration-limit rows sit at the end and are skipped while those components are off
#define FBC_LIVE_ROWS(cactive) ((cactive)[FBC_DISTANCE] ? FB_NCON : (((cactive)[FBC_ACC_LO] | (cactive)[FBC_ACC_UP]) ? 136 : 112))

struct FbDevProblem {
  double T;
  int N, max_num_impulse;
  double q_weight[FB_NV], v_weight[FB_NV], a_weight[FB_NV], qf_weight[FB_NV], vf_weight[FB_NV], qi_weight[FB_NV], vi_weight[FB_NV],
      dvi_weight[FB_NV];
  double f_weight[FB_MAXF], f_ref[FB_MAXF], fi_weight[FB_MAXF], fi_ref[FB_MAXF];
  double q_min[FB_NU], q_max[FB_NU], v_max[FB_NU], u_max[FB_NU];
  double mu, barrier, fraction_rate;
  int enable[FBC_NCOMP];
  int cone_nonlinear[2];   // FrictionCone / ImpulseFrictionCone (2 rows per contact) instead of the linearised cones (5 rows)
  double a_min[FB_NU], a_max[FB_NU];   // JointAcceleration{Lower,Upper}Limit
  int distance_mode;       // ContactDistance: 1 = row 2 of the LOCAL frame Jacobian (the reference, literally), 2 = d z / d q
};
// rows per contact of cone component c, live rows of a component (the rest of its storage stays zero)
// (nl = fbc_cone_bits(pr), read ONCE per kernel: the problem record lives in global memory and these kernels are latency bound)
__host__ __device__ inline int fbc_cone_bits(const FbDevProblem& pr) { return (pr.cone_nonlinear[0] ? 1 : 0) | (pr.cone_nonlinear[1] ? 2 : 0); }
__host__ __device__ inline int fbc_cone_rows(int nl, int c) { return ((nl >> (c - FBC_FRICTION)) & 1) ? 2 : 5; }
__host__ __device__ inline int fbc_rows(int nl, int c) { return fbc_is_cone(c) ? FB_NC * fbc_cone_rows(nl, c) : (c == FBC_DISTANCE ? FB_NC : 12); }
// contact of row j of cone component c, and the row within that contact's cone (no division by a run-time value).  The row is
// formed from the contact rather than as j % 5: k_fb_expand would otherwise keep it live across its active-contact count and spill.
__host__ __device__ inline void fbc_cone_row(int nl, int c, int j, int& contact, int& row) {
  const int rpc = fbc_cone_rows(nl, c);
  contact = rpc == 2 ? (j >> 1) : (j / 5);
  row = j - rpc * contact;
}

// margin of row j of box component c (joint position / velocity / torque / acceleration limit): >= 0 is feasible; the residual
// of the row is slack - margin
__device__ __forceinline__ double fbc_box_margin(int c, int j, const FbDevProblem& pr, const double* q, const double* v, const double* a,
                                                 const double* u) {
  switch (c) {
    case FBC_ACC_LO: return a[6 + j] - pr.a_min[j];
    case FBC_ACC_UP: return pr.a_max[j] - a[6 + j];
    case FBC_POS_LO: return q[7 + j] - pr.q_min[j];
    case FBC_POS_UP: return pr.q_max[j] - q[7 + j];
    case FBC_VEL_LO: return v[6 + j] - (-pr.v_max[j]);
    case FBC_VEL_UP: return pr.v_max[j] - v[6 + j];
    case FBC_TRQ_LO: return u[j] - (-pr.u_max[j]);
    default:         return pr.u_max[j] - u[j];
  }
}

// one element of the hybrid chain (shared by the whole batch)
struct FbElem {
  int kind, slot, next_slot, prev_slot, sw, dimf, dimi, pad;
  int active[FB_NC], imp_active[FB_NC], cactive[FBC_NCOMP];
  int ls_next_slot, ls_sw, ls_imp_active[FB_NC], pad2[2];   // LineSearch::computeCostAndViolation (line_search.cpp:64-197)
  double t, dt, dt_next, ls_dt_next, ls_ipoints[FB_MAXF];
  double cpoints[FB_MAXF], ipoints[FB_MAXF], ref_q[FB_NQ], ref_v[FB_NV];
};

// ---- HBM records, [slot][instance] ----
struct FbSol {   // SplitSolution / ImpulseSplitSolution (a = dv at an impulse) + slack / dual of ConstraintsData
  double lmd[FB_NV], gmm[FB_NV], q[FB_NQ], v[FB_NV], a[FB_NV], u[FB_NU], beta[FB_NV], nu_passive[FB_NPASS], f[FB_MAXF], mu[FB_MAXF],
      xi[FB_MAXF];
  double slack[FB_NCON], dual[FB_NCON];
};
struct FbDir {   // SplitDirection + the direction part of ConstraintsData
  double dlmd[FB_NV], dgmm[FB_NV], dq[FB_NV], dv[FB_NV], du[FB_NU], daf[FB_NVF], dbetamu[FB_NVF], dnu_passive[FB_NPASS], dxi[FB_MAXF];
  double residual[FB_NCON], duality[FB_NCON], dslack[FB_NCON], ddual[FB_NCON];
  double max_primal, max_dual, kkt_sq, info;
  double ls_cost, ls_viol;   // LineSearch: stage cost / constraint violation of the trial point
};
struct FbKKT {   // condensed SplitKKTMatrix / SplitKKTResidual + SplitStateConstraintJacobian
  double Qxx[FB_NX * FB_NX], Qxu[FB_NX * FB_NV], Quu[FB_NV * FB_NV];
  double Fqq6[36], Fqv6[36], Fqq_prev_inv[36], Fvq[FB_NV * FB_NV], Fvv[FB_NV * FB_NV], Fvu[FB_NV * FB_NU];
  double lq[FB_NV], lv[FB_NV], lu[FB_NU], lu_passive[FB_NPASS], Fq[FB_NV], Fv[FB_NV];
  double Phix[FB_MAXF * FB_NX], Phiu[FB_MAXF * FB_NU], P[FB_MAXF];
};
struct FbExp {   // ContactDynamicsData needed by the expansion
  double MJtJinv[FB_NVF * FB_NVF], MJ_dIDC[FB_NVF * FB_NX], MJ_IDC[FB_NVF], Qafqv[FB_NVF * FB_NX], Qafu[FB_NVF * FB_NV], laf[FB_NVF];
};
struct FbRic {   // LQRStateFeedbackPolicy, SplitRiccatiFactorization, SplitConstrainedRiccatiFactorization
  double K[FB_NU * FB_NX], k[FB_NU], Pqq[FB_NV * FB_NV], Pqv[FB_NV * FB_NV], Pvv[FB_NV * FB_NV], sq[FB_NV], sv[FB_NV], cM[FB_MAXF * FB_NX],
      cm[FB_MAXF];
};

struct FbArrays {
  int B, n_slots, n_elems;
  const FbDevProblem* prob;
  const FbElem* elems;
  FbSol* sol;
  FbDir* dir;
  FbKKT* kkt;
  FbExp* exp;
  FbRic* ric;
  struct FbLin* lin;   // K1a -> K1b hand-over records
  const double* q0;   // [B][19]
  const double* v0;   // [B][18]
  double* steps;      // [B][2]
  double* kkt_err;    // [B]
  LsFilter ls;        // filter line search of B instances (line_search_filter.cuh)
  int* ls_status;     // [B] IDOCP_B200_STATUS_FILTER_FULL
  const double* iref; // [slot][B][FB_IREF] per-instance (q_ref, v_ref) (the IREF instantiations); nullptr in shared mode
};
constexpr int FB_IREF = FB_NQ + FB_NV;
// the cost reference (q_ref, then v_ref) of record `rec` = (slot, instance): per instance (IREF) or shared by the batch
template <bool IREF>
__device__ __forceinline__ const double* fb_ref_q(const FbArrays& A, const FbElem& el, size_t rec) {
  return IREF ? A.iref + rec * FB_IREF : el.ref_q;
}
template <bool IREF>
__device__ __forceinline__ const double* fb_ref_v(const FbArrays& A, const FbElem& el, size_t rec) {
  return IREF ? A.iref + rec * FB_IREF + FB_NQ : el.ref_v;
}

#define FB_FOR(i, n) for (int i = threadIdx.x; i < (n); i += blockDim.x)
enum { FBM_SET = 0, FBM_ADD = 1, FBM_SUB = 2 };

// C (m x n) {=, +=, -=} A (m x k) B (k x n): one ascending-k fma chain per element.  A thread owns a 2 x 2 tile of C
// (3 x 3 and 4 x 4 tiles save shared-memory loads but measured 25-30 % slower: too few threads per product)
// -- rows (i, i + ceil(m/2)), columns (j, j + ceil(n/2)), so that neighbouring lanes read neighbouring columns of B
// (no shared-memory bank conflicts) and write neighbouring elements of C: four independent chains in flight (the
// chains are latency-bound otherwise) and half the shared-memory loads per fma.  The chain of every element is
// unchanged, so the bits do not depend on the tiling.  FBM_SET starts a chain with the plain product a_0 b_0;
// FBM_ADD / FBM_SUB start it from init(i, j); store(i, j, value) receives the finished element.
// The caller separates dependent calls with __syncthreads().
template <int MODE, class Init, class Store>
__device__ __forceinline__ void fb_mm_simt_f(int m, int n, int k, const double* __restrict__ A, int ars, int acs, const double* __restrict__ B,
                                        int brs, int bcs, Init init, Store store) {
  const int tm = (m + 1) >> 1, tn = (n + 1) >> 1, total = tm * tn;
  for (int t = threadIdx.x; t < total; t += blockDim.x) {
    const int i0 = t / tn, j0 = t - i0 * tn;
    const int i1 = i0 + tm, j1 = j0 + tn;
    const bool hi = i1 < m, hj = j1 < n;
    const double* a0 = A + i0 * ars;
    const double* a1 = A + (hi ? i1 : i0) * ars;
    const double* b0 = B + j0 * bcs;
    const double* b1 = B + (hj ? j1 : j0) * bcs;
    double c00, c01, c10, c11;
    int l0 = 0;
    if (MODE == FBM_SET) {
      if (k == 0) {
        c00 = c01 = c10 = c11 = 0.0;
      } else {
        const double x0 = a0[0], x1 = a1[0], y0 = b0[0], y1 = b1[0];
        c00 = x0 * y0; c01 = x0 * y1; c10 = x1 * y0; c11 = x1 * y1;
        l0 = 1;
      }
    } else {
      c00 = init(i0, j0);
      c01 = hj ? init(i0, j1) : 0.0;
      c10 = hi ? init(i1, j0) : 0.0;
      c11 = (hi && hj) ? init(i1, j1) : 0.0;
    }
    for (int l = l0; l < k; ++l) {
      double x0 = a0[l * acs], x1 = a1[l * acs];
      const double y0 = b0[l * brs], y1 = b1[l * brs];
      if (MODE == FBM_SUB) { x0 = -x0; x1 = -x1; }
      c00 = fma(x0, y0, c00); c01 = fma(x0, y1, c01); c10 = fma(x1, y0, c10); c11 = fma(x1, y1, c11);
    }
    store(i0, j0, c00);
    if (hj) store(i0, j1, c01);
    if (hi) { store(i1, j0, c10); if (hj) store(i1, j1, c11); }
  }
}
// ---------------------------------------------------------------------------------------------------------------------
// The same products on the FP64 tensor cores.  mma.sync.aligned.m8n8k4.f64 computes, for every element of an 8 x 8 tile,
// d = fma(a_3, b_3, fma(a_2, b_2, fma(a_1, b_1, fma(a_0, b_0, c)))) -- measured on the B200: bit-identical to the ascending
// fma chain on 262 144 random elements with widely spread exponents, 120 529 of which tell ascending / descending / fused
// summation apart (tools/dmma_probe.cu, profiles/dmma_probe.json).  Chaining the accumulator over k in steps of 4 therefore
// IS the canonical chain of the oracle, and zero-padding the ragged edges adds fma(0, 0, c) = c.  What it buys: the SIMT
// form reads one shared-memory operand per fma and warp (the LSU was ~65 % busy, FP64 pipe 14-16 %); one DMMA does 256 fma
// from two operand loads, i.e. 5 x fewer shared-memory wavefronts and 8 x fewer FP64 instructions for the same chain.
// A warp owns an 8 x 16 strip of C (two tiles sharing the A fragment: two independent accumulator chains).
// Fragment layout (PTX ISA, m8n8k4 .f64): a = A[g][t], b = B[t][g], c / d = C[g][2 t + {0, 1}] with g = lane / 4, t = lane % 4.
// `rot` (optional): independent products issued back to back without a barrier start their strip -> warp assignment where
// the previous one stopped (*rot is advanced by the strip count), so that the warps share out the strips of all of them.
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void fb_dmma(double& d0, double& d1, double a, double b) {
#ifndef IDOCP_B200_EMU
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
#else
  emu_dmma_m8n8k4(d0, d1, a, b);   // the ascending chain the hardware was measured to execute (tests/emu/cuda_emu.h)
#endif
}
template <int MODE, class Init, class Store>
__device__ __forceinline__ void fb_mm_f(int m, int n, int k, const double* __restrict__ A, int ars, int acs, const double* __restrict__ B,
                                        int brs, int bcs, Init init, Store store, int* rot = nullptr) {
  const int nw = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const int tm = (m + 7) >> 3, tn = (n + 15) >> 4, total = tm * tn;
  int first = warp;
  if (rot) {
    first = warp - *rot;
    if (first < 0) first += nw;
    *rot = (*rot + total) % nw;
  }
  for (int s = first; s < total; s += nw) {          // warp-uniform: every lane executes every mma.sync
    const int i0 = (s / tn) << 3, j0 = (s - (s / tn) * tn) << 4;
    const int row = i0 + g, ca = j0 + 2 * t, cb = ca + 8, ba = j0 + g, bb = ba + 8;
    const bool rok = row < m, baok = ba < n, bbok = bb < n;
    // FBM_SET: a chain that starts with the plain product a_0 b_0 = fma(a_0, b_0, -0.0), sign of zero included
    double c00 = (k > 0) ? -0.0 : 0.0, c01 = c00, c10 = c00, c11 = c00;
    if (MODE != FBM_SET) {
      c00 = (rok && ca < n) ? init(row, ca) : 0.0;
      c01 = (rok && ca + 1 < n) ? init(row, ca + 1) : 0.0;
      c10 = (rok && cb < n) ? init(row, cb) : 0.0;
      c11 = (rok && cb + 1 < n) ? init(row, cb + 1) : 0.0;
    }
    const double* ap = A + (rok ? row : 0) * ars + t * acs;
    const double* bpa = B + (baok ? ba : 0) * bcs + t * brs;
    const double* bpb = B + (bbok ? bb : 0) * bcs + t * brs;
    for (int l = 0; l < k; l += 4) {
      const bool kin = l + t < k;
      double a = (rok && kin) ? ap[l * acs] : 0.0;
      const double b0 = (baok && kin) ? bpa[l * brs] : 0.0, b1 = (bbok && kin) ? bpb[l * brs] : 0.0;
      if (MODE == FBM_SUB) a = -a;
      fb_dmma(c00, c01, a, b0);
      fb_dmma(c10, c11, a, b1);
    }
    if (rok) {
      if (ca < n) store(row, ca, c00);
      if (ca + 1 < n) store(row, ca + 1, c01);
      if (cb < n) store(row, cb, c10);
      if (cb + 1 < n) store(row, cb + 1, c11);
    }
  }
}
template <int MODE>
__device__ __forceinline__ void fb_mm(int m, int n, int k, const double* __restrict__ A, int ars, int acs, const double* __restrict__ B,
                                      int brs, int bcs, double* C, int ldc, int* rot = nullptr) {
  fb_mm_f<MODE>(m, n, k, A, ars, acs, B, brs, bcs, [=](int i, int j) { return C[i * ldc + j]; },
                [=](int i, int j, double v) { C[i * ldc + j] = v; }, rot);
}
// matrix-vector products stay on the SIMT path (one column would waste 7 / 8 of a tensor-core tile)
template <int MODE>
__device__ __forceinline__ void fb_mv(int m, int k, const double* A, int ars, int acs, const double* x, double* y) {
  fb_mm_simt_f<MODE>(m, 1, k, A, ars, acs, x, 1, 1, [=](int i, int j) { return y[i + j]; }, [=](int i, int j, double v) { y[i + j] = v; });
}
__device__ inline double fb_sqnorm(const double* x, int n) {
  double acc = 0.0;
  for (int i = 0; i < n; ++i) acc = fma(x[i], x[i], acc);
  return acc;
}
__device__ inline void fb_copy(double* dst, const double* src, int n) { FB_FOR(i, n) dst[i] = src[i]; }
// HBM record -> shared memory by a 128-thread CTA: ALL of a thread's loads are issued before its first store.  (A plain copy
// loop through generic pointers keeps load -> store -> load order, i.e. one DRAM round trip per element and thread.)
// index(x) maps the destination element to the source element.
template <int N, class Index>
__device__ __forceinline__ void fb_load_f(double* dst, const double* __restrict__ src, Index index) {
  constexpr int R = (N + 127) / 128;
  double r[R];
#pragma unroll
  for (int i = 0; i < R; ++i) {
    const int x = threadIdx.x + i * 128;
    r[i] = x < N ? __ldg(src + index(x)) : 0.0;
  }
#pragma unroll
  for (int i = 0; i < R; ++i) {
    const int x = threadIdx.x + i * 128;
    if (x < N) dst[x] = r[i];
  }
}
template <int N>
__device__ __forceinline__ void fb_load(double* dst, const double* __restrict__ src) {
  fb_load_f<N>(dst, src, [](int x) { return x; });
}
// ask the L2 for the `bytes` starting at p (one 128-byte line per thread and round); no effect on results
__device__ __forceinline__ void fb_prefetch_l2(const void* p, int bytes) {
#ifndef IDOCP_B200_EMU
  const char* c = static_cast<const char*>(p);
  for (int o = threadIdx.x * 128; o < bytes; o += blockDim.x * 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(c + o));
#endif
}
__device__ inline void fb_zero(double* dst, int n) { FB_FOR(i, n) dst[i] = 0.0; }

// Cholesky of an n x n matrix by the WHOLE CTA (128 threads), right-looking, n (n + 1) / 2 <= 128 E.  Every element of the
// lower triangle is owned by one thread and lives in a register for the whole factorisation.  Column k: the owner of
// (k, k) takes the square root and the reciprocal while the owners of (i, k) publish their finished entries; after ONE
// barrier every owner of a trailing element reads the two entries and the reciprocal, forms the two multipliers and
// applies its fma -- no dependent chain, no load -> store ordering, and a rolled loop (the fully unrolled register /
// shuffle form of this ran out of instruction cache).  Every element receives its updates in ascending k and
// L_ik = A_ik * (1 / L_kk), so the bits equal the serial left-looking form of the oracle.  A is only read.
// L[j*ldl + i] = L_ij (i >= j), rd[k] = 1 / L_kk; *info = code + first failing pivot + 1 unless *info is set already.
template <int E>
__device__ __forceinline__ void fb_llt_cta(const double* A, int lda, int n, double* L, int ldl, double* rd, int* info, int code) {
  const int total = n * (n + 1) / 2;
  int ei[E], ej[E];
  double a[E];
#pragma unroll
  for (int e = 0; e < E; ++e) {
    const int x = threadIdx.x + e * 128;
    ei[e] = -1; ej[e] = -1; a[e] = 0.0;
    if (x < total) {
      int i = 0;
      while ((i + 1) * (i + 2) / 2 <= x) ++i;
      ei[e] = i; ej[e] = x - i * (i + 1) / 2;
      a[e] = A[i * lda + ej[e]];
    }
  }
  for (int k = 0; k < n; ++k) {
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if (ej[e] == k) {
        if (ei[e] == k) {
          const double r = canon_rsqrt(a[e]);
          if (!canon_pivot_ok(a[e]) && *info == 0) *info = code + k + 1;
          rd[k] = r;
          L[k * ldl + k] = a[e] * r;
        } else {
          L[k * ldl + ei[e]] = a[e];   // still unscaled
        }
      }
    }
    __syncthreads();
    const double r = rd[k];
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if (ej[e] > k) {
        const double lik = L[k * ldl + ei[e]] * r, ljk = L[k * ldl + ej[e]] * r;
        a[e] = fma(-lik, ljk, a[e]);
      }
    }
  }
  __syncthreads();
#pragma unroll
  for (int e = 0; e < E; ++e)
    if (ej[e] >= 0 && ei[e] > ej[e]) L[ej[e] * ldl + ei[e]] *= rd[ej[e]];
  __syncthreads();
}
// ---- M^-1 of the joint-space inertia with the tree structure of the robot ----
// M couples a leg joint only with the joints of its own leg and with the base, so eliminating the legs FIRST keeps the factor
// sparse (pinocchio's cholesky::decompose does the same from the leaves to the root).  Elimination order (oracle/fb_robot.h
// FB_MPERM): position 4 s + i = joint s of leg i, positions 12..17 = base.  The four pivots 4 s .. 4 s + 3 belong to different
// legs and are independent: they share ONE barrier step, so the factorisation + forward substitution take 3 + 6 steps and the
// backward substitution 6 + 3 instead of 18 + 18.  Every element still receives its non-zero updates in ascending (backward:
// descending) pivot order; the skipped updates have an exactly zero factor, so the bits equal the oracle's dense Cholesky of
// the permuted matrix.  Minv (n x n, original order) holds the identity on entry... it is rebuilt here; L, rd: scratch.
__device__ __forceinline__ int fbm_perm(int p) { return p < 12 ? 6 + 3 * (p & 3) + (p >> 2) : p - 12; }
__device__ __forceinline__ bool fbm_nz(int r, int k) { return k >= 12 || r >= 12 || ((r & 3) == (k & 3)); }   // L[r][k], r >= k
__device__ __forceinline__ void fb_minv_tree_cta(const double* M, double* L, double* rd, double* X, int* fail, int* info, int code) {
  constexpr int n = FB_NV, EY = 3;
  const int t = threadIdx.x;
  // the 117 structurally non-zero entries of the lower triangle, one per thread: base x legs, base x base, leg blocks
  int ai = -1, aj = -1;
  if (t < 72) { ai = 12 + t / 12; aj = t % 12; }
  else if (t < 93) { int u = t - 72, i = 0; while ((i + 1) * (i + 2) / 2 <= u) ++i; ai = 12 + i; aj = 12 + u - i * (i + 1) / 2; }
  else if (t < 117) { const int u = t - 93, leg = u / 6, v = u % 6; const int sr = v < 1 ? 0 : (v < 3 ? 1 : 2), sc = v - sr * (sr + 1) / 2; ai = 4 * sr + leg; aj = 4 * sc + leg; }
  double a = ai >= 0 ? M[fbm_perm(ai) * n + fbm_perm(aj)] : 0.0;
  int yi[EY], yc[EY];
  double y[EY];
#pragma unroll
  for (int e = 0; e < EY; ++e) {
    const int x = t + e * 128;
    yi[e] = -1; yc[e] = 0; y[e] = 0.0;
    if (x < n * n) { yi[e] = x / n; yc[e] = x - yi[e] * n; y[e] = yi[e] == yc[e] ? 1.0 : 0.0; }
  }
  if (t < n) fail[t] = 0;
  __syncthreads();
  for (int g = 0; g < 9; ++g) {
    const int k0 = g < 3 ? 4 * g : 9 + g, nk = g < 3 ? 4 : 1;
    if (aj >= k0 && aj < k0 + nk) {
      if (ai == aj) {
        const double r = canon_rsqrt(a);
        if (!canon_pivot_ok(a)) fail[aj] = 1;
        rd[aj] = r;
        L[aj * n + aj] = a * r;
      } else {
        L[aj * n + ai] = a;   // still unscaled
      }
    }
#pragma unroll
    for (int e = 0; e < EY; ++e)
      if (yi[e] >= k0 && yi[e] < k0 + nk) X[yi[e] * n + yc[e]] = y[e];   // still unscaled
    __syncthreads();
    for (int k = k0; k < k0 + nk; ++k) {
      const double r = rd[k];
      if (aj >= k0 + nk && fbm_nz(ai, k) && fbm_nz(aj, k)) {
        const double lik = L[k * n + ai] * r, ljk = L[k * n + aj] * r;
        a = fma(-lik, ljk, a);
      }
#pragma unroll
      for (int e = 0; e < EY; ++e) {
        if (yi[e] == k) y[e] *= r;
        else if (yi[e] >= k0 + nk && fbm_nz(yi[e], k)) y[e] = fma(-(L[k * n + yi[e]] * r), X[k * n + yc[e]] * r, y[e]);
      }
    }
  }
  __syncthreads();
  if (ai > aj) L[aj * n + ai] *= rd[aj];
  if (t == 0) {
    for (int k = 0; k < n; ++k)
      if (fail[k] && *info == 0) *info = code + k + 1;
  }
  __syncthreads();
  for (int g = 8; g >= 0; --g) {
    const int k0 = g < 3 ? 4 * g : 9 + g, nk = g < 3 ? 4 : 1;
#pragma unroll
    for (int e = 0; e < EY; ++e)
      if (yi[e] >= k0 && yi[e] < k0 + nk) { y[e] *= rd[yi[e]]; X[yi[e] * n + yc[e]] = y[e]; }
    __syncthreads();
    for (int j = k0 + nk - 1; j >= k0; --j) {
#pragma unroll
      for (int e = 0; e < EY; ++e)
        if (yi[e] >= 0 && yi[e] < k0 && fbm_nz(j, yi[e])) y[e] = fma(-L[yi[e] * n + j], X[j * n + yc[e]], y[e]);
    }
  }
  __syncthreads();
  // back to the original order: every entry sits in a register of its owner
#pragma unroll
  for (int e = 0; e < EY; ++e)
    if (yi[e] >= 0) X[fbm_perm(yi[e]) * n + fbm_perm(yc[e])] = y[e];
  __syncthreads();
}

// fb_llt_cta and X := (L L^T)^-1 X for an n x m block of right-hand sides (X[i*ldx + c], n m <= 128 EY, every entry owned
// by one thread in a register) in ONE sweep: column k of the factor and step k of the forward substitution need the same
// barrier (the forward step uses L_ik = A_ik r_k and the scaled y_k = y_k r_k, both formed from values published before
// it), so the factorisation plus both substitutions cost 2 n barriers instead of 3 n.  Same arithmetic, element by element.
template <int EA, int EY>
__device__ __forceinline__ void fb_llt_factor_solve_cta(const double* A, int lda, int n, double* L, int ldl, double* rd, double* X, int ldx,
                                                        int m, int* info, int code) {
  const int na = n * (n + 1) / 2, ny = n * m;
  int ai[EA], aj[EA], yi[EY], yc[EY];
  double a[EA], y[EY];
#pragma unroll
  for (int e = 0; e < EA; ++e) {
    const int x = threadIdx.x + e * 128;
    ai[e] = -1; aj[e] = -1; a[e] = 0.0;
    if (x < na) {
      int i = 0;
      while ((i + 1) * (i + 2) / 2 <= x) ++i;
      ai[e] = i; aj[e] = x - i * (i + 1) / 2;
      a[e] = A[i * lda + aj[e]];
    }
  }
#pragma unroll
  for (int e = 0; e < EY; ++e) {
    const int x = threadIdx.x + e * 128;
    yi[e] = -1; yc[e] = 0; y[e] = 0.0;
    if (x < ny) { yi[e] = x / m; yc[e] = x - yi[e] * m; y[e] = X[yi[e] * ldx + yc[e]]; }
  }
  for (int k = 0; k < n; ++k) {
#pragma unroll
    for (int e = 0; e < EA; ++e) {
      if (aj[e] == k) {
        if (ai[e] == k) {
          const double r = canon_rsqrt(a[e]);
          if (!canon_pivot_ok(a[e]) && *info == 0) *info = code + k + 1;
          rd[k] = r;
          L[k * ldl + k] = a[e] * r;
        } else {
          L[k * ldl + ai[e]] = a[e];   // still unscaled
        }
      }
    }
#pragma unroll
    for (int e = 0; e < EY; ++e)
      if (yi[e] == k) X[k * ldx + yc[e]] = y[e];   // still unscaled
    __syncthreads();
    const double r = rd[k];
#pragma unroll
    for (int e = 0; e < EA; ++e) {
      if (aj[e] > k) {
        const double lik = L[k * ldl + ai[e]] * r, ljk = L[k * ldl + aj[e]] * r;
        a[e] = fma(-lik, ljk, a[e]);
      }
    }
#pragma unroll
    for (int e = 0; e < EY; ++e) {
      if (yi[e] == k) y[e] *= r;
      else if (yi[e] > k) y[e] = fma(-(L[k * ldl + yi[e]] * r), X[k * ldx + yc[e]] * r, y[e]);
    }
  }
  __syncthreads();
#pragma unroll
  for (int e = 0; e < EA; ++e)
    if (aj[e] >= 0 && ai[e] > aj[e]) L[aj[e] * ldl + ai[e]] *= rd[aj[e]];
  __syncthreads();
  for (int j = n - 1; j >= 0; --j) {
#pragma unroll
    for (int e = 0; e < EY; ++e)
      if (yi[e] == j) { y[e] *= rd[j]; X[j * ldx + yc[e]] = y[e]; }
    __syncthreads();
#pragma unroll
    for (int e = 0; e < EY; ++e)
      if (yi[e] >= 0 && yi[e] < j) y[e] = fma(-L[yi[e] * ldl + j], X[j * ldx + yc[e]], y[e]);
  }
  __syncthreads();
}
// x := (L L^T)^-1 x for one right-hand side (stride incx) by the calling thread, in place and column-oriented: as soon
// as x_j is known every remaining entry is updated by an independent fma (no dependent chain across i).
// Forward: entry i receives its terms in ascending j; backward: in descending j (the oracle's order).
template <int N>
__device__ __forceinline__ void fb_llt_solve_n(const double* __restrict__ L, int ldl, const double* __restrict__ rd, double* x, int incx,
                                               int n = N) {
  // volatile: the loads stay in program order; hoisting all N (N - 1) / 2 of them ahead of the chain spills
  const volatile double* Lv = L;
  double y[N];
#pragma unroll
  for (int i = 0; i < N; ++i) y[i] = i < n ? x[i * incx] : 0.0;
#pragma unroll
  for (int j = 0; j < N; ++j) {
    if (j < n) {
      y[j] *= rd[j];
#pragma unroll
      for (int i = j + 1; i < N; ++i)
        if (i < n) y[i] = fma(-Lv[j * ldl + i], y[j], y[i]);
    }
  }
#pragma unroll
  for (int j = N - 1; j >= 0; --j) {
    if (j < n) {
      y[j] *= rd[j];
#pragma unroll
      for (int i = 0; i < j; ++i) y[i] = fma(-Lv[i * ldl + j], y[j], y[i]);
    }
  }
#pragma unroll
  for (int i = 0; i < N; ++i)
    if (i < n) x[i * incx] = y[i];
}
// same arithmetic for a run-time n (row-oriented, in place)
__device__ __noinline__ void fb_llt_solve(const double* L, int ldl, const double* rd, int n, double* x, int incx) {
  for (int i = 0; i < n; ++i) {
    double y = x[i * incx];
    for (int j = 0; j < i; ++j) y = fma(-L[j * ldl + i], x[j * incx], y);
    x[i * incx] = y * rd[i];
  }
  for (int i = n - 1; i >= 0; --i) {
    double y = x[i * incx];
    for (int j = n - 1; j > i; --j) y = fma(-L[i * ldl + j], x[j * incx], y);
    x[i * incx] = y * rd[i];
  }
}

// ---- friction cone (constraints/linearized_friction_cone.hpp:72-85, .cpp:25-29); nonlinear: normalForceResidual and
// frictionConeResidual of FrictionCone / ImpulseFrictionCone (friction_cone.hpp:72-82), Jacobian rows d(-fz)/df and
// data.r[i] = (2 fx, 2 fy, -2 mu^2 fz) (friction_cone.cpp:109-111) ----
__device__ inline void fb_friction_residual(double mu, bool nonlinear, const double* f, double* r) {
  if (nonlinear) {
    r[0] = -f[2];
    r[1] = fma(-((mu * mu) * f[2]), f[2], fma(f[1], f[1], f[0] * f[0]));
    r[2] = r[3] = r[4] = 0.0;
    return;
  }
  const double s = mu * f[2] / 1.41421356237309514547e+00;
  r[0] = -f[2];
  r[1] = f[0] - s;
  r[2] = -f[0] - s;
  r[3] = f[1] - s;
  r[4] = -f[1] - s;
}
__device__ inline double fb_friction_jac(double mu, bool nonlinear, const double* f, int e, int x) {
  if (nonlinear) {
    if (e == 0) return x == 2 ? -1.0 : 0.0;
    return x == 2 ? -(((2.0 * mu) * mu) * f[2]) : 2.0 * f[x];
  }
  const double m = -(mu / 1.41421356237309514547e+00);
  if (x == 2) return e == 0 ? -1.0 : m;
  if (x == 0) return e == 1 ? 1.0 : (e == 2 ? -1.0 : 0.0);
  return e == 3 ? 1.0 : (e == 4 ? -1.0 : 0.0);
}

// compile-time cone type for the hot kernel (the type is uniform over the launch: one branch, then constant-folded rows)
template <bool NL>
__device__ __forceinline__ double fb_friction_jac_t(double mu, const double* f, int e, int x) {
  return fb_friction_jac(mu, NL, f, e, x);
}
// augmentDualResidual of a cone: dt * sum_e J[e][cx] dual[e]
template <bool NL>
__device__ __forceinline__ double fb_cone_augment(double mu, const double* fi, const double* du5, int cx) {
  constexpr int RPC = NL ? 2 : 5;
  double acc = fb_friction_jac_t<NL>(mu, fi, 0, cx) * du5[0];
#pragma unroll
  for (int ee = 1; ee < RPC; ++ee) acc = fma(fb_friction_jac_t<NL>(mu, fi, ee, cx), du5[ee], acc);
  return acc;
}
// condenseSlackAndDual of a cone: gradient term of column cx and the row cx of the 3 x 3 Hessian block J^T diag(dual / slack) J
template <bool NL>
__device__ __forceinline__ double fb_cone_condense(double mu, const double* fi, const double* slack, const double* dual,
                                                   const double* residual, const double* duality, int cx, double* h3) {
  constexpr int RPC = NL ? 2 : 5;
  double r5[RPC], w5[RPC];
#pragma unroll
  for (int ee = 0; ee < RPC; ++ee) {
    const double rs = 1.0 / slack[ee];
    r5[ee] = fma(dual[ee], residual[ee], -duality[ee]) * rs;
    w5[ee] = dual[ee] * rs;
  }
  double acc = fb_friction_jac_t<NL>(mu, fi, 0, cx) * r5[0];
#pragma unroll
  for (int ee = 1; ee < RPC; ++ee) acc = fma(fb_friction_jac_t<NL>(mu, fi, ee, cx), r5[ee], acc);
#pragma unroll
  for (int y = 0; y < 3; ++y) {
    double h = fb_friction_jac_t<NL>(mu, fi, 0, cx) * (w5[0] * fb_friction_jac_t<NL>(mu, fi, 0, y));
#pragma unroll
    for (int ee = 1; ee < RPC; ++ee) h = fma(fb_friction_jac_t<NL>(mu, fi, ee, cx), w5[ee] * fb_friction_jac_t<NL>(mu, fi, ee, y), h);
    h3[y] = h;
  }
  return acc;
}

// =====================================================================================================
// K1a: rigid-body + stage-local linearisation, ONE WARP per (instance, stage)
//   forward kinematics, RNEA and its derivatives with contact wrenches, Baumgarte / impulse-velocity rows, cost
//   gradient + sparse Hessian, PDIPM residuals and condensing, SE(3) state-equation blocks, switching constraint.
//   Everything here is O(n) .. O(n^2) with at most 18-way parallelism: a warp per stage keeps 8+ stages in flight
//   per SM without block barriers.  The dense O(n^3) condensing is K1b.
// =====================================================================================================
#define FBW_FOR(i, n) for (int i = lane; i < (n); i += 32)

// per-stage record handed from K1a to K1b (HBM, [slot][instance])
struct FbLin {
  double IDC[FB_NVF], dIDCdqv[FB_NVF * FB_NX], Mm[FB_NV * FB_NV], dCda[FB_MAXF * FB_NV];
  double lq[FB_NV], lv[FB_NV], la[FB_NV], lf[FB_MAXF], lu_passive[FB_NPASS], lu[FB_NU], Fq[FB_NV], Fv[FB_NV], P[FB_MAXF];
  double Qqq6[36], Qqq_d[FB_NV], Qvv_d[FB_NV], Quu_d[FB_NU], Qaa[FB_NV], Qff[FB_MAXF * FB_MAXF];
  double Fqq6[36], Fqv6[36], Fqq_prev_inv[36];
  double Phix[FB_MAXF * FB_NX], Phia[FB_MAXF * FB_NV];
  double cdJ[FB_NC * FB_NV], cdw[FB_NC];   // ContactDistance: J2 rows and dt dual / slack (written and read only while it is active)
};

struct FbRobotWork {
  // inputs (same order as FbSol)
  double lmd[FB_NV], gmm[FB_NV], q[FB_NQ], v[FB_NV], a[FB_NV], u[FB_NU], beta[FB_NV], nu_passive[FB_NPASS], f[FB_MAXF], mu[FB_MAXF],
      xi[FB_MAXF];
  // slack / dual of the constraint rows are read where they lie (FbSol, read-only here) and residual / duality live in FbDir only:
  // 4.5 KB less per warp, i.e. 12 instead of 10 warps per SM
  double nlmd[FB_NV], ngmm[FB_NV], nq[FB_NQ], nv[FB_NV], qprev[FB_NQ];
  double fm[FB_MAXF], mu_stack[FB_MAXF];
  // kinematics (world frame)
  double R[FB_NB][9], p[FB_NB][3], S[FB_NV][6], ov[FB_NB][6], oa[FB_NB][6], dV[FB_NV][6];
  // dynamics
  fb_inertia_t Y[FB_NB];
  fb_dinertia_t D[FB_NB];
  double F[FB_NB][6], agf[FB_NB][6];
  union {   // the RNEA derivative columns are dead before the switching constraint starts
    struct { double U[FB_NV][6], W[FB_NV][6], dFv[FB_NV][6], dFq[FB_NV][6], dFqa[FB_NV][6], dAq[FB_NV][6], dAv[FB_NV][6]; };
    struct { double dqv[FB_NV], q2[FB_NQ], Jq6[36], Jv6[36], Pq[FB_MAXF * FB_NV], PJv[FB_MAXF * FB_NV]; };
  };
  double frP[3], frV[6], frA[6];
  // SE(3) blocks: three relative placements (cost reference, next stage, previous stage)
  double relR[3][9], relp[3][3], relJ[3][36], rellog[3][6], Fqq_prev6[36], Fqq_inv[36], tmp6[36], fq6[6];
  double t18[FB_NV], part[8];
};
// the line search evaluates trial slacks and per-row terms of the barrier cost / violation: it keeps the four row arrays
struct FbLsWork : FbRobotWork {
  double slack[FB_NCON], dual[FB_NCON], residual[FB_NCON], duality[FB_NCON];
};

template <int MODE>
__device__ __forceinline__ void fbw_mm(int lane, int m, int n, int k, const double* A, int ars, int acs, const double* B, int brs, int bcs,
                                       double* C, int ldc) {
  const int total = m * n;
  for (int e = lane; e < total; e += 32) {
    const int i = e / n, j = e - i * n;
    const double* a = A + i * ars;
    const double* b = B + j * bcs;
    double acc;
    int l0 = 0;
    if (MODE == FBM_SET) {
      if (k == 0) { C[i * ldc + j] = 0.0; continue; }
      acc = a[0] * b[0];
      l0 = 1;
    } else {
      acc = C[i * ldc + j];
    }
    if (MODE == FBM_SUB)
      for (int l = l0; l < k; ++l) acc = fma(-a[l * acs], b[l * brs], acc);
    else
      for (int l = l0; l < k; ++l) acc = fma(a[l * acs], b[l * brs], acc);
    C[i * ldc + j] = acc;
  }
}

// sum_k a[k * stride] x[k], k < n <= N, as one product and an ascending fma chain; a lives in HBM / L2 and its N loads are
// issued together
template <int N>
__device__ __forceinline__ double fbw_colT_dot(const double* a, int stride, const double* x, int n) {
  double r[N];
#pragma unroll
  for (int k = 0; k < N; ++k) r[k] = k < n ? __ldcg(a + k * stride) : 0.0;
  double acc = r[0] * x[0];
#pragma unroll
  for (int k = 1; k < N; ++k)
    if (k < n) acc = fma(r[k], x[k], acc);
  return acc;
}

// forwardKinematics in the world frame: base by lane 0, then one lane per leg (robot.hxx:193-230); v, a may be null
__device__ __noinline__ void fbw_forward_kinematics(FbRobotWork& w, int lane, const double* q, const double* v, const double* a) {
  if (lane == 0) {
    fb_quat_to_R(q + 3, w.R[0]);
    for (int i = 0; i < 3; ++i) w.p[0][i] = q[i];
    for (int c = 0; c < 3; ++c) {
      const double e[3] = {w.R[0][c], w.R[0][3 + c], w.R[0][6 + c]};
      for (int i = 0; i < 3; ++i) { w.S[c][i] = e[i]; w.S[c][3 + i] = 0.0; }
      fb_cross(w.p[0], e, w.S[3 + c]);
      for (int i = 0; i < 3; ++i) w.S[3 + c][3 + i] = e[i];
    }
    for (int i = 0; i < 6; ++i) {
      double accv = 0.0, acca = 0.0;
      if (v) { accv = w.S[0][i] * v[0]; for (int c = 1; c < 6; ++c) accv = fma(w.S[c][i], v[c], accv); }
      if (a) { acca = w.S[0][i] * a[0]; for (int c = 1; c < 6; ++c) acca = fma(w.S[c][i], a[c], acca); }
      w.ov[0][i] = accv;
      w.oa[0][i] = acca;
    }
    for (int c = 0; c < 6; ++c)
      for (int i = 0; i < 6; ++i) w.dV[c][i] = 0.0;
  }
  __syncwarp();
  if (lane < 4) {
    for (int jj = 0; jj < 3; ++jj) {
      const int j = 3 * lane + jj;
      const int b = 1 + j, pb = fb_parent_body(b), c = 6 + j;
      const double* Rp = w.R[pb];
      double* Rb = w.R[b];
      double sn, cs;
      canon_sincos(q[7 + j], &sn, &cs);
      if (ANYMAL_JOINT_AXIS[j] == 0) {
        for (int i = 0; i < 3; ++i) {
          Rb[3 * i] = Rp[3 * i];
          Rb[3 * i + 1] = fma(cs, Rp[3 * i + 1], sn * Rp[3 * i + 2]);
          Rb[3 * i + 2] = fma(cs, Rp[3 * i + 2], -(sn * Rp[3 * i + 1]));
        }
      } else {
        for (int i = 0; i < 3; ++i) {
          Rb[3 * i] = fma(cs, Rp[3 * i], -(sn * Rp[3 * i + 2]));
          Rb[3 * i + 1] = Rp[3 * i + 1];
          Rb[3 * i + 2] = fma(cs, Rp[3 * i + 2], sn * Rp[3 * i]);
        }
      }
      const double* P = ANYMAL_JOINT_P[j];
      for (int i = 0; i < 3; ++i) w.p[b][i] = fma(Rp[3 * i + 2], P[2], fma(Rp[3 * i + 1], P[1], fma(Rp[3 * i], P[0], w.p[pb][i])));
      const int ax = ANYMAL_JOINT_AXIS[j];
      const double e[3] = {Rb[ax], Rb[3 + ax], Rb[6 + ax]};
      fb_cross(w.p[b], e, w.S[c]);
      for (int i = 0; i < 3; ++i) w.S[c][3 + i] = e[i];
      fb_mxm(w.ov[pb], w.S[c], w.dV[c]);
      const double qd = v ? v[c] : 0.0, qdd = a ? a[c] : 0.0;
      for (int i = 0; i < 6; ++i) {
        w.ov[b][i] = fma(w.S[c][i], qd, w.ov[pb][i]);
        w.oa[b][i] = fma(w.dV[c][i], qd, fma(w.S[c][i], qdd, w.oa[pb][i]));
      }
    }
  }
  __syncwarp();
}

__device__ inline void fbw_contact_point(const FbRobotWork& w, int i, double* P) {
  const int b = 1 + ANYMAL_CONTACT_PARENT_JOINT[i];
  const double* R = w.R[b];
  const double* pc = ANYMAL_CONTACT_P[i];
  for (int r = 0; r < 3; ++r) P[r] = fma(R[3 * r + 2], pc[2], fma(R[3 * r + 1], pc[1], fma(R[3 * r], pc[0], w.p[b][r])));
}
__device__ inline void fbw_body_inertia(const FbRobotWork& w, int b, fb_inertia_t* Y) {
  const double m = ANYMAL_MASS[b];
  double c[3], T[9];
  const double* R = w.R[b];
  for (int i = 0; i < 3; ++i)
    c[i] = fma(R[3 * i + 2], ANYMAL_COM[b][2], fma(R[3 * i + 1], ANYMAL_COM[b][1], fma(R[3 * i], ANYMAL_COM[b][0], w.p[b][i])));
  const double* Ic = ANYMAL_INERTIA[b];
  const double If[9] = {Ic[0], Ic[1], Ic[2], Ic[1], Ic[3], Ic[4], Ic[2], Ic[4], Ic[5]};
  fb_mul33(R, If, T);
  const double cc = fb_dot3(c, c);
  const int ii[6] = {0, 0, 0, 1, 1, 2}, jj[6] = {0, 1, 2, 1, 2, 2};
  for (int e = 0; e < 6; ++e) {
    const int i = ii[e], j = jj[e];
    const double iw = fma(T[3 * i + 2], R[3 * j + 2], fma(T[3 * i + 1], R[3 * j + 1], T[3 * i] * R[3 * j]));
    const double par = (i == j) ? (cc - c[i] * c[j]) : -(c[i] * c[j]);
    Y->I[e] = fma(m, par, iw);
  }
  Y->m = m;
  for (int i = 0; i < 3; ++i) Y->h[i] = m * c[i];
}
__device__ inline void fb_pullback(const double* Rf, const double* Pf, const double* x, double* y) {
  double t[3], u[3];
  fb_cross(x + 3, Pf, t);
  for (int i = 0; i < 3; ++i) u[i] = x[i] + t[i];
  fb_rotT(Rf, u, y);
  fb_rotT(Rf, x + 3, y + 3);
}
__device__ inline int fb_in_support(int contact, int c) { return c < 6 || (c - 6) / 3 == contact; }

// RNEA + computeRNEADerivatives with the contact wrenches (robot.hxx:444-500): tau -> L.IDC[0:18], d tau/dq, /dv ->
// L.dIDCdqv rows 0..17, d tau/da -> L.Mm (all in HBM; written once).  with_dv = false: RNEAImpulseDerivatives.
__device__ __noinline__ void fbw_rnea_derivatives(FbRobotWork& w, int lane, double gravity, bool with_dv, FbLin& L, bool derivatives) {
  if (lane < FB_NB) {
    const int b = lane;
    fbw_body_inertia(w, b, &w.Y[b]);
    for (int i = 0; i < 6; ++i) w.agf[b][i] = w.oa[b][i];
    w.agf[b][2] = w.oa[b][2] + gravity;
    double Ya[6], h[6], vh[6];
    fb_Ymul(&w.Y[b], w.agf[b], Ya);
    fb_Ymul(&w.Y[b], w.ov[b], h);
    fb_mxf(w.ov[b], h, vh);
    for (int i = 0; i < 6; ++i) w.F[b][i] = Ya[i] + vh[i];
    fb_dinertia(&w.Y[b], w.ov[b], &w.D[b]);
  }
  __syncwarp();
  if (lane < FB_NC) {   // every contact sits on its own body (the shank of its leg)
    const int b = 1 + ANYMAL_CONTACT_PARENT_JOINT[lane];
    double P[3], W6[6];
    fbw_contact_point(w, lane, P);
    fb_rot(w.R[b], w.fm + 3 * lane, W6);
    fb_cross(P, W6, W6 + 3);
    for (int e = 0; e < 6; ++e) w.F[b][e] -= W6[e];
  }
  __syncwarp();
  // composites, leaves to root: inside every leg by its own lane, then the base collects the hips in the serial
  // order b = 10, 7, 4, 1 (the reverse body order of pinocchio's backward pass)
  if (lane < 4) {
    for (int b = 3 * lane + 3; b > 3 * lane + 1; --b) {
      const int pb = b - 1;
      w.Y[pb].m += w.Y[b].m;
      for (int i = 0; i < 3; ++i) { w.Y[pb].h[i] += w.Y[b].h[i]; w.D[pb].pl[i] += w.D[b].pl[i]; w.D[pb].pa[i] += w.D[b].pa[i]; }
      for (int i = 0; i < 6; ++i) { w.Y[pb].I[i] += w.Y[b].I[i]; w.D[pb].S[i] += w.D[b].S[i]; w.F[pb][i] += w.F[b][i]; }
    }
  }
  __syncwarp();
  if (lane == 0) {
    for (int b = 10; b >= 1; b -= 3) {
      w.Y[0].m += w.Y[b].m;
      for (int i = 0; i < 3; ++i) { w.Y[0].h[i] += w.Y[b].h[i]; w.D[0].pl[i] += w.D[b].pl[i]; w.D[0].pa[i] += w.D[b].pa[i]; }
      for (int i = 0; i < 6; ++i) { w.Y[0].I[i] += w.Y[b].I[i]; w.D[0].S[i] += w.D[b].S[i]; w.F[0][i] += w.F[b][i]; }
    }
  }
  __syncwarp();
  if (lane < FB_NV) {
    const int c = lane, b = fb_body_of_dof(c);
    L.IDC[c] = fb_dot6(w.S[c], w.F[b]);
    if (derivatives) {
      double dJ[6], t1[6], t2[6];
      fb_mxm(w.ov[b], w.S[c], dJ);
      if (b == 0) {
        const double a0[6] = {0.0, 0.0, gravity, 0.0, 0.0, 0.0};
        fb_mxm(a0, w.S[c], w.dAq[c]);
      } else {
        const int pb = fb_parent_body(b);
        fb_mxm(w.agf[pb], w.S[c], t1);
        fb_mxm(w.ov[pb], w.dV[c], t2);
        for (int i = 0; i < 6; ++i) w.dAq[c][i] = t1[i] + t2[i];
      }
      for (int i = 0; i < 6; ++i) w.dAv[c][i] = dJ[i] + w.dV[c][i];
      fb_Ymul(&w.Y[b], w.S[c], w.U[c]);
      fb_DTmul(&w.D[b], w.S[c], w.W[c]);
      fb_Dmul(&w.D[b], w.S[c], t1);
      fb_Ymul(&w.Y[b], w.dAv[c], t2);
      for (int i = 0; i < 6; ++i) w.dFv[c][i] = t1[i] + t2[i];
      fb_Dmul(&w.D[b], w.dV[c], t1);
      fb_Ymul(&w.Y[b], w.dAq[c], t2);
      for (int i = 0; i < 6; ++i) w.dFq[c][i] = t1[i] + t2[i];
      fb_mxf(w.S[c], w.F[b], t1);
      for (int i = 0; i < 6; ++i) w.dFqa[c][i] = w.dFq[c][i] + t1[i];
    }
  }
  __syncwarp();
  if (!derivatives) return;
  FBW_FOR(e, FB_NV * FB_NV) {
    const int r = e / FB_NV, c = e - r * FB_NV;
    double eq = 0.0, ev = 0.0, em = 0.0;
    // d tau/da: robot.hxx:496-499 overwrites the strictly lower triangle with the mirror of the upper one
    if (fb_same_joint(r, c)) {
      eq = fb_dot6(w.S[r], w.dFq[c]);
      ev = fb_dot6(w.S[r], w.dFv[c]);
      em = c >= r ? fb_dot6(w.S[r], w.U[c]) : fb_dot6(w.S[c], w.U[r]);
    } else if (fb_is_ancestor(r, c)) {
      eq = fb_dot6(w.S[r], w.dFqa[c]);
      ev = fb_dot6(w.S[r], w.dFv[c]);
      em = fb_dot6(w.S[r], w.U[c]);
    } else if (fb_is_ancestor(c, r)) {
      eq = fb_dot6(w.dAq[c], w.U[r]) + fb_dot6(w.dV[c], w.W[r]);
      ev = fb_dot6(w.dAv[c], w.U[r]) + fb_dot6(w.S[c], w.W[r]);
      em = fb_dot6(w.S[c], w.U[r]);
    }
    L.dIDCdqv[r * FB_NX + c] = eq;
    L.dIDCdqv[r * FB_NX + FB_NV + c] = with_dv ? ev : 0.0;
    L.Mm[e] = em;
  }
  __syncwarp();
}

// one relative placement M = M(q_minus)^-1 M(q_plus), its log6 and Jlog6 (robot.hxx subtractConfiguration /
// dSubtractdConfigurationPlus); lanes 0..2 run it in lock-step on three pairs
__device__ __noinline__ void fbw_se3_pair(const double* q_plus, const double* q_minus, double* R, double* p, double* log18, double* J) {
  fb_relative(q_minus, q_plus, R, p);
  fb_log6(R, p, log18);   // the base block; the joint part of the difference is a plain subtraction (done by the callers)
  fb_Jlog6(R, p, J);
}
// dSubtractdConfigurationMinus from the pieces above: J1 (-Ad(M^-1)) (robot.hxx:138-153)
__device__ __noinline__ void fbw_dminus(const double* R, const double* p, const double* J1, double* J6) {
  double X[36];
  double Sk[9] = {0, -p[2], p[1], p[2], 0, -p[0], -p[1], p[0], 0}, RtS[9];
  fb_mulT33(R, Sk, RtS);
  for (int r = 0; r < 3; ++r)
    for (int k = 0; k < 3; ++k) {
      X[6 * r + k] = -R[3 * k + r];
      X[6 * r + 3 + k] = RtS[3 * r + k];
      X[6 * (3 + r) + k] = 0.0;
      X[6 * (3 + r) + 3 + k] = -R[3 * k + r];
    }
  for (int r = 0; r < 6; ++r)
    for (int k = 0; k < 6; ++k) {
      double acc = J1[6 * r] * X[k];
      for (int j = 1; j < 6; ++j) acc = fma(J1[6 * r + j], X[6 * j + k], acc);
      J6[6 * r + k] = acc;
    }
}

constexpr int FB_ROBOT_WARPS = 6;   // x 2 CTAs per SM: 12 warps (18.6 KB of shared memory and 168 registers each)
constexpr int FB_ROBOT_MINB = 2;
constexpr int FB_LS_WARPS = 5;      // k_fb_ls_eval (FbLsWork, 23 KB per warp)

// IREF: the cost reference of (slot, instance) comes from A.iref instead of the chain element shared by the batch
template <bool RESIDUAL_ONLY, bool IREF>
__global__ void __launch_bounds__(32 * FB_ROBOT_WARPS, FB_ROBOT_MINB) k_fb_robot(FbArrays A, FbLin* lin) {
  IDOCP_DYN_SMEM(FbRobotWork, wbase);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int stage = blockIdx.x * FB_ROBOT_WARPS + warp;
  if (stage >= A.B * A.n_elems) return;
  FbRobotWork& w = wbase[warp];
  const int b = stage / A.n_elems, e = stage - b * A.n_elems;
  const FbElem& el = A.elems[e];
  const FbDevProblem& pr = *A.prob;
  const int nl = fbc_cone_bits(pr);
  const int kind = el.kind;
  const bool impulse = kind == FB_IMPULSE, terminal = kind == FB_TERMINAL;
  const double dt = (impulse || terminal) ? 1.0 : el.dt;
  const int dimf = terminal ? 0 : el.dimf, nvf = FB_NV + dimf, dimi = el.sw ? el.dimi : 0;
  const size_t rec = (size_t)el.slot * A.B + b;
  const FbSol& S = A.sol[rec];
  FbDir& Dr = A.dir[rec];
  FbLin& L = lin[rec];

  // ---- load ----
  // every load of the lane is issued before its first store (a copy loop through generic pointers keeps load -> store order:
  // one DRAM round trip per element)
  {
    constexpr int NS = (int)(offsetof(FbSol, slack) / sizeof(double)), RS = (NS + 31) / 32;   // lmd ... xi
    const double* src = S.lmd;
    const FbSol& Nx = A.sol[(size_t)(terminal ? el.slot : el.next_slot) * A.B + b];
    const double* qp = el.prev_slot >= 0 ? A.sol[(size_t)el.prev_slot * A.B + b].q : A.q0 + (size_t)b * FB_NQ;
    double r[RS], n0 = 0.0, n1 = 0.0, n2 = 0.0, n3 = 0.0, p0 = 0.0;
#pragma unroll
    for (int i = 0; i < RS; ++i) { const int x = lane + 32 * i; r[i] = x < NS ? __ldcg(src + x) : 0.0; }
    if (!terminal) {
      if (lane < FB_NV) { n0 = __ldcg(Nx.lmd + lane); n1 = __ldcg(Nx.gmm + lane); n2 = __ldcg(Nx.v + lane); }
      if (lane < FB_NQ) n3 = __ldcg(Nx.q + lane);
    }
    if (lane < FB_NQ) p0 = __ldcg(qp + lane);
    double* dst = w.lmd;
#pragma unroll
    for (int i = 0; i < RS; ++i) { const int x = lane + 32 * i; if (x < NS) dst[x] = r[i]; }
    if (!terminal) {
      if (lane < FB_NV) { w.nlmd[lane] = n0; w.ngmm[lane] = n1; w.nv[lane] = n2; }
      if (lane < FB_NQ) w.nq[lane] = n3;
    }
    if (lane < FB_NQ) w.qprev[lane] = p0;
  }
  __syncwarp();
  if (lane < FB_MAXF) {   // forces of inactive contacts are zero for the dynamics; stacks of the active ones
    const int i = lane / 3;
    w.fm[lane] = (!terminal && el.active[i]) ? w.f[lane] : 0.0;
    if (!terminal && el.active[i]) {
      int k = 0;
      for (int j = 0; j < i; ++j) k += el.active[j];
      w.mu_stack[3 * k + lane % 3] = w.mu[lane];
    }
  }
  // ---- SE(3): lanes 0..2 in lock-step on (q, q_ref), (q, q_next), (q_prev, q) ----
  if (lane < 3 && !(terminal && lane == 1)) {
    const double* qp = lane == 2 ? w.qprev : w.q;
    const double* qm = lane == 0 ? fb_ref_q<IREF>(A, el, rec) : (lane == 1 ? w.nq : w.q);
    fbw_se3_pair(qp, qm, w.relR[lane], w.relp[lane], w.rellog[lane], w.relJ[lane]);
  }
  __syncwarp();
  // (rellog holds 6 base entries; the joint differences are recomputed where needed)
  if (!RESIDUAL_ONLY) {
    if ((lane == 1 && !terminal) || lane == 2) fbw_dminus(w.relR[lane], w.relp[lane], w.relJ[lane], lane == 1 ? w.tmp6 : w.Fqq_prev6);
    __syncwarp();
    if ((lane == 1 && !terminal) || lane == 2) fb_dsubtract_inverse(lane == 1 ? w.tmp6 : w.Fqq_prev6, lane == 1 ? w.Fqq_inv : L.Fqq_prev_inv);
  } else {
    if (lane == 2) fbw_dminus(w.relR[2], w.relp[2], w.relJ[2], w.Fqq_prev6);
  }
  __syncwarp();
  const double* J6c = w.relJ[0];
  const double* Fqq6 = w.relJ[1];

  // ---- cost gradient (trotting_configuration_space_cost.cpp:283-311) ----
  const double* wq = terminal ? pr.qf_weight : (impulse ? pr.qi_weight : pr.q_weight);
  const double* wv = terminal ? pr.vf_weight : (impulse ? pr.vi_weight : pr.v_weight);
  const double* wa = impulse ? pr.dvi_weight : pr.a_weight;
  const double sc = (terminal || impulse) ? 1.0 : dt;
  double lq = 0.0, lv = 0.0, la = 0.0, Fq = 0.0, Fv = 0.0;   // lane j < 18 owns element j of the stage vectors
  double lf = 0.0;                                             // lane j < 12 owns lf[j] (stacked)
  double lu = 0.0, lup = 0.0;                                  // lane j < 12 owns lu[j]; lane j < 6 owns lu_passive[j]
  // contact owning stacked row `lane` (for lf): ci = contact index, cx = axis
  int ci = -1, cx = 0;
  if (!terminal && lane < dimf) {
    int k = lane / 3, cnt = 0;
    for (int i = 0; i < FB_NC; ++i)
      if (el.active[i]) { if (cnt == k) ci = i; ++cnt; }
    cx = lane % 3;
  }
  if (lane < FB_NV) {
    const int j = lane;
    const double qd = j < 6 ? w.rellog[0][j] : (w.q[1 + j] - fb_ref_q<IREF>(A, el, rec)[1 + j]);
    if (j < 6) {
      double acc = J6c[j] * (wq[0] * w.rellog[0][0]);
      for (int k = 1; k < 6; ++k) acc = fma(J6c[6 * k + j], wq[k] * w.rellog[0][k], acc);
      lq += sc * acc;
    } else {
      lq += sc * (wq[j] * qd);
    }
    lv += sc * (wv[j] * (w.v[j] - fb_ref_v<IREF>(A, el, rec)[j]));
    if (!terminal) la += sc * (wa[j] * w.a[j]);
  }
  if (ci >= 0) {   // ContactForceCost gradient (contact_force_cost.cpp:161-187)
    const double* fw = impulse ? pr.fi_weight : pr.f_weight;
    const double* fr = impulse ? pr.fi_ref : pr.f_ref;
    lf += sc * (fw[3 * ci + cx] * (w.f[3 * ci + cx] - fr[3 * ci + cx]));
  }
  // computePrimalAndDualResidual
  if (!terminal) {
    const int ncon = FBC_LIVE_ROWS(el.cactive);
    FBW_FOR(idx, ncon) {
      const int c = fbc_comp(idx);
      const int j = idx - fbc_offset(c);
      double res = 0.0, dua = 0.0;
      if (el.cactive[c] && j < fbc_rows(nl, c) && c != FBC_DISTANCE) {   // ContactDistance: after the kinematics, below
        const double sl = S.slack[idx];
        if (fbc_is_cone(c)) {
          int i, ee;
          fbc_cone_row(nl, c, j, i, ee);
          if (el.active[i]) {
            double r5[5];
            fb_friction_residual(pr.mu, fbc_cone_rows(nl, c) == 2, w.f + 3 * i, r5);
            res = r5[ee] + sl;
            dua = sl * S.dual[idx] - pr.barrier;
          }
        } else {
          res = sl - fbc_box_margin(c, j, pr, w.q, w.v, w.a, w.u);
          dua = sl * S.dual[idx] - pr.barrier;
        }
      }
      Dr.residual[idx] = res;
      Dr.duality[idx] = dua;
    }
  }
  __syncwarp();
  if (terminal) {
    // TerminalOCP::linearizeOCP (terminal_ocp.hxx:50-66), linearizeForwardEulerTerminal (state_equation.hxx:66-82)
    if (lane < FB_NV) {
      const int j = lane;
      if (j < 6) {
        for (int k = 0; k < 6; ++k) lq = fma(w.Fqq_prev6[6 * k + j], w.lmd[k], lq);
      } else {
        lq -= w.lmd[j];
      }
      lv -= w.gmm[j];
      L.lq[j] = lq;
      L.lv[j] = lv;
    }
    if (!RESIDUAL_ONLY) {
      FBW_FOR(x, 36) {
        const int r = x / 6, c = x - 6 * r;
        double acc = J6c[r] * (wq[0] * J6c[c]);
        for (int k = 1; k < 6; ++k) acc = fma(J6c[6 * k + r], wq[k] * J6c[6 * k + c], acc);
        L.Qqq6[x] = 0.0 + acc;
      }
      if (lane < FB_NV) {
        L.Qqq_d[lane] = lane >= 6 ? 0.0 + wq[lane] : 0.0;
        L.Qvv_d[lane] = 0.0 + wv[lane];
      }
    }
    __syncwarp();
    if (lane == 0) {
      Dr.kkt_sq = fb_sqnorm(L.lq, FB_NV) + fb_sqnorm(L.lv, FB_NV);
      Dr.info = 0.0;
    }
    return;
  }
  // augmentDualResidual: joint limits on the lq / lv / lu tails, friction cones on lf
  if (lane >= 6 && lane < FB_NV) {
    const int j = lane - 6;
    for (int c = 0; c < 4; ++c) {
      if (!el.cactive[c]) continue;
      const double sg = (c & 1) ? 1.0 : -1.0;
      if (c <= FBC_POS_UP) lq += sg * (dt * S.dual[fbc_offset(c) + j]);
      else lv += sg * (dt * S.dual[fbc_offset(c) + j]);
    }
    for (int c = FBC_ACC_LO; c <= FBC_ACC_UP; ++c) {   // JointAcceleration{Lower,Upper}Limit: la.tail(12) -/+= dt dual
      if (!el.cactive[c]) continue;
      const double sg = (c & 1) ? 1.0 : -1.0;
      la += sg * (dt * S.dual[fbc_offset(c) + j]);
    }
  }
  if (lane < FB_NU) {
    for (int c = 4; c < 6; ++c) {
      if (!el.cactive[c]) continue;
      const double sg = (c & 1) ? 1.0 : -1.0;
      lu += sg * (dt * S.dual[fbc_offset(c) + lane]);
    }
  }
  const int cfr = impulse ? FBC_IMPULSE_FRICTION : FBC_FRICTION;
  const int rpc = fbc_cone_rows(nl, cfr);
  const bool nlc = rpc == 2;
  if (ci >= 0 && el.cactive[cfr]) {
    const double* du5 = S.dual + fbc_offset(cfr) + rpc * ci;
    const double* fi = w.f + 3 * ci;
    const double acc = nlc ? fb_cone_augment<true>(pr.mu, fi, du5, cx) : fb_cone_augment<false>(pr.mu, fi, du5, cx);
    lf += dt * acc;
  }
  // linearizeForwardEuler / linearizeImpulseForwardEuler (state_equation.hxx:11-40)
  if (lane < FB_NV) {
    const int j = lane;
    Fq = j < 6 ? w.rellog[1][j] : (w.q[1 + j] - w.nq[1 + j]);
    if (!impulse) {
      Fq = fma(dt, w.v[j], Fq);
      Fv = fma(dt, w.a[j], w.v[j]) - w.nv[j];
    } else {
      Fv = (w.v[j] + w.a[j]) - w.nv[j];
    }
    if (j < 6) {
      for (int k = 0; k < 6; ++k) lq = fma(Fqq6[6 * k + j], w.nlmd[k], lq);
      for (int k = 0; k < 6; ++k) lq = fma(w.Fqq_prev6[6 * k + j], w.lmd[k], lq);
    } else {
      lq += w.nlmd[j] - w.lmd[j];
    }
    if (!impulse) {
      lv += (fma(dt, w.nlmd[j], w.ngmm[j]) - w.gmm[j]);
      la = fma(dt, w.ngmm[j], la);
    } else {
      lv += (w.ngmm[j] - w.gmm[j]);
      la += w.ngmm[j];
    }
    w.t18[j] = Fq;
  }
  __syncwarp();
  if (!RESIDUAL_ONLY) {
    // condenseForwardEuler: Fqq := -Fqq_inv Fqq, Fqv := -dt Fqq_inv, Fq[0:6] := -Fqq_inv Fq[0:6]
    FBW_FOR(x, 36) {
      const int r = x / 6, c = x - 6 * r;
      double acc = w.Fqq_inv[6 * r] * Fqq6[c];
      for (int k = 1; k < 6; ++k) acc = fma(w.Fqq_inv[6 * r + k], Fqq6[6 * k + c], acc);
      L.Fqq6[x] = -acc;
      L.Fqv6[x] = impulse ? 0.0 : -dt * w.Fqq_inv[x];
    }
    if (lane < 6) {
      double acc = w.Fqq_inv[6 * lane] * w.t18[0];
      for (int k = 1; k < 6; ++k) acc = fma(w.Fqq_inv[6 * lane + k], w.t18[k], acc);
      Fq = -acc;
    }
  }
  __syncwarp();

  // ---- contact dynamics: kinematics, RNEA + derivatives, contact rows ----
  const double baumgarte = pr.T / pr.N;
  if (!impulse) {
    fbw_forward_kinematics(w, lane, w.q, w.v, w.a);
    fbw_rnea_derivatives(w, lane, ANYMAL_GRAVITY, true, L, true);
    if (lane < FB_NU) L.IDC[6 + lane] -= w.u[lane];
  } else {
    fbw_forward_kinematics(w, lane, w.q, nullptr, w.a);
    fbw_rnea_derivatives(w, lane, 0.0, false, L, true);
    if (lane < FB_NV) w.t18[lane] = w.v[lane] + w.a[lane];
    __syncwarp();
    fbw_forward_kinematics(w, lane, w.q, w.t18, nullptr);
  }
  // rows of every active contact, one after the other; lane = dof
  {
    int k = 0;
    for (int i = 0; i < FB_NC; ++i) {
      if (!el.active[i]) continue;
      const int bi = 1 + ANYMAL_CONTACT_PARENT_JOINT[i];
      const double* Rf = w.R[bi];
      if (lane == 0) fbw_contact_point(w, i, w.frP);
      __syncwarp();
      if (lane == 0) fb_pullback(Rf, w.frP, w.ov[bi], w.frV);
      if (lane == 1) fb_pullback(Rf, w.frP, w.oa[bi], w.frA);
      __syncwarp();
      const double* P = w.frP;
      const double* vF = w.frV;
      if (lane == 31) {
        double* C = L.IDC + FB_NV + 3 * k;
        if (!impulse) {
          const double wvv = 2.0 / baumgarte, wpp = 1.0 / (baumgarte * baumgarte);
          double wxv[3];
          fb_cross(vF + 3, vF, wxv);
          for (int x = 0; x < 3; ++x) {
            const double acl = w.frA[x] + wxv[x];
            C[x] = fma(wpp, P[x] - el.cpoints[3 * i + x], fma(wvv, vF[x], acl));
          }
        } else {
          for (int x = 0; x < 3; ++x) C[x] = vF[x];
        }
      }
      if (lane < FB_NV) {
        const int c = lane;
        double J[6] = {0, 0, 0, 0, 0, 0}, vq[6] = {0, 0, 0, 0, 0, 0}, aq[6] = {0, 0, 0, 0, 0, 0}, av[6] = {0, 0, 0, 0, 0, 0};
        if (fb_in_support(i, c)) {
          fb_pullback(Rf, P, w.S[c], J);
          const int bb = fb_body_of_dof(c);
          double u[6], x6[6], t1[6], t2[6];
          if (bb == 0) {
            for (int ee = 0; ee < 6; ++ee) u[ee] = w.ov[bi][ee];
          } else {
            const int pb = fb_parent_body(bb);
            for (int ee = 0; ee < 6; ++ee) u[ee] = w.ov[bi][ee] - w.ov[pb][ee];
            fb_pullback(Rf, P, w.dV[c], vq);
          }
          if (!impulse) {
            fb_mxm(w.ov[bb], w.S[c], t1);
            fb_mxm(w.S[c], u, t2);
            for (int ee = 0; ee < 6; ++ee) x6[ee] = t1[ee] + t2[ee];
            fb_pullback(Rf, P, x6, av);
            if (bb != 0) {
              const int pb = fb_parent_body(bb);
              fb_mxm(w.oa[pb], w.S[c], t1);
              fb_mxm(w.dV[c], u, t2);
              for (int ee = 0; ee < 6; ++ee) x6[ee] = t1[ee] + t2[ee];
              fb_pullback(Rf, P, x6, aq);
            }
          }
        }
        double* rq = L.dIDCdqv + (FB_NV + 3 * k) * FB_NX + c;
        double* rv = rq + FB_NV;
        double* ra = L.dCda + (3 * k) * FB_NV + c;
        if (!impulse) {
          const double wvv = 2.0 / baumgarte, wpp = 1.0 / (baumgarte * baumgarte);
          const double* vl = vF;
          const double* va = vF + 3;
          double t1[3], t2[3], RJ[3];
          fb_cross(va, vq, t1);
          fb_cross(vl, vq + 3, t2);
          fb_rot(Rf, J, RJ);
          for (int x = 0; x < 3; ++x) rq[x * FB_NX] = fma(wpp, RJ[x], fma(wvv, vq[x], (aq[x] + t1[x]) + t2[x]));
          fb_cross(va, J, t1);
          fb_cross(vl, J + 3, t2);
          for (int x = 0; x < 3; ++x) rv[x * FB_NX] = fma(wvv, J[x], (av[x] + t1[x]) + t2[x]);
          for (int x = 0; x < 3; ++x) ra[x * FB_NV] = J[x];
        } else {
          for (int x = 0; x < 3; ++x) { rq[x * FB_NX] = vq[x]; rv[x * FB_NX] = J[x]; ra[x * FB_NV] = J[x]; }
        }
      }
      __syncwarp();
      ++k;
    }
  }
  __syncwarp();
  // augment: lq += dt dIDdq^T beta, lv += dt dIDdv^T beta, la += dt M^T beta, lf -= dt dCda beta, lu ...
  {
    const double* dIDdq = L.dIDCdqv;
    const double* dIDdv = L.dIDCdqv + FB_NV;
    const double* dCdq = L.dIDCdqv + FB_NV * FB_NX;
    const double* dCdv = dCdq + FB_NV;
    // the matrices were written to HBM by other lanes of this warp; a column is fetched in one batch (all loads in flight),
    // then folded in ascending k
    if (lane < FB_NV) {
      const int j = lane;
      lq = fma(dt, fbw_colT_dot<FB_NV>(dIDdq + j, FB_NX, w.beta, FB_NV), lq);
      if (!impulse) lv = fma(dt, fbw_colT_dot<FB_NV>(dIDdv + j, FB_NX, w.beta, FB_NV), lv);
      la = fma(dt, fbw_colT_dot<FB_NV>(L.Mm + j, FB_NV, w.beta, FB_NV), la);
      if (dimf > 0) {
        lq = fma(dt, fbw_colT_dot<FB_MAXF>(dCdq + j, FB_NX, w.mu_stack, dimf), lq);
        lv = fma(dt, fbw_colT_dot<FB_MAXF>(dCdv + j, FB_NX, w.mu_stack, dimf), lv);
        la = fma(dt, fbw_colT_dot<FB_MAXF>(L.dCda + j, FB_NV, w.mu_stack, dimf), la);
      }
    }
    if (lane < dimf) lf = fma(-dt, fbw_colT_dot<FB_NV>(L.dCda + lane * FB_NV, 1, w.beta, FB_NV), lf);
    if (!impulse) {
      if (lane < FB_NPASS) lup = fma(-dt, w.beta[lane], dt * w.nu_passive[lane]);
      if (lane < FB_NU) lu = fma(-dt, w.beta[6 + lane], lu);
    }
  }
  // ---- ContactDistance (contact_distance.cpp:73-110,134-150) on the contacts that are NOT active: residual = -z + slack with z
  // the height of the contact frame, lq -= dt dual J2, J2 = row 2 of the frame Jacobian (distance_mode 1: LOCAL frame, the
  // reference literally; 2: world-aligned = d z / d q).  After the dynamics terms, like the oracle (it needs these kinematics).
  // (nothing of this block stays in registers: the condensing below re-reads J2 and the residuals, so that the kernel keeps its
  // register allocation while the component is off)
  const bool cd_on = !impulse && el.cactive[FBC_DISTANCE];
  if (cd_on) {
    const int o = fbc_offset(FBC_DISTANCE);
    for (int i = 0; i < FB_NC; ++i) {
      double cdres = 0.0, cddua = 0.0;
      if (!el.active[i]) {   // (uniform over the warp)
        const int bi = 1 + ANYMAL_CONTACT_PARENT_JOINT[i];
        const double* Rf = w.R[bi];
        __syncwarp();
        if (lane == 0) fbw_contact_point(w, i, w.frP);
        __syncwarp();
        if (lane < FB_NV) {
          double J[6] = {0, 0, 0, 0, 0, 0};
          if (fb_in_support(i, lane)) fb_pullback(Rf, w.frP, w.S[lane], J);
          const double j2 = pr.distance_mode == 2 ? fma(Rf[8], J[2], fma(Rf[7], J[1], Rf[6] * J[0])) : J[2];
          L.cdJ[i * FB_NV + lane] = j2;   // read again by the condensing below, by k_fb_condense and by k_fb_expand
          lq -= (dt * S.dual[o + i]) * j2;
        }
        cdres = -w.frP[2] + S.slack[o + i];
        cddua = S.slack[o + i] * S.dual[o + i] - pr.barrier;
      }
      if (lane == 0) {
        Dr.residual[o + i] = cdres; Dr.duality[o + i] = cddua;
      }
    }
    __syncwarp();
  }

  if (!RESIDUAL_ONLY) {
    // ---- cost Hessian (sparse part of Qxx, Qaa, Qff) and condenseSlackAndDual ----
    FBW_FOR(x, 36) {
      const int r = x / 6, c = x - 6 * r;
      double acc = J6c[r] * (wq[0] * J6c[c]);
      for (int k = 1; k < 6; ++k) acc = fma(J6c[6 * k + r], wq[k] * J6c[6 * k + c], acc);
      L.Qqq6[x] = 0.0 + sc * acc;
    }
    FBW_FOR(x, FB_MAXF * FB_MAXF) L.Qff[x] = 0.0;
    __syncwarp();
    double qqd = 0.0, qvd = 0.0, qud = 0.0;
    if (lane < FB_NV) {
      const int j = lane;
      if (j >= 6) qqd += sc * wq[j];
      qvd += sc * wv[j];
      double qad = 0.0 + sc * wa[j];
      if (j >= 6) {
        for (int c = FBC_ACC_LO; c <= FBC_ACC_UP; ++c) {
          if (!el.cactive[c]) continue;
          const int idx = fbc_offset(c) + j - 6;
          double h, g;
          pdipm_condense(dt, S.slack[idx], S.dual[idx], Dr.residual[idx], Dr.duality[idx], h, g);
          qad += h;
          const double sg = (c & 1) ? 1.0 : -1.0;
          la += sg * g;
        }
      }
      L.Qaa[j] = qad;
    }
    double qff_d = 0.0;   // diagonal entry of Qff owned by this lane (stacked row `lane`); no read-modify-write on HBM
    if (ci >= 0) {
      const double* fw = impulse ? pr.fi_weight : pr.f_weight;
      qff_d = 0.0 + sc * fw[3 * ci + cx];
    }
    if (lane >= 6 && lane < FB_NV) {
      const int j = lane - 6;
      for (int c = 0; c < 4; ++c) {
        if (!el.cactive[c]) continue;
        const int idx = fbc_offset(c) + j;
        double h, g;
        pdipm_condense(dt, S.slack[idx], S.dual[idx], Dr.residual[idx], Dr.duality[idx], h, g);
        const double sg = (c & 1) ? 1.0 : -1.0;
        if (c <= FBC_POS_UP) { qqd += h; lq += sg * g; }
        else { qvd += h; lv += sg * g; }
      }
    }
    if (lane < FB_NU) {
      for (int c = 4; c < 6; ++c) {
        if (!el.cactive[c]) continue;
        const int idx = fbc_offset(c) + lane;
        double h, g;
        pdipm_condense(dt, S.slack[idx], S.dual[idx], Dr.residual[idx], Dr.duality[idx], h, g);
        qud += h;
        const double sg = (c & 1) ? 1.0 : -1.0;
        lu += sg * g;
      }
      L.Quu_d[lane] = qud;
    }
    if (lane < FB_NV) { L.Qqq_d[lane] = qqd; L.Qvv_d[lane] = qvd; }
    if (ci >= 0 && el.cactive[cfr]) {
      int k = lane / 3;
      const int o = fbc_offset(cfr) + rpc * ci;
      const double* fi = w.f + 3 * ci;
      double h3[3];
      const double acc = nlc ? fb_cone_condense<true>(pr.mu, fi, S.slack + o, S.dual + o, Dr.residual + o, Dr.duality + o, cx, h3)
                             : fb_cone_condense<false>(pr.mu, fi, S.slack + o, S.dual + o, Dr.residual + o, Dr.duality + o, cx, h3);
      lf += dt * acc;
      for (int y = 0; y < 3; ++y) {
        const double h = h3[y];
        L.Qff[(3 * k + cx) * FB_MAXF + 3 * k + y] = (y == cx ? qff_d : 0.0) + dt * h;
      }
    } else if (ci >= 0) {
      L.Qff[lane * FB_MAXF + lane] = qff_d;
    }
    if (cd_on) {   // ContactDistance::condenseSlackAndDual: lq -= g J2 here, Qqq += w J2^T J2 in k_fb_condense (dense 18 x 18)
      const int o = fbc_offset(FBC_DISTANCE);
      for (int i = 0; i < FB_NC; ++i) {
        double wgt = 0.0;
        if (!el.active[i]) {
          double g2;
          pdipm_condense(dt, S.slack[o + i], S.dual[o + i], Dr.residual[o + i], Dr.duality[o + i], wgt, g2);
          if (lane < FB_NV) lq -= g2 * L.cdJ[i * FB_NV + lane];   // written by this very lane above
        }
        if (lane == 0) L.cdw[i] = wgt;
      }
    }
  }

  // ---- ForwardSwitchingConstraint::linearizeSwitchingConstraint (:27-68) ----
  if (dimi > 0) {
    const double c1 = el.dt + el.dt_next, c2 = el.dt * el.dt_next;
    __syncwarp();
    if (lane < FB_NV) w.dqv[lane] = fma(c2, w.a[lane], c1 * w.v[lane]);
    __syncwarp();
    if (lane == 0) fb_integrate(w.q, w.dqv, 1.0, w.q2);
    __syncwarp();
    if (lane == 0) fb_dintegrate_dq(w.dqv, w.Jq6);
    __syncwarp();
    if (lane == 0) fb_dintegrate_dv(w.dqv, w.Jv6);
    __syncwarp();
    fbw_forward_kinematics(w, lane, w.q2, nullptr, nullptr);
    {
      int k = 0;
      for (int i = 0; i < FB_NC; ++i) {
        if (!el.imp_active[i]) continue;
        const double* Rf = w.R[1 + ANYMAL_CONTACT_PARENT_JOINT[i]];
        if (lane == 0) fbw_contact_point(w, i, w.frP);
        __syncwarp();
        if (lane < 3) L.P[3 * k + lane] = w.frP[lane] - el.ipoints[3 * i + lane];
        if (lane < FB_NV) {
          const int c = lane;
          double J[6] = {0, 0, 0, 0, 0, 0}, wl[3];
          if (fb_in_support(i, c)) fb_pullback(Rf, w.frP, w.S[c], J);
          fb_rot(Rf, J, wl);
          for (int x = 0; x < 3; ++x) w.Pq[(3 * k + x) * FB_NV + c] = wl[x];
        }
        __syncwarp();
        ++k;
      }
    }
    __syncwarp();
    fbw_mm<FBM_SET>(lane, dimi, 6, 6, w.Pq, FB_NV, 1, w.Jq6, 6, 1, L.Phix, FB_NX);
    fbw_mm<FBM_SET>(lane, dimi, 6, 6, w.Pq, FB_NV, 1, w.Jv6, 6, 1, w.PJv, FB_NV);
    FBW_FOR(x, dimi * (FB_NV - 6)) {
      const int r = x / (FB_NV - 6), c = 6 + x - r * (FB_NV - 6);
      L.Phix[r * FB_NX + c] = w.Pq[r * FB_NV + c];
      w.PJv[r * FB_NV + c] = w.Pq[r * FB_NV + c];
    }
    __syncwarp();
    FBW_FOR(x, dimi * FB_NV) {
      const int r = x / FB_NV, c = x - r * FB_NV;
      L.Phix[r * FB_NX + FB_NV + c] = c1 * w.PJv[x];
      L.Phia[x] = c2 * w.PJv[x];
    }
    __syncwarp();
    if (lane < FB_NV) {
      const int j = lane;
      for (int l = 0; l < dimi; ++l) lq = fma(L.Phix[l * FB_NX + j], w.xi[l], lq);
      for (int l = 0; l < dimi; ++l) lv = fma(L.Phix[l * FB_NX + FB_NV + j], w.xi[l], lv);
      for (int l = 0; l < dimi; ++l) la = fma(L.Phia[l * FB_NV + j], w.xi[l], la);
    }
  }
  // ---- store the stage vectors ----
  if (lane < FB_NV) { L.lq[lane] = lq; L.lv[lane] = lv; L.la[lane] = la; L.Fq[lane] = Fq; L.Fv[lane] = Fv; }
  if (lane < FB_MAXF) L.lf[lane] = lane < dimf ? lf : 0.0;
  if (lane < FB_NU) L.lu[lane] = lu;
  if (lane < FB_NPASS) L.lu_passive[lane] = lup;
  __syncwarp();

  if (RESIDUAL_ONLY) {
    // squaredNormKKTResidual (split_ocp.hxx:263-279, impulse_split_ocp.hxx:131-142): partial sums by seven lanes,
    // added in the reference's order
    if (lane == 0) w.part[0] = fb_sqnorm(L.lq, FB_NV) + fb_sqnorm(L.lv, FB_NV);
    if (lane == 1) w.part[1] = fb_sqnorm(L.la, FB_NV);
    if (lane == 2) w.part[2] = fb_sqnorm(L.lf, dimf);
    if (lane == 3) { w.part[3] = fb_sqnorm(L.lu_passive, FB_NPASS); w.part[7] = fb_sqnorm(L.lu, FB_NU); }
    if (lane == 4) w.part[4] = fb_sqnorm(L.Fq, FB_NV) + fb_sqnorm(L.Fv, FB_NV);
    if (lane == 5) w.part[5] = fb_sqnorm(L.IDC, nvf);
    {
      // rows of FbDir (L2): the lanes fetch 32 rows at a time and hand them round, every lane running the serial chain
      // sum_c (|residual_c|^2 + |duality_c|^2) of the reference in its order (dead rows: 0)
      double e2 = 0.0;
      for (int c = 0; c < FBC_NCOMP; ++c) {
        if (!el.cactive[c]) continue;
        const int o = fbc_offset(c), n = fbc_dim(c);
        double part2[2];
        for (int h = 0; h < 2; ++h) {
          const double* rows = (h ? Dr.duality : Dr.residual) + o;
          double acc = 0.0;
          for (int base = 0; base < n; base += 32) {
            const double mine = base + lane < n ? rows[base + lane] : 0.0;
            const int m = n - base < 32 ? n - base : 32;
            for (int t = 0; t < m; ++t) {
              const double x = __shfl_sync(0xffffffffu, mine, t);
              acc = fma(x, x, acc);
            }
          }
          part2[h] = acc;
        }
        e2 += part2[0] + part2[1];
      }
      if (lane == 6) w.part[6] = e2;
    }
    __syncwarp();
    if (lane == 0) {
      double e2 = 0.0;
      e2 += w.part[0];
      e2 += w.part[1];
      e2 += w.part[2];
      if (!impulse) { e2 += w.part[3]; e2 += w.part[7]; }
      e2 += w.part[4];
      if (!impulse) {
        e2 += dt * dt * w.part[5];
        e2 += dt * dt * w.part[6];
        e2 += fb_sqnorm(L.P, dimi);
      } else {
        e2 += w.part[5];
        e2 += w.part[6];
      }
      Dr.kkt_sq = e2;
    }
  }
}

// =====================================================================================================
// K1b: dense condensing of one stage, one CTA (128 threads) per (instance, stage)
//   computeMJtJinv (robot.hxx:576-615), condenseContactDynamics (contact_dynamics.hxx:105-158) /
//   condenseImpulseDynamics (impulse_dynamics_forward_euler.hxx:64-105), condenseSwitchingConstraint (:194-200).
//   Results go straight to the HBM records of the Riccati sweep (FbKKT) and of the expansion (FbExp).
// =====================================================================================================
struct FbDenseWork {
  // IDC and dIDCdqv as FbLin holds them (one load).  dIDCdqv is dead once MJ_dIDC = MJtJinv dIDCdqv exists; Qafqv, formed from
  // MJ_dIDC right after, takes its place
  double IDC[FB_NVF];
  union { double dIDCdqv[FB_NVF * FB_NX]; double Qafqv[FB_NVF * FB_NX]; };
  // FbLin from dCda to Fqq_prev_inv, same order
  double dCda[FB_MAXF * FB_NV];
  double lq[FB_NV], lv[FB_NV], la[FB_NV], lf[FB_MAXF], lu_passive[FB_NPASS], lu[FB_NU], Fq[FB_NV], Fv[FB_NV], P[FB_MAXF];
  double Qqq6[36], Qqq_d[FB_NV], Qvv_d[FB_NV], Quu_d[FB_NU], Qaa[FB_NV], Qff[FB_MAXF * FB_MAXF];
  double Fqq6[36], Fqv6[36], Fqq_prev_inv[36];
  // MJtJinv, MJ_dIDC, MJ_IDC: same order as FbExp.  The joint-space inertia matrix, its inverse and J M^-1 are dead once
  // MJtJinv is formed (before MJ_dIDC is) and share its storage.  Phix / Phia of the switching stages stay in HBM.
  double MJtJinv[FB_NVF * FB_NVF];
  union {
    struct { double MJ_dIDC[FB_NVF * FB_NX], MJ_IDC[FB_NVF]; };
    struct { double Mm[FB_NV * FB_NV], Minv[FB_NV * FB_NV], JMi[FB_MAXF * FB_NV], Sm[FB_MAXF * FB_MAXF]; };
  };
  double laf[FB_NVF];
  union {
    struct { double L[FB_NV * FB_NV], rd[FB_NV], Ls[FB_MAXF * FB_MAXF], rds[FB_MAXF], Si[FB_MAXF * FB_MAXF]; int fail[FB_NV + 2]; } f;   // factorisation scratch
    double Qafu[FB_NVF * FB_NV];                                                                                                        // condensing product
  } s;
  int info;
};
// 36 KB: six CTAs share the 228 KB of an SM (43.8 KB, five CTAs, with Qafqv and M^-1 / J M^-1 in storage of their own)
static_assert(6 * (sizeof(FbDenseWork) + 1024) <= 228 * 1024, "six CTAs of k_fb_condense per SM");

constexpr int FB_DENSE_MINB = 6;
static_assert(FB_MAXF * FB_NV + FB_MAXF * FB_MAXF >= FB_NV * (FB_NV + 1), "the JMi / Sm scratch holds the 18 x 19 trailing matrix of LLT(M)");
__global__ void __launch_bounds__(128, FB_DENSE_MINB) k_fb_condense(FbArrays A, const FbLin* lin) {
  IDOCP_DYN_SMEM(FbDenseWork, wp);
  FbDenseWork& w = *wp;
  const int tid = threadIdx.x;
  const int b = blockIdx.x / A.n_elems, e = blockIdx.x - b * A.n_elems;
  const FbElem& el = A.elems[e];
  const size_t rec = (size_t)el.slot * A.B + b;
  FbKKT& Kt = A.kkt[rec];
  const FbLin& L = lin[rec];
  const int NV = FB_NV, NX = FB_NX, NU = FB_NU, NVF = FB_NVF, NPASS = FB_NPASS, MAXF = FB_MAXF;
  if (el.kind == FB_TERMINAL) {
    // the terminal stage has no dynamics: Qxx = cost Hessian, lx
    FB_FOR(x, NX * NX) {
      const int r = x / NX, c = x - r * NX;
      double v = 0.0;
      if (r < 6 && c < 6) v = L.Qqq6[6 * r + c];
      else if (r == c) v = r < NV ? L.Qqq_d[r] : L.Qvv_d[r - NV];
      Kt.Qxx[x] = v;
    }
    fb_copy(Kt.Fqq_prev_inv, L.Fqq_prev_inv, 36);
    fb_copy(Kt.lq, L.lq, NV);
    fb_copy(Kt.lv, L.lv, NV);
    return;
  }
  const bool impulse = el.kind == FB_IMPULSE;
  const double dt = impulse ? 1.0 : el.dt;
  const int dimf = el.dimf, nvf = NV + dimf, dimi = el.sw ? el.dimi : 0;
  FbExp& Ex = A.exp[rec];
  FbDir& Dr = A.dir[rec];
  fb_load<FB_NVF + FB_NVF * FB_NX>(w.IDC, L.IDC);
  fb_load<FB_NV * FB_NV>(w.Mm, L.Mm);
  fb_load<(offsetof(FbLin, Phix) - offsetof(FbLin, dCda)) / sizeof(double)>(w.dCda, L.dCda);
  if (tid == 0) w.info = 0;
  __syncthreads();
  // ---- MJtJinv = [[M, J^T], [J, 0]]^-1 by dense Cholesky ----
  {
    const int n = NV, ld = NVF;
    // Minv = M^-1 by the whole CTA (owner-per-element sweep, fb_llt_factor_solve_cta).  Two one-warp forms were measured
    // and are slower for this 18 x 18 inverse: fully unrolled in registers (warp_llt.cuh) 47 k cycles, rolled loops over
    // shared memory (fb_inverse_warp) 44 k, against 28 k here (profiles/r2j / r2k_fb_phase_clocks.json): one warp per CTA
    // leaves the SM with five active warps
    // (the dense owner-per-element sweep fb_llt_factor_solve_cta<2, 3> took 36 barrier steps: 28 k of the 74 k cycles per stage)
    fb_minv_tree_cta(w.Mm, w.s.f.L, w.s.f.rd, w.Minv, w.s.f.fail, &w.info, 0);
    fb_mm<FBM_SET>(dimf, n, n, w.dCda, n, 1, w.Minv, n, 1, w.JMi, n);
    __syncthreads();
    fb_mm<FBM_SET>(dimf, dimf, n, w.JMi, n, 1, w.dCda, 1, n, w.Sm, dimf);
    __syncthreads();
    if (dimf > 0) {
      FB_FOR(x, dimf * dimf) { const int r = x / dimf; w.s.f.Si[x] = (x - r * dimf == r) ? 1.0 : 0.0; }
      __syncthreads();
      fb_llt_factor_solve_cta<1, 2>(w.Sm, dimf, dimf, w.s.f.Ls, dimf, w.s.f.rds, w.s.f.Si, dimf, dimf, &w.info, 100);
    }
    FB_FOR(x, dimf * dimf) { const int r = x / dimf, c = x - r * dimf; w.MJtJinv[(n + r) * ld + n + c] = -w.s.f.Si[x]; }
    fb_mm<FBM_SET>(n, dimf, dimf, w.JMi, 1, n, w.s.f.Si, dimf, 1, w.MJtJinv + n, ld);     // TR = (J Minv)^T S^-1
    __syncthreads();
    {                                                                                           // TL = Minv - TR (J Minv)
      const double* Minv = w.Minv;
      double* TL = w.MJtJinv;
      fb_mm_f<FBM_SUB>(n, n, dimf, w.MJtJinv + n, ld, 1, w.JMi, n, 1, [=](int r, int c) { return Minv[r * n + c]; },
                       [=](int r, int c, double v) { TL[r * ld + c] = v; });
    }
    FB_FOR(x, dimf * n) { const int r = x / n, c = x - r * n; w.MJtJinv[(n + r) * ld + c] = w.MJtJinv[c * ld + n + r]; }   // BL = TR^T
    __syncthreads();
  }
  // ---- condensing ----
  fb_mm<FBM_SET>(nvf, NX, nvf, w.MJtJinv, NVF, 1, w.dIDCdqv, NX, 1, w.MJ_dIDC, NX);
  fb_mv<FBM_SET>(nvf, nvf, w.MJtJinv, NVF, 1, w.IDC, w.MJ_IDC);
  __syncthreads();
  double* Qafqv = w.Qafqv;
  double* Qafu = w.s.Qafu;
  FB_FOR(x, NV * NX) { const int r = x / NX; Qafqv[x] = -w.Qaa[r] * w.MJ_dIDC[x]; }
  fb_mm<FBM_SET>(dimf, NX, dimf, w.Qff, MAXF, 1, w.MJ_dIDC + NV * NX, NX, 1, Qafqv + NV * NX, NX);
  if (!impulse) {
    FB_FOR(x, NV * NV) { const int r = x / NV, c = x - r * NV; Qafu[x] = w.Qaa[r] * w.MJtJinv[r * NVF + c]; }
    fb_mm<FBM_SET>(dimf, NV, dimf, w.Qff, MAXF, 1, w.MJtJinv + NV * NVF, NVF, 1, Qafu + NV * NV, NV);
  }
  if (tid < NV) w.laf[tid] = fma(-w.Qaa[tid], w.MJ_IDC[tid], w.la[tid]);
  if (tid >= 32 && tid < 32 + dimf) w.laf[NV + tid - 32] = -w.lf[tid - 32];
  __syncthreads();
  FB_FOR(x, dimf * NX) Qafqv[NV * NX + x] = -Qafqv[NV * NX + x];
  fb_mv<FBM_SUB>(dimf, dimf, w.Qff, MAXF, 1, w.MJ_IDC + NV, w.laf + NV);
  __syncthreads();
  // Qxx -= MJ_dIDC^T Qafqv, starting from the sparse cost / constraint Hessian; the Qvq block is never read
  // (the Riccati sweep rebuilds it from Qqv, backward_riccati_recursion_factorizer.hxx:93) and is left untouched
  int rot = 0;   // tile rotation across the independent products below (fb_mm_f)
  {
    const double *Qqq6 = w.Qqq6, *Qqq_d = w.Qqq_d, *Qvv_d = w.Qvv_d;
    double* Qxx = Kt.Qxx;
    fb_mm_f<FBM_SUB>(NX, NX, nvf, w.MJ_dIDC, 1, NX, Qafqv, NX, 1,
                     [=](int r, int c) {
                       if (r < 6 && c < 6) return Qqq6[6 * r + c];
                       if (r == c) return r < NV ? Qqq_d[r] : Qvv_d[r - NV];
                       return 0.0;
                     },
                     [=](int r, int c, double v) { if (!(r >= NV && c < NV)) Qxx[r * NX + c] = v; }, &rot);
  }
  if (tid < NV) {
    double acc = w.lq[tid];
    for (int l = 0; l < nvf; ++l) acc = fma(-w.MJ_dIDC[l * NX + tid], w.laf[l], acc);
    Kt.lq[tid] = acc;
  } else if (tid >= 32 && tid < 32 + NV) {
    const int j = tid - 32;
    double acc = w.lv[j];
    for (int l = 0; l < nvf; ++l) acc = fma(-w.MJ_dIDC[l * NX + NV + j], w.laf[l], acc);
    Kt.lv[j] = acc;
  }
  if (!impulse) {
    {
      const double* Quu_d = w.Quu_d;
      double *Qxu = Kt.Qxu, *Quu = Kt.Quu;
      fb_mm_f<FBM_SUB>(NX, NV, nvf, w.MJ_dIDC, 1, NX, Qafu, NV, 1, [](int, int) { return 0.0; },
                       [=](int r, int c, double v) { Qxu[r * NV + c] = v; }, &rot);
      fb_mm_f<FBM_ADD>(NV, NV, nvf, w.MJtJinv, NVF, 1, Qafu, NV, 1, [=](int r, int c) { return (r == c && r >= NPASS) ? Quu_d[r - NPASS] : 0.0; },
                       [=](int r, int c, double v) { Quu[r * NV + c] = v; }, &rot);
    }
    if (tid >= 64 && tid < 64 + NV) {
      const int j = tid - 64;
      double acc = j < NPASS ? w.lu_passive[j] : w.lu[j - NPASS];
      for (int l = 0; l < nvf; ++l) acc = fma(w.MJtJinv[j * NVF + l], w.laf[l], acc);
      if (j < NPASS) Kt.lu_passive[j] = acc; else Kt.lu[j - NPASS] = acc;
    }
    FB_FOR(x, NV * NV) {
      const int r = x / NV, c = x - r * NV;
      Kt.Fvq[x] = -dt * w.MJ_dIDC[r * NX + c];
      Kt.Fvv[x] = -dt * w.MJ_dIDC[r * NX + NV + c] + (r == c ? 1.0 : 0.0);
    }
    FB_FOR(x, NV * NU) { const int r = x / NU, c = x - r * NU; Kt.Fvu[x] = dt * w.MJtJinv[r * NVF + NPASS + c]; }
    if (tid >= 96 && tid < 96 + NV) Kt.Fv[tid - 96] = fma(-dt, w.MJ_IDC[tid - 96], w.Fv[tid - 96]);
  } else {
    FB_FOR(x, NV * NV) {
      const int r = x / NV, c = x - r * NV;
      Kt.Fvq[x] = -w.MJ_dIDC[r * NX + c];
      Kt.Fvv[x] = (r == c ? 1.0 : 0.0) - w.MJ_dIDC[r * NX + NV + c];
    }
    if (tid >= 96 && tid < 96 + NV) Kt.Fv[tid - 96] = w.Fv[tid - 96] - w.MJ_IDC[tid - 96];
  }
  fb_copy(Kt.Fq, w.Fq, NV);
  fb_copy(Kt.Fqq6, w.Fqq6, 3 * 36);   // Fqq6, Fqv6, Fqq_prev_inv
  // ---- condenseSwitchingConstraint ----
  if (dimi > 0) {
    {
      const double *Phix0 = L.Phix, *Phia = L.Phia;   // HBM operands: switching stages only
      double* Phix = Kt.Phix;
      fb_mm_f<FBM_SUB>(dimi, NX, NV, Phia, NV, 1, w.MJ_dIDC, NX, 1, [=](int r, int c) { return Phix0[r * NX + c]; },
                       [=](int r, int c, double v) { Phix[r * NX + c] = v; }, &rot);
      fb_mm<FBM_SET>(dimi, NU, NV, Phia, NV, 1, w.MJtJinv + NPASS, NVF, 1, Kt.Phiu, NU, &rot);
    }
    if (tid < dimi) {
      double acc = w.P[tid];
      for (int l = 0; l < NV; ++l) acc = fma(-L.Phia[tid * NV + l], w.MJ_IDC[l], acc);
      Kt.P[tid] = acc;
    }
  }
  // ---- expansion record ----
  fb_copy(Ex.MJtJinv, w.MJtJinv, NVF * NVF + NVF * NX + NVF);   // MJtJinv, MJ_dIDC, MJ_IDC
  fb_copy(Ex.Qafqv, Qafqv, NVF * NX);
  fb_copy(Ex.Qafu, Qafu, NVF * NV);
  fb_copy(Ex.laf, w.laf, NVF);
  if (tid == 0) Dr.info = (double)w.info;
  // ---- ContactDistance::condenseSlackAndDual (contact_distance.cpp:91-93): Qqq += (dt dual / slack) J2^T J2 per contact that
  // is not active -- the one dense term of the stage Hessian, added AFTER the condensed products (the oracle's order) so that
  // the product kernels above stay as they are; J2 and the weights come from k_fb_robot (FbLin::cdJ, cdw)
  if (!impulse && el.cactive[FBC_DISTANCE]) {
    __syncthreads();   // the qq block of Kt.Qxx was written by other threads of this CTA
    FB_FOR(x, NV * NV) {
      const int r = x / NV, c = x - r * NV;
      double v = Kt.Qxx[r * NX + c];
      for (int i = 0; i < FB_NC; ++i)
        if (!el.active[i]) v += (L.cdw[i] * L.cdJ[i * NV + r]) * L.cdJ[i * NV + c];
      Kt.Qxx[r * NX + c] = v;
    }
  }
}


// =====================================================================================================
// K2: backward Riccati recursion, one CTA per instance, serial over the chain
// (riccati_recursion_solver.cpp:48-107, split_riccati_factorizer.hxx:36-100, backward_riccati_recursion_factorizer.hxx:44-161,
//  impulse twins)
// =====================================================================================================
struct FbRicWork {
  // stage record: the blocks of FbKKT the recursion reads, Qxu / Quu reduced to their actuated columns (leading dimension NU)
  double Qxx[FB_NX * FB_NX], Qxu[FB_NX * FB_NU], Quu[FB_NU * FB_NU];
  double Fqq6[36], Fqv6[36], Fvq[FB_NV * FB_NV], Fvv[FB_NV * FB_NV], Fvu[FB_NV * FB_NU];
  double lq[FB_NV], lv[FB_NV], lu[FB_NU], Fq[FB_NV], Fv[FB_NV];
  // Phix / Phiu / P (and the cM / cm of FbRic) exist on the stage before an impulse only (one or two stages of a horizon):
  // they are operated on where they lie in HBM / L2, which keeps the CTA under 56 KB, i.e. four CTAs on an SM instead of three
  // the factorisation (same order as FbRic): on entry to a stage Pqq / Pqv / Pvv still hold the NEXT stage's P, which is dead once
  // the A^T P / B^T P products are formed, so the stage's own P is built in the same place
  double K[FB_NU * FB_NX], k[FB_NU], Pqq[FB_NV * FB_NV], Pqv[FB_NV * FB_NV], Pvv[FB_NV * FB_NV], sq[FB_NV], sv[FB_NV];
  double nsq[FB_NV], nsv[FB_NV];
  // scratch whose lifetimes do not overlap shares storage
  union {
    struct { double AtPqq[FB_NV * FB_NV], AtPqv[FB_NV * FB_NV], AtPvq[FB_NV * FB_NV], AtPvv[FB_NV * FB_NV]; };   // until sq / sv
    double KtDtM[FB_NX * FB_NX];                                                                                   // after sq / sv
  };
  union {
    struct { double BtPq[FB_NU * FB_NV], BtPv[FB_NU * FB_NV]; };   // until lu is complete
    double GK[FB_NU * FB_NX];                                      // factorizeRiccatiFactorization
  };
  double L[FB_NU * FB_NU], rd[FB_NU];
  union {
    struct { double Ginv[FB_NU * FB_NU], DGinv[FB_MAXF * FB_NU], Sm[FB_MAXF * FB_MAXF]; };   // gain computation
    double DtM[FB_NU * FB_NX];                                                               // constrained tail
  };
  double Ls[FB_MAXF * FB_MAXF], rds[FB_MAXF], SinvDGinv[FB_MAXF * FB_NU];
  int info;
};

static_assert(offsetof(FbRicWork, L) % 16 == 0, "warp_llt.cuh reads the factor two doubles at a time");
static_assert(4 * (sizeof(FbRicWork) + 1024) <= 228 * 1024, "four CTAs of the backward recursion share the 228 KB of an SM");
constexpr int FB_RIC_MINB = 4;
__global__ void __launch_bounds__(128, FB_RIC_MINB) k_fb_riccati_backward(FbArrays A) {
  IDOCP_DYN_SMEM(FbRicWork, wp);
  FbRicWork& w = *wp;
  const int tid = threadIdx.x, b = blockIdx.x, n = A.n_elems;
  const int NV = FB_NV, NX = FB_NX, NU = FB_NU, MAXF = FB_MAXF;
  // terminal stage: P = (Qqq, 0, Qvv), s = -(lq, lv)
  {
    const FbElem& el = A.elems[n - 1];
    const FbKKT& Kt = A.kkt[(size_t)el.slot * A.B + b];
    FbRic& Rc = A.ric[(size_t)el.slot * A.B + b];
    FB_FOR(x, NV * NV) {
      const int r = x / NV, c = x - r * NV;
      w.Pqq[x] = Kt.Qxx[r * NX + c];
      w.Pvv[x] = Kt.Qxx[(NV + r) * NX + NV + c];
      w.Pqv[x] = 0.0;
    }
    if (tid < NV) {
      const double a = -Kt.lq[tid], c = -Kt.lv[tid];
      w.nsq[tid] = a; w.sq[tid] = a; w.nsv[tid] = c; w.sv[tid] = c;
    }
    __syncthreads();
    fb_copy(Rc.Pqq, w.Pqq, 3 * NV * NV + 2 * NV);
  }
  for (int e = n - 2; e >= 0; --e) {
    const FbElem& el = A.elems[e];
    const bool impulse = el.kind == FB_IMPULSE;
    const double dt = el.dt;
    const int dimi = el.sw ? el.dimi : 0;
    const FbKKT& Kt = A.kkt[(size_t)el.slot * A.B + b];
    FbRic& Rc = A.ric[(size_t)el.slot * A.B + b];
    __syncthreads();
    fb_load<FB_NX * FB_NX>(w.Qxx, Kt.Qxx);
    fb_load_f<FB_NX * FB_NU>(w.Qxu, Kt.Qxu, [](int x) { const int r = x / FB_NU; return r * FB_NV + FB_NPASS + (x - r * FB_NU); });
    fb_load_f<FB_NU * FB_NU>(w.Quu, Kt.Quu, [](int x) { const int r = x / FB_NU; return (FB_NPASS + r) * FB_NV + FB_NPASS + (x - r * FB_NU); });
    fb_load<72>(w.Fqq6, Kt.Fqq6);
    fb_load<2 * FB_NV * FB_NV + FB_NV * FB_NU>(w.Fvq, Kt.Fvq);
    fb_load<2 * FB_NV + FB_NU>(w.lq, Kt.lq);
    fb_load<2 * FB_NV>(w.Fq, Kt.Fq);
    const double* const Phix = Kt.Phix;
    const double* const Phiu = Kt.Phiu;
    const double* const Pc = Kt.P;
    double* const cM = Rc.cM;
    double* const cm = Rc.cm;
    // the record of the stage before this one is needed ~40 k cycles from now: bring it into the L2 meanwhile
    if (e > 0) fb_prefetch_l2(&A.kkt[(size_t)A.elems[e - 1].slot * A.B + b], (int)sizeof(FbKKT));
    if (tid == 0) w.info = 0;
    __syncthreads();
    double* Qqq = w.Qxx;
    double* Qqv = w.Qxx + NV;
    double* Qvv = w.Qxx + NV * NX + NV;
    // ---- factorizeKKTMatrix ----
    fb_mm<FBM_SET>(6, NV, 6, w.Fqq6, 1, 6, w.Pqq, NV, 1, w.AtPqq, NV);
    fb_mm<FBM_SET>(6, NV, 6, w.Fqq6, 1, 6, w.Pqv, NV, 1, w.AtPqv, NV);
    FB_FOR(x, (NV - 6) * NV) { w.AtPqq[6 * NV + x] = w.Pqq[6 * NV + x]; w.AtPqv[6 * NV + x] = w.Pqv[6 * NV + x]; }
    if (!impulse) {
      fb_mm<FBM_SET>(6, NV, 6, w.Fqv6, 1, 6, w.Pqq, NV, 1, w.AtPvq, NV);
      fb_mm<FBM_SET>(6, NV, 6, w.Fqv6, 1, 6, w.Pqv, NV, 1, w.AtPvv, NV);
      FB_FOR(x, (NV - 6) * NV) { w.AtPvq[6 * NV + x] = dt * w.Pqq[6 * NV + x]; w.AtPvv[6 * NV + x] = dt * w.Pqv[6 * NV + x]; }
    }
    __syncthreads();
    fb_mm<FBM_ADD>(NV, NV, NV, w.Fvq, 1, NV, w.Pqv, 1, NV, w.AtPqq, NV);
    fb_mm<FBM_ADD>(NV, NV, NV, w.Fvq, 1, NV, w.Pvv, NV, 1, w.AtPqv, NV);
    if (!impulse) {
      fb_mm<FBM_ADD>(NV, NV, NV, w.Fvv, 1, NV, w.Pqv, 1, NV, w.AtPvq, NV);
      fb_mm<FBM_ADD>(NV, NV, NV, w.Fvv, 1, NV, w.Pvv, NV, 1, w.AtPvv, NV);
      fb_mm<FBM_SET>(NU, NV, NV, w.Fvu, 1, NU, w.Pqv, 1, NV, w.BtPq, NV);
      fb_mm<FBM_SET>(NU, NV, NV, w.Fvu, 1, NU, w.Pvv, NV, 1, w.BtPv, NV);
    } else {
      fb_mm<FBM_SET>(NV, NV, NV, w.Fvv, 1, NV, w.Pqv, 1, NV, w.AtPvq, NV);
      fb_mm<FBM_SET>(NV, NV, NV, w.Fvv, 1, NV, w.Pvv, NV, 1, w.AtPvv, NV);
    }
    __syncthreads();
    // Factorize F: the three blocks are independent of each other, each gets its terms in the reference's order
    fb_mm<FBM_ADD>(NV, 6, 6, w.AtPqq, NV, 1, w.Fqq6, 6, 1, Qqq, NX);
    FB_FOR(x, NV * (NV - 6)) { const int r = x / (NV - 6), c = 6 + x - r * (NV - 6); Qqq[r * NX + c] += w.AtPqq[r * NV + c]; }
    if (!impulse) {
      fb_mm<FBM_ADD>(NV, 6, 6, w.AtPqq, NV, 1, w.Fqv6, 6, 1, Qqv, NX);
      FB_FOR(x, NV * (NV - 6)) { const int r = x / (NV - 6), c = 6 + x - r * (NV - 6); Qqv[r * NX + c] = fma(dt, w.AtPqq[r * NV + c], Qqv[r * NX + c]); }
      fb_mm<FBM_ADD>(NV, 6, 6, w.AtPvq, NV, 1, w.Fqv6, 6, 1, Qvv, NX);
      FB_FOR(x, NV * (NV - 6)) { const int r = x / (NV - 6), c = 6 + x - r * (NV - 6); Qvv[r * NX + c] = fma(dt, w.AtPvq[r * NV + c], Qvv[r * NX + c]); }
    }
    __syncthreads();
    fb_mm<FBM_ADD>(NV, NV, NV, w.AtPqv, NV, 1, w.Fvq, NV, 1, Qqq, NX);
    fb_mm<FBM_ADD>(NV, NV, NV, w.AtPqv, NV, 1, w.Fvv, NV, 1, Qqv, NX);
    fb_mm<FBM_ADD>(NV, NV, NV, w.AtPvv, NV, 1, w.Fvv, NV, 1, Qvv, NX);
    if (!impulse) {
      fb_mm<FBM_ADD>(NV, NU, NV, w.AtPqv, NV, 1, w.Fvu, NU, 1, w.Qxu, NU);
      fb_mm<FBM_ADD>(NV, NU, NV, w.AtPvv, NV, 1, w.Fvu, NU, 1, w.Qxu + NV * NU, NU);
      fb_mm<FBM_ADD>(NU, NU, NV, w.BtPv, NV, 1, w.Fvu, NU, 1, w.Quu, NU);
      if (tid < NU) {    // lu += BtPq Fq; lu += BtPv Fv; lu -= Fvu^T sv_next
        double acc = w.lu[tid];
        for (int l = 0; l < NV; ++l) acc = fma(w.BtPq[tid * NV + l], w.Fq[l], acc);
        for (int l = 0; l < NV; ++l) acc = fma(w.BtPv[tid * NV + l], w.Fv[l], acc);
        for (int l = 0; l < NV; ++l) acc = fma(-w.Fvu[l * NU + tid], w.nsv[l], acc);
        w.lu[tid] = acc;
      }
    }
    __syncthreads();
    const double* Qxu = w.Qxu;   // 36 x 12, leading dimension NU
    if (!impulse) {
      // LLT(G), G = Quu (12 x 12), factor only: warp 0, lane = row, rows in registers (warp_llt.cuh).  Measured on the whole
      // kernel: 6.70 ms CTA-wide (fb_llt_cta), 6.05 ms this form, 7.28 ms the rolled one-warp loop (fb_llt_warp)
      if (tid < 32) {
        const int row = tid < NU ? tid : NU - 1;
        double a[FB_NU];
#pragma unroll
        for (int c = 0; c < FB_NU; ++c) a[c] = w.Quu[row * NU + (c <= row ? c : row)];
        __syncwarp();
        const int fail = warp_llt_rows<FB_NU, FB_NU>(a, w.L, nullptr, w.rd, tid);
        if (fail && tid == 0 && w.info == 0) w.info = 200 + fail;
      }
      __syncthreads();
      if (dimi == 0) {
        // K = -G^-1 Qxu^T, k = -G^-1 lu: one right-hand side per thread
        if (tid < NX) {
          double col[FB_NU];
          for (int r = 0; r < NU; ++r) col[r] = Qxu[tid * NU + r];
          fb_llt_solve_n<FB_NU>(w.L, NU, w.rd, col, 1);
          for (int r = 0; r < NU; ++r) w.K[r * NX + tid] = -col[r];
        } else if (tid == NX) {
          double col[FB_NU];
          for (int r = 0; r < NU; ++r) col[r] = w.lu[r];
          fb_llt_solve_n<FB_NU>(w.L, NU, w.rd, col, 1);
          for (int r = 0; r < NU; ++r) w.k[r] = -col[r];
        }
        __syncthreads();
      } else {
        // Schur complement on the switching constraint (split_riccati_factorizer.hxx:55-100)
        if (tid < NU) {
          for (int r = 0; r < NU; ++r) w.Ginv[r * NU + tid] = (r == tid) ? 1.0 : 0.0;
          fb_llt_solve_n<FB_NU>(w.L, NU, w.rd, w.Ginv + tid, NU);
        } else if (tid >= 32 && tid < 32 + dimi) {
          const int r = tid - 32;
          for (int c = 0; c < NU; ++c) w.DGinv[r * NU + c] = Phiu[r * NU + c];
          fb_llt_solve_n<FB_NU>(w.L, NU, w.rd, w.DGinv + r * NU, 1);
        }
        __syncthreads();
        fb_mm<FBM_SET>(dimi, dimi, NU, w.DGinv, NU, 1, Phiu, 1, NU, w.Sm, MAXF);
        __syncthreads();
        fb_llt_cta<1>(w.Sm, MAXF, dimi, w.Ls, MAXF, w.rds, &w.info, 300);
        if (tid < NU) {
          for (int r = 0; r < dimi; ++r) w.SinvDGinv[r * NU + tid] = w.DGinv[r * NU + tid];
          fb_llt_solve(w.Ls, MAXF, w.rds, dimi, w.SinvDGinv + tid, NU);
        }
        __syncthreads();
        fb_mm<FBM_SUB>(NU, NU, dimi, w.SinvDGinv, 1, NU, w.DGinv, NU, 1, w.Ginv, NU);
        __syncthreads();
        fb_mm<FBM_SET>(NU, NX, NU, w.Ginv, NU, 1, Qxu, 1, NU, w.K, NX);
        fb_mv<FBM_SET>(NU, NU, w.Ginv, NU, 1, w.lu, w.k);
        __syncthreads();
        FB_FOR(x, NU * NX) w.K[x] = -w.K[x];
        if (tid < NU) w.k[tid] = -w.k[tid];
        __syncthreads();
        fb_mm<FBM_SUB>(NU, NX, dimi, w.SinvDGinv, 1, NU, Phix, NX, 1, w.K, NX);
        fb_mv<FBM_SUB>(NU, dimi, w.SinvDGinv, 1, NU, Pc, w.k);
        if (tid >= 64 && tid < 64 + NX) {
          const int c = tid - 64;
          for (int r = 0; r < dimi; ++r) cM[r * NX + c] = Phix[r * NX + c];
          fb_llt_solve(w.Ls, MAXF, w.rds, dimi, cM + c, NX);
        } else if (tid == 127) {
          for (int r = 0; r < dimi; ++r) cm[r] = Pc[r];
          fb_llt_solve(w.Ls, MAXF, w.rds, dimi, cm, 1);
        }
        __syncthreads();
        fb_mm<FBM_SUB>(dimi, NX, NU, w.SinvDGinv, NU, 1, Qxu, 1, NU, cM, NX);
        fb_mv<FBM_SUB>(dimi, NU, w.SinvDGinv, NU, 1, w.lu, cm);
        __syncthreads();
      }
    }
    // ---- factorizeRiccatiFactorization ----
    FB_FOR(x, NV * NV) {
      const int r = x / NV, c = x - r * NV;
      w.Pqq[x] = Qqq[r * NX + c];
      w.Pqv[x] = Qqv[r * NX + c];
      w.Pvv[x] = Qvv[r * NX + c];
    }
    if (!impulse) fb_mm<FBM_SET>(NU, NX, NU, w.Quu, NU, 1, w.K, NX, 1, w.GK, NX);
    __syncthreads();
    if (!impulse) {
      fb_mm<FBM_SUB>(NV, NV, NU, w.K, 1, NX, w.GK, NX, 1, w.Pqq, NV);
      fb_mm<FBM_SUB>(NV, NV, NU, w.K, 1, NX, w.GK + NV, NX, 1, w.Pqv, NV);
      fb_mm<FBM_SUB>(NV, NV, NU, w.K + NV, 1, NX, w.GK + NV, NX, 1, w.Pvv, NV);
      __syncthreads();
    }
    FB_FOR(x, NV * NV) {   // preserve the symmetry: one thread per unordered pair
      const int r = x / NV, c = x - r * NV;
      if (c >= r) {
        const double a = 0.5 * (w.Pqq[r * NV + c] + w.Pqq[c * NV + r]);
        const double bb = 0.5 * (w.Pvv[r * NV + c] + w.Pvv[c * NV + r]);
        w.Pqq[r * NV + c] = a; w.Pqq[c * NV + r] = a;
        w.Pvv[r * NV + c] = bb; w.Pvv[c * NV + r] = bb;
      }
    }
    if (tid >= 64 && tid < 64 + NV) {   // sq
      const int j = tid - 64;
      double acc;
      if (j < 6) {
        acc = w.Fqq6[j] * w.nsq[0];
        for (int l = 1; l < 6; ++l) acc = fma(w.Fqq6[6 * l + j], w.nsq[l], acc);
      } else {
        acc = w.nsq[j];
      }
      for (int l = 0; l < NV; ++l) acc = fma(w.Fvq[l * NV + j], w.nsv[l], acc);
      for (int l = 0; l < NV; ++l) acc = fma(-w.AtPqq[j * NV + l], w.Fq[l], acc);
      for (int l = 0; l < NV; ++l) acc = fma(-w.AtPqv[j * NV + l], w.Fv[l], acc);
      acc -= w.lq[j];
      if (!impulse)
        for (int l = 0; l < NU; ++l) acc = fma(-w.Qxu[j * NU + l], w.k[l], acc);
      w.sq[j] = acc;
    }
    if (tid >= 96 && tid < 96 + NV) {   // sv
      const int j = tid - 96;
      double acc;
      if (!impulse) {
        if (j < 6) {
          acc = w.Fqv6[j] * w.nsq[0];
          for (int l = 1; l < 6; ++l) acc = fma(w.Fqv6[6 * l + j], w.nsq[l], acc);
        } else {
          acc = dt * w.nsq[j];
        }
        for (int l = 0; l < NV; ++l) acc = fma(w.Fvv[l * NV + j], w.nsv[l], acc);
      } else {
        acc = w.Fvv[j] * w.nsv[0];
        for (int l = 1; l < NV; ++l) acc = fma(w.Fvv[l * NV + j], w.nsv[l], acc);
      }
      for (int l = 0; l < NV; ++l) acc = fma(-w.AtPvq[j * NV + l], w.Fq[l], acc);
      for (int l = 0; l < NV; ++l) acc = fma(-w.AtPvv[j * NV + l], w.Fv[l], acc);
      acc -= w.lv[j];
      if (!impulse)
        for (int l = 0; l < NU; ++l) acc = fma(-w.Qxu[(NV + j) * NU + l], w.k[l], acc);
      w.sv[j] = acc;
    }
    __syncthreads();
    if (dimi > 0) {
      fb_mm<FBM_SET>(NU, NX, dimi, Phiu, 1, NU, cM, NX, 1, w.DtM, NX);
      __syncthreads();
      fb_mm<FBM_SET>(NX, NX, NU, w.K, 1, NX, w.DtM, NX, 1, w.KtDtM, NX);
      __syncthreads();
      FB_FOR(x, NV * NV) {
        const int r = x / NV, c = x - r * NV;
        w.Pqq[x] = (w.Pqq[x] - w.KtDtM[r * NX + c]) - w.KtDtM[c * NX + r];
        w.Pqv[x] = (w.Pqv[x] - w.KtDtM[r * NX + NV + c]) - w.KtDtM[(NV + c) * NX + r];
        w.Pvv[x] = (w.Pvv[x] - w.KtDtM[(NV + r) * NX + NV + c]) - w.KtDtM[(NV + c) * NX + NV + r];
      }
      fb_mv<FBM_SUB>(NV, dimi, Phix, 1, NX, cm, w.sq);
      fb_mv<FBM_SUB>(NV, dimi, Phix + NV, 1, NX, cm, w.sv);
      __syncthreads();
    }
    // store the factorisation; it stays in place as the "next" one
    fb_copy(Rc.K, w.K, (int)(offsetof(FbRic, cM) / sizeof(double)));
    if (tid < NV) { w.nsq[tid] = w.sq[tid]; w.nsv[tid] = w.sv[tid]; }
    if (tid == 0 && w.info) {
      FbDir& Dr = A.dir[(size_t)el.slot * A.B + b];
      if (Dr.info == 0.0) Dr.info = (double)w.info;
    }
  }
}

// =====================================================================================================
// K3: initial state direction + forward Riccati recursion (riccati_recursion_solver.cpp:110-162), one CTA
// (64 threads) per instance
// =====================================================================================================
__global__ void __launch_bounds__(64) k_fb_riccati_forward(FbArrays A) {
  __shared__ double dq[FB_NV], dv[FB_NV], du[FB_NU], nq[FB_NV], nvv[FB_NV], t6[6];
  const int tid = threadIdx.x, b = blockIdx.x, n = A.n_elems;
  const int NV = FB_NV, NX = FB_NX, NU = FB_NU;
  {
    const FbElem& el = A.elems[0];
    const FbSol& S = A.sol[(size_t)el.slot * A.B + b];
    const FbKKT& Kt = A.kkt[(size_t)el.slot * A.B + b];
    if (tid == 0) fb_subtract(A.q0 + (size_t)b * FB_NQ, S.q, dq);
    if (tid >= 32 && tid < 32 + NV) dv[tid - 32] = A.v0[(size_t)b * NV + tid - 32] - S.v[tid - 32];
    __syncthreads();
    if (tid < 6) {
      double acc = Kt.Fqq_prev_inv[6 * tid] * dq[0];
      for (int l = 1; l < 6; ++l) acc = fma(Kt.Fqq_prev_inv[6 * tid + l], dq[l], acc);
      t6[tid] = -acc;
    }
    __syncthreads();
    if (tid < 6) dq[tid] = t6[tid];
    __syncthreads();
  }
  for (int e = 0; e < n; ++e) {
    const FbElem& el = A.elems[e];
    const bool impulse = el.kind == FB_IMPULSE;
    FbDir& Dr = A.dir[(size_t)el.slot * A.B + b];
    if (tid < NV) { Dr.dq[tid] = dq[tid]; Dr.dv[tid] = dv[tid]; }
    if (el.kind == FB_TERMINAL) break;
    const FbKKT& Kt = A.kkt[(size_t)el.slot * A.B + b];
    const FbRic& Rc = A.ric[(size_t)el.slot * A.B + b];
    const double dt = el.dt;
    if (e + 1 < n && A.elems[e + 1].kind != FB_TERMINAL) {   // the serial chain pays the DRAM latency of every stage otherwise
      const size_t nrec = (size_t)A.elems[e + 1].slot * A.B + b;
      fb_prefetch_l2(A.ric[nrec].K, (NU * NX + NU) * (int)sizeof(double));
      fb_prefetch_l2(A.kkt[nrec].Fqq6, (int)(offsetof(FbKKT, Phix) - offsetof(FbKKT, Fqq6)));
    }
    if (!impulse) {
      if (tid < NU) {
        double acc = Rc.K[tid * NX] * dq[0];
        for (int l = 1; l < NV; ++l) acc = fma(Rc.K[tid * NX + l], dq[l], acc);
        for (int l = 0; l < NV; ++l) acc = fma(Rc.K[tid * NX + NV + l], dv[l], acc);
        acc += Rc.k[tid];
        du[tid] = acc;
        Dr.du[tid] = acc;
      }
      __syncthreads();
    }
    if (tid < NV) {
      const int j = tid;
      double acc = Kt.Fq[j];
      if (j < 6) {
        for (int l = 0; l < 6; ++l) acc = fma(Kt.Fqq6[6 * j + l], dq[l], acc);
        if (!impulse)
          for (int l = 0; l < 6; ++l) acc = fma(Kt.Fqv6[6 * j + l], dv[l], acc);
      } else {
        acc += dq[j];
        if (!impulse) acc = fma(dt, dv[j], acc);
      }
      nq[j] = acc;
    } else if (tid >= 32 && tid < 32 + NV) {
      const int j = tid - 32;
      double acc = Kt.Fv[j];
      for (int l = 0; l < NV; ++l) acc = fma(Kt.Fvq[j * NV + l], dq[l], acc);
      for (int l = 0; l < NV; ++l) acc = fma(Kt.Fvv[j * NV + l], dv[l], acc);
      if (!impulse)
        for (int l = 0; l < NU; ++l) acc = fma(Kt.Fvu[j * NU + l], du[l], acc);
      nvv[j] = acc;
    }
    __syncthreads();
    if (tid < NV) { dq[tid] = nq[tid]; dv[tid] = nvv[tid]; }
    __syncthreads();
  }
}

// =====================================================================================================
// K4: expansion of one stage (riccati_recursion_solver.cpp:165-241): costate direction, condensed primal
// direction, slack / dual directions, multiplier of the switching constraint, fraction-to-boundary steps.
// grid = B * n_elems, 64 threads.
// =====================================================================================================
__device__ inline double fb_fraction_to_boundary(double rate, int nn, const double* vec, const double* dvec) {
  double mn = 1.0;
  for (int i = 0; i < nn; ++i) mn = pdipm_fraction_row(rate, vec[i], dvec[i], mn);
  return mn;
}

// no minimum CTAs per SM: 38 registers; a cap at 24 CTAs per SM (40 registers) measured 2 % slower (r2zzc)
__global__ void __launch_bounds__(64) k_fb_expand(FbArrays A) {
  __shared__ double dx[FB_NX], du[FB_NU], daf[FB_NVF], dslack[FB_NCON], ddual[FB_NCON], steps[2 * FBC_NCOMP];
  const int tid = threadIdx.x;
  const int b = blockIdx.x / A.n_elems, e = blockIdx.x - b * A.n_elems;
  const int NV = FB_NV, NX = FB_NX, NU = FB_NU, NVF = FB_NVF;
  const FbElem& el = A.elems[e];
  const FbDevProblem& pr = *A.prob;
  const int nl = fbc_cone_bits(pr);
  const bool impulse = el.kind == FB_IMPULSE, terminal = el.kind == FB_TERMINAL;
  const size_t rec = (size_t)el.slot * A.B + b;
  FbDir& Dr = A.dir[rec];
  const FbRic& Rc = A.ric[rec];
  const FbSol& S = A.sol[rec];
  // every thread walks its own row of P and of the expansion record below (one ascending fma chain per output): put all of the
  // CTA's DRAM requests in flight first, so that the walks find their lines in the L2
  fb_prefetch_l2(Rc.Pqq, (3 * NV * NV + 2 * NV) * (int)sizeof(double));
  if (!terminal) fb_prefetch_l2(A.exp[rec].MJtJinv, (int)offsetof(FbExp, Qafqv));
  if (tid < NV) { dx[tid] = Dr.dq[tid]; dx[NV + tid] = Dr.dv[tid]; }
  if (tid >= 32 && tid < 32 + NU) du[tid - 32] = Dr.du[tid - 32];
  __syncthreads();
  // computeCostateDirection (split_riccati_factorizer.hxx:131-139)
  if (tid < NV) {
    const int j = tid;
    double acc = Rc.Pqq[j * NV] * dx[0];
    for (int l = 1; l < NV; ++l) acc = fma(Rc.Pqq[j * NV + l], dx[l], acc);
    for (int l = 0; l < NV; ++l) acc = fma(Rc.Pqv[j * NV + l], dx[NV + l], acc);
    Dr.dlmd[j] = acc - Rc.sq[j];
  } else if (tid >= 32 && tid < 32 + NV) {
    const int j = tid - 32;
    double acc = Rc.Pqv[j] * dx[0];
    for (int l = 1; l < NV; ++l) acc = fma(Rc.Pqv[l * NV + j], dx[l], acc);
    for (int l = 0; l < NV; ++l) acc = fma(Rc.Pvv[j * NV + l], dx[NV + l], acc);
    Dr.dgmm[j] = acc - Rc.sv[j];
  }
  if (terminal) {
    if (tid == 0) { Dr.max_primal = 1.0; Dr.max_dual = 1.0; }
    return;
  }
  const FbExp& Ex = A.exp[rec];
  const int dimf = el.dimf, nvf = NV + dimf;
  // computeCondensedPrimalDirection (contact_dynamics.hxx:161-168)
  if (tid < nvf) {
    const int j = tid;
    double acc = Ex.MJ_dIDC[j * NX] * dx[0];
    for (int l = 1; l < NX; ++l) acc = fma(Ex.MJ_dIDC[j * NX + l], dx[l], acc);
    acc = -acc;
    if (!impulse)
      for (int l = 0; l < NU; ++l) acc = fma(Ex.MJtJinv[j * NVF + FB_NPASS + l], du[l], acc);
    acc -= Ex.MJ_IDC[j];
    if (j >= NV) acc = -acc;
    daf[j] = acc;
    Dr.daf[j] = acc;
  }
  if (el.sw && tid >= 32 && tid < 32 + el.dimi) {   // computeLagrangeMultiplierDirection (:142-148)
    const int j = tid - 32;
    double acc = Rc.cM[j * NX] * dx[0];
    for (int l = 1; l < NX; ++l) acc = fma(Rc.cM[j * NX + l], dx[l], acc);
    Dr.dxi[j] = acc + Rc.cm[j];
  }
  __syncthreads();
  // computeSlackAndDualDirection
  const int ncon_live = FBC_LIVE_ROWS(el.cactive);
  const int ncon = ncon_live < 136 ? ncon_live : 136;   // the four ContactDistance rows: their own loop below
  for (int idx = tid; idx < ncon; idx += blockDim.x) {
    const int c = fbc_comp(idx);
    const int j = idx - fbc_offset(c);
    double ds = 0.0, dd = 0.0;
    if (el.cactive[c] && j < fbc_rows(nl, c)) {
      if (fbc_is_cone(c)) {
        int i, ee;
        fbc_cone_row(nl, c, j, i, ee);
        ds = 1.0; dd = 1.0;
        if (el.active[i]) {
          int k = 0;
          for (int jj = 0; jj < i; ++jj) k += el.active[jj];
          const double* df = daf + NV + 3 * k;
          const double* fi = S.f + 3 * i;
          const bool nlc = fbc_cone_rows(nl, c) == 2;
          const double Jdf = fma(fb_friction_jac(pr.mu, nlc, fi, ee, 2), df[2],
                                 fma(fb_friction_jac(pr.mu, nlc, fi, ee, 1), df[1], fb_friction_jac(pr.mu, nlc, fi, ee, 0) * df[0]));
          ds = -Jdf - Dr.residual[idx];
          dd = pdipm_dual_direction(S.slack[idx], S.dual[idx], Dr.duality[idx], ds);
        }
      } else {
        const double d = c <= FBC_POS_UP ? dx[6 + j] : (c <= FBC_VEL_UP ? dx[NV + 6 + j] : (c >= FBC_ACC_LO ? daf[6 + j] : du[j]));
        ds = ((c & 1) ? -d : d) - Dr.residual[idx];
        dd = pdipm_dual_direction(S.slack[idx], S.dual[idx], Dr.duality[idx], ds);
      }
    }
    dslack[idx] = ds;
    ddual[idx] = dd;
    Dr.dslack[idx] = ds;
    Dr.ddual[idx] = dd;
  }
  if (el.cactive[FBC_DISTANCE] && tid < FB_NC) {
    // ContactDistance::computeSlackAndDualDirection (contact_distance.cpp:112-131): J2 dq - residual for the contacts that are not
    // active, (1, 1) for the others.  Kept out of the loop above, whose code (and register count) it would change for everybody.
    const int idx = fbc_offset(FBC_DISTANCE) + tid;
    double ds = 1.0, dd = 1.0;
    if (!el.active[tid]) {
      const double* J2 = A.lin[(size_t)el.slot * A.B + b].cdJ + tid * NV;
      double acc = J2[0] * dx[0];
#pragma unroll 1
      for (int l = 1; l < NV; ++l) acc = fma(J2[l], dx[l], acc);
      ds = acc - Dr.residual[idx];
      dd = pdipm_dual_direction(S.slack[idx], S.dual[idx], Dr.duality[idx], ds);
    }
    dslack[idx] = ds;
    ddual[idx] = dd;
    Dr.dslack[idx] = ds;
    Dr.ddual[idx] = dd;
  }
  __syncthreads();
  if (tid < 2 * FBC_NCOMP) {
    const int c = tid >> 1, o = fbc_offset(c);
    double r = 1.0;
    if (el.cactive[c]) r = (tid & 1) ? fb_fraction_to_boundary(pr.fraction_rate, fbc_rows(nl, c), S.dual + o, ddual + o)
                                     : fb_fraction_to_boundary(pr.fraction_rate, fbc_rows(nl, c), S.slack + o, dslack + o);
    steps[tid] = r;
  }
  __syncthreads();
  if (tid == 0) {
    double mp = 1.0, md = 1.0;
    for (int c = 0; c < FBC_NCOMP; ++c) {
      if (steps[2 * c] < mp) mp = steps[2 * c];
      if (steps[2 * c + 1] < md) md = steps[2 * c + 1];
    }
    Dr.max_primal = mp;
    Dr.max_dual = md;
  }
}

// step sizes of every instance: min over the chain (exact, order-free); one thread per instance
__global__ void k_fb_steps(FbArrays A) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= A.B) return;
  double ap = 1.0, ad = 1.0;
  for (int e = 0; e < A.n_elems; ++e) {
    const FbDir& Dr = A.dir[(size_t)A.elems[e].slot * A.B + b];
    if (Dr.max_primal < ap) ap = Dr.max_primal;
    if (Dr.max_dual < ad) ad = Dr.max_dual;
  }
  A.steps[2 * b] = ap;
  A.steps[2 * b + 1] = ad;
}

// =====================================================================================================
// K5: condensed dual direction, costate correction, update of the solution and of slack / dual
// (ocp_linearizer.cpp:140-221, contact_dynamics.hxx:171-190, state_equation.hxx:96-108, split_solution.hxx:215-239)
// grid = B * n_elems, 64 threads.  Reads dgmm of the NEXT stage, which no CTA of this kernel writes.
// =====================================================================================================
constexpr int FB_UPD_MINB = 16;   // 64 registers: 16 CTAs (32 warps) per SM; measured 1.07 -> 0.96 ms (r2zzc)
__global__ void __launch_bounds__(64, FB_UPD_MINB) k_fb_update(FbArrays A) {
  __shared__ double dx[FB_NX], du[FB_NU], laf[FB_NVF], dbetamu[FB_NVF], dgn[FB_NV], dlmd[FB_NV], qn[FB_NQ], dqs[FB_NV], qs[FB_NQ];
  const int tid = threadIdx.x;
  const int b = blockIdx.x / A.n_elems, e = blockIdx.x - b * A.n_elems;
  const int NV = FB_NV, NX = FB_NX, NU = FB_NU, NVF = FB_NVF, NPASS = FB_NPASS;
  const FbElem& el = A.elems[e];
  const bool impulse = el.kind == FB_IMPULSE, terminal = el.kind == FB_TERMINAL;
  const size_t rec = (size_t)el.slot * A.B + b;
  FbDir& Dr = A.dir[rec];
  FbSol& S = A.sol[rec];
  const FbKKT& Kt = A.kkt[rec];
  const double ap = A.steps[2 * b], ad = A.steps[2 * b + 1];
  const double dt = el.dt;
  if (!terminal) {   // the row walks below (see k_fb_expand)
    const FbExp& Ep = A.exp[rec];
    fb_prefetch_l2(Ep.MJtJinv, FB_NVF * FB_NVF * (int)sizeof(double));
    fb_prefetch_l2(Ep.Qafqv, (int)(sizeof(FbExp) - offsetof(FbExp, Qafqv)));
    if (!impulse) fb_prefetch_l2(Kt.Qxu, (FB_NX * FB_NV + FB_NPASS * FB_NV) * (int)sizeof(double));
  }
  if (tid < NV) { dx[tid] = Dr.dq[tid]; dx[NV + tid] = Dr.dv[tid]; dlmd[tid] = Dr.dlmd[tid]; dqs[tid] = Dr.dq[tid]; }
  if (tid >= 32 && tid < 32 + NU) du[tid - 32] = Dr.du[tid - 32];
  if (tid < FB_NQ) qs[tid] = S.q[tid];
  if (!terminal) {
    const FbDir& Dn = A.dir[(size_t)el.next_slot * A.B + b];
    if (tid >= 32 && tid < 32 + NV) dgn[tid - 32] = Dn.dgmm[tid - 32];
  }
  __syncthreads();
  const int dimf = terminal ? 0 : el.dimf, nvf = NV + dimf;
  if (!terminal) {
    const FbExp& Ex = A.exp[rec];
    if (!impulse && tid >= 32 && tid < 32 + NPASS) {
      const int j = tid - 32;
      const double rdt = 1.0 / dt;
      double acc = Kt.lu_passive[j];
      for (int l = 0; l < NU; ++l) acc = fma(Kt.Quu[j * NV + NPASS + l], du[l], acc);
      for (int l = 0; l < NX; ++l) acc = fma(Kt.Qxu[l * NV + j], dx[l], acc);
      double t = Ex.MJtJinv[j * NVF] * dgn[0];
      for (int l = 1; l < NV; ++l) t = fma(Ex.MJtJinv[j * NVF + l], dgn[l], t);
      Dr.dnu_passive[j] = -(fma(dt, t, acc)) * rdt;
    }
    if (tid < nvf) {
      const int j = tid;
      double acc = Ex.laf[j];
      for (int l = 0; l < NX; ++l) acc = fma(Ex.Qafqv[j * NX + l], dx[l], acc);
      if (!impulse) {
        for (int l = 0; l < NU; ++l) acc = fma(Ex.Qafu[j * NV + NPASS + l], du[l], acc);
        if (j < NV) acc = fma(dt, dgn[j], acc);
      } else {
        if (j < NV) acc += dgn[j];
      }
      laf[j] = acc;
    }
    __syncthreads();
    if (tid < nvf) {
      const int j = tid;
      double acc = Ex.MJtJinv[j * NVF] * laf[0];
      for (int l = 1; l < nvf; ++l) acc = fma(Ex.MJtJinv[j * NVF + l], laf[l], acc);
      acc = impulse ? -acc : -acc * (1.0 / dt);
      dbetamu[j] = acc;
      Dr.dbetamu[j] = acc;
    }
  }
  // correctCostateDirectionForwardEuler: dlmd[0:6] = -Fqq_prev_inv^T dlmd[0:6]
  if (tid >= 48 && tid < 54) {
    const int j = tid - 48;
    double acc = Kt.Fqq_prev_inv[j] * dlmd[0];
    for (int l = 1; l < 6; ++l) acc = fma(Kt.Fqq_prev_inv[6 * l + j], dlmd[l], acc);
    Dr.dlmd[j] = -acc;
  }
  if (tid == 63) fb_integrate(qs, dqs, ap, qn);
  __syncthreads();
  // SplitSolution::integrate
  if (tid < NV) {
    const int j = tid;
    const double dl = (j < 6) ? Dr.dlmd[j] : dlmd[j];
    S.lmd[j] = fma(ap, dl, S.lmd[j]);
    S.gmm[j] = fma(ap, Dr.dgmm[j], S.gmm[j]);
    S.v[j] = fma(ap, dx[NV + j], S.v[j]);
    if (!terminal) {
      S.a[j] = fma(ap, Dr.daf[j], S.a[j]);
      S.beta[j] = fma(ap, dbetamu[j], S.beta[j]);
    }
  }
  if (tid < FB_NQ) S.q[tid] = qn[tid];
  if (terminal) return;
  if (!impulse) {
    if (tid >= 32 && tid < 32 + NU) S.u[tid - 32] = fma(ap, du[tid - 32], S.u[tid - 32]);
    if (tid >= 48 && tid < 48 + NPASS) S.nu_passive[tid - 48] = fma(ap, Dr.dnu_passive[tid - 48], S.nu_passive[tid - 48]);
    if (el.sw && tid < el.dimi) S.xi[tid] = fma(ap, Dr.dxi[tid], S.xi[tid]);
  }
  if (tid >= 20 && tid < 20 + FB_MAXF) {
    const int x = tid - 20, i = x / 3;
    if (el.active[i]) {
      int k = 0;
      for (int j = 0; j < i; ++j) k += el.active[j];
      S.f[x] = fma(ap, Dr.daf[NV + 3 * k + x % 3], S.f[x]);
      S.mu[x] = fma(ap, dbetamu[NV + 3 * k + x % 3], S.mu[x]);
    }
  }
  const int ncon = FBC_LIVE_ROWS(el.cactive);
  for (int idx = tid; idx < ncon; idx += blockDim.x) {
    const int c = fbc_comp(idx);
    if (el.cactive[c]) {
      S.slack[idx] = fma(ap, Dr.dslack[idx], S.slack[idx]);
      S.dual[idx] = fma(ad, Dr.ddual[idx], S.dual[idx]);
    }
  }
}

// the reference's order of sums over the chain (ocp_linearizer.cpp:97-137, line_search.hpp:174-182): pass 0 the grid
// stages and the terminal stage, pass 1 impulse, pass 2 aux, pass 3 lift
__host__ __device__ inline bool fb_in_pass(int kind, int pass) {
  return (pass == 0 && (kind == FB_GRID || kind == FB_TERMINAL)) || (pass == 1 && kind == FB_IMPULSE) || (pass == 2 && kind == FB_AUX) ||
         (pass == 3 && kind == FB_LIFT);
}

// KKT error of every instance (ocp_linearizer.cpp:97-137), one thread per instance
__global__ void k_fb_kkt_sum(FbArrays A) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= A.B) return;
  double sum = 0.0;
  for (int pass = 0; pass < 4; ++pass)
    for (int e = 0; e < A.n_elems; ++e)
      if (fb_in_pass(A.elems[e].kind, pass)) sum += A.dir[(size_t)A.elems[e].slot * A.B + b].kkt_sq;
  A.kkt_err[b] = sqrt(sum);
}

// initConstraints (ocp_linearizer.cpp:40-68): Constraints::setSlackAndDual on every used slot; one thread per
// (instance, slot-table row).  rows[]: slot, kind, cactive[8]
struct FbInitRow { int slot, kind, cactive[FBC_NCOMP]; };
__global__ void k_fb_init_constraints(FbArrays A, const FbInitRow* rows, int n_rows) {
  const int g = blockIdx.x * blockDim.x + threadIdx.x;
  if (g >= A.B * n_rows) return;
  const int b = g / n_rows;
  const FbInitRow& row = rows[g - b * n_rows];
  const FbDevProblem& pr = *A.prob;
  const int nl = fbc_cone_bits(pr);
  FbSol& S = A.sol[(size_t)row.slot * A.B + b];
  for (int c = 0; c < FBC_NCOMP; ++c) {
    const int o = fbc_offset(c);
    for (int j = 0; j < fbc_dim(c); ++j) {
      double sl = 0.0, du = 0.0;
      if (c == FBC_DISTANCE && row.cactive[c]) continue;   // needs the forward kinematics: k_fb_init_distance
      if (row.cactive[c] && j < fbc_rows(nl, c)) {
        double margin;
        if (fbc_is_cone(c)) {
          int i, ee;
          fbc_cone_row(nl, c, j, i, ee);
          double r5[5];
          fb_friction_residual(pr.mu, fbc_cone_rows(nl, c) == 2, S.f + 3 * i, r5);
          margin = -r5[ee];
        } else {
          margin = fbc_box_margin(c, j, pr, S.q, S.v, S.a, S.u);
        }
        pdipm_set_slack_and_dual_positive(margin, pr.barrier, sl, du);
      }
      S.slack[o + j] = sl;
      S.dual[o + j] = du;
    }
  }
}

// ContactDistance::setSlackAndDual (contact_distance.cpp:62-70): slack = height of the contact frame of EVERY contact; needs the
// forward kinematics, hence a warp per (instance, slot-table row) with the work area of k_fb_robot
__global__ void __launch_bounds__(32 * FB_ROBOT_WARPS) k_fb_init_distance(FbArrays A, const FbInitRow* rows, int n_rows) {
  IDOCP_DYN_SMEM(FbRobotWork, wbase);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int g = blockIdx.x * FB_ROBOT_WARPS + warp;
  if (g >= A.B * n_rows) return;
  const int b = g / n_rows;
  const FbInitRow& row = rows[g - b * n_rows];
  if (!row.cactive[FBC_DISTANCE]) return;
  const FbDevProblem& pr = *A.prob;
  FbRobotWork& w = wbase[warp];
  FbSol& S = A.sol[(size_t)row.slot * A.B + b];
  if (lane < FB_NQ) w.q[lane] = S.q[lane];
  __syncwarp();
  fbw_forward_kinematics(w, lane, w.q, nullptr, nullptr);
  if (lane < FB_NC) {
    double P[3];
    fbw_contact_point(w, lane, P);
    double sl, du;
    pdipm_set_slack_and_dual_positive(P[2], pr.barrier, sl, du);
    S.slack[fbc_offset(FBC_DISTANCE) + lane] = sl;
    S.dual[fbc_offset(FBC_DISTANCE) + lane] = du;
  }
}

// =====================================================================================================
// LineSearch for OCPSolver (line_search/line_search.hpp:62-158, src/line_search/line_search.cpp:64-197): the lock-step
// rounds of line_search_filter.cuh  k_fb_ls_eval (warp per (instance, stage): stage cost and constraint violation of
// the trial point s + alpha d)  ->  k_fb_ls_filter (thread per instance); finished instances drop out.
// =====================================================================================================
template <bool INITIAL, bool IREF>
__global__ void __launch_bounds__(32 * FB_LS_WARPS) k_fb_ls_eval(FbArrays A, FbLin* lin) {
  IDOCP_DYN_SMEM(FbLsWork, wbase);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int stage = blockIdx.x * FB_LS_WARPS + warp;
  if (stage >= A.B * A.n_elems) return;
  FbLsWork& w = wbase[warp];
  const int b = stage / A.n_elems, e = stage - b * A.n_elems;
  if (INITIAL) { if (A.ls.n[b] != 0) return; } else { if (A.ls.state[b] != 0) return; }
  const double alpha = INITIAL ? 0.0 : A.ls.alpha[b];
  const FbElem& el = A.elems[e];
  const FbDevProblem& pr = *A.prob;
  const int nl = fbc_cone_bits(pr);
  const int kind = el.kind;
  const bool impulse = kind == FB_IMPULSE, terminal = kind == FB_TERMINAL;
  const double dt = el.dt;
  const size_t rec = (size_t)el.slot * A.B + b;
  const FbSol& S = A.sol[rec];
  FbDir& Dr = A.dir[rec];
  FbLin& L = lin[rec];
  const int dimf = terminal ? 0 : el.dimf, nvf = FB_NV + dimf;
  // ---- trial point (computeSolution, line_search.hpp:130-158); alpha = 0: the current point itself ----
  const int ncon = FBC_LIVE_ROWS(el.cactive);
  FBW_FOR(i, ncon) { w.slack[i] = S.slack[i]; w.dual[i] = Dr.dslack[i]; }   // w.dual holds dslack here
  if (lane < FB_NV) {
    const int j = lane;
    w.v[j] = INITIAL ? S.v[j] : fma(alpha, Dr.dv[j], S.v[j]);
    if (!terminal) w.a[j] = INITIAL ? S.a[j] : fma(alpha, Dr.daf[j], S.a[j]);
    w.dqv[j] = Dr.dq[j];
  }
  if (lane < FB_NU && !terminal) {
    if (!impulse) w.u[lane] = INITIAL ? S.u[lane] : fma(alpha, Dr.du[lane], S.u[lane]);
    const int i = lane / 3;
    int k = 0;
    for (int j = 0; j < i; ++j) k += el.active[j];
    const double fcur = S.f[lane];
    w.f[lane] = (INITIAL || !el.active[i]) ? fcur : fma(alpha, Dr.daf[FB_NV + 3 * k + lane % 3], fcur);
    w.fm[lane] = el.active[i] ? w.f[lane] : 0.0;
  }
  FBW_FOR(i, FB_NQ) w.q2[i] = S.q[i];
  if (!terminal) {
    const size_t nrec = (size_t)el.ls_next_slot * A.B + b;
    const FbSol& Nx = A.sol[nrec];
    const FbDir& Dn = A.dir[nrec];
    FBW_FOR(i, FB_NQ) w.qprev[i] = Nx.q[i];
    if (lane < FB_NV) { w.t18[lane] = Dn.dq[lane]; w.nv[lane] = INITIAL ? Nx.v[lane] : fma(alpha, Dn.dv[lane], Nx.v[lane]); }
  }
  __syncwarp();
  if (INITIAL) {
    FBW_FOR(i, FB_NQ) { w.q[i] = w.q2[i]; w.nq[i] = w.qprev[i]; }
  } else if (lane < 2 && !(terminal && lane == 1)) {
    fb_integrate(lane == 0 ? w.q2 : w.qprev, lane == 0 ? w.dqv : w.t18, alpha, lane == 0 ? w.q : w.nq);
  }
  __syncwarp();
  // q - q_ref and (not terminal) q - q_next, base blocks by lanes 0 and 1 in lock-step
  if (lane < 2 && !(terminal && lane == 1)) {
    double R[9], p3[3];
    fb_relative(lane == 0 ? fb_ref_q<IREF>(A, el, rec) : w.nq, w.q, R, p3);
    fb_log6(R, p3, w.rellog[lane]);
  }
  __syncwarp();
  // ---- stage cost (split_ocp.hxx:282-298 / impulse_split_ocp.hxx:145-158 / terminal_ocp.hxx:89-95) ----
  const double* wq = terminal ? pr.qf_weight : (impulse ? pr.qi_weight : pr.q_weight);
  const double* wv = terminal ? pr.vf_weight : (impulse ? pr.vi_weight : pr.v_weight);
  const double* wa = impulse ? pr.dvi_weight : pr.a_weight;
  // logs of the trial slacks by all lanes, summed in ascending order below
  if (!terminal) {
    FBW_FOR(idx, ncon) {
      const int c = fbc_comp(idx);
      const int j = idx - fbc_offset(c);
      double lg = 0.0, ar = 0.0;
      if (el.cactive[c] && j < fbc_rows(nl, c)) {
        lg = canon_log(INITIAL ? w.slack[idx] : fma(alpha, w.dual[idx], w.slack[idx]));
        if (c == FBC_DISTANCE) {
          // violation of the contact distances: after the kinematics of the trial point, below
        } else if (fbc_is_cone(c)) {
          int i, ee;
          fbc_cone_row(nl, c, j, i, ee);
          if (el.active[i]) {
            double r5[5];
            fb_friction_residual(pr.mu, fbc_cone_rows(nl, c) == 2, w.f + 3 * i, r5);
            ar = fabs(r5[ee] + w.slack[idx]);
          }
        } else {
          ar = fabs(w.slack[idx] - fbc_box_margin(c, j, pr, w.q, w.v, w.a, w.u));
        }
      }
      w.duality[idx] = lg;
      w.residual[idx] = ar;
    }
  }
  __syncwarp();
  if (lane == 0) {
    const double half = (terminal || impulse) ? 0.5 : 0.5 * dt;
    double l = 0.0;
    for (int j = 0; j < FB_NV; ++j) { const double d = j < 6 ? w.rellog[0][j] : (w.q[1 + j] - fb_ref_q<IREF>(A, el, rec)[1 + j]); l = fma(wq[j] * d, d, l); }
    for (int j = 0; j < FB_NV; ++j) { const double d = w.v[j] - fb_ref_v<IREF>(A, el, rec)[j]; l = fma(wv[j] * d, d, l); }
    if (!terminal)
      for (int j = 0; j < FB_NV; ++j) l = fma(wa[j] * w.a[j], w.a[j], l);
    double cost = half * l;
    if (!terminal) {
      const double* fw = impulse ? pr.fi_weight : pr.f_weight;
      const double* fr = impulse ? pr.fi_ref : pr.f_ref;
      double lf = 0.0;
      for (int i = 0; i < FB_NC; ++i)
        if (el.active[i])
          for (int x = 0; x < 3; ++x) { const double d = w.f[3 * i + x] - fr[3 * i + x]; lf = fma(fw[3 * i + x] * d, d, lf); }
      cost += half * lf;
      double bc = 0.0;
      for (int c = 0; c < FBC_NCOMP; ++c) {
        if (!el.cactive[c]) continue;
        double sl = 0.0;
        for (int j = 0; j < fbc_rows(nl, c); ++j) sl += w.duality[fbc_offset(c) + j];
        bc += -pr.barrier * sl;
      }
      cost += (impulse ? 1.0 : dt) * bc;
    }
    Dr.ls_cost = cost;
    if (terminal) Dr.ls_viol = 0.0;
  }
  if (terminal) return;
  // ---- constraint violation (split_ocp.hxx:301-346 / impulse_split_ocp.hxx:178-194) ----
  if (lane == 1) {
    double cl1 = 0.0;
    for (int c = 0; c < FBC_NCOMP; ++c) {
      if (!el.cactive[c]) continue;
      double s1 = 0.0;
      for (int j = 0; j < fbc_rows(nl, c); ++j) s1 += w.residual[fbc_offset(c) + j];
      cl1 += s1;
    }
    w.part[0] = cl1;
  }
  if (lane == 2) {
    double fx = 0.0;
    for (int j = 0; j < FB_NV; ++j) {
      const double d = j < 6 ? w.rellog[1][j] : (w.q[1 + j] - w.nq[1 + j]);
      fx += fabs(impulse ? d : fma(dt, w.v[j], d));
    }
    for (int j = 0; j < FB_NV; ++j) fx += fabs(impulse ? (w.v[j] + w.a[j]) - w.nv[j] : fma(dt, w.a[j], w.v[j]) - w.nv[j]);
    w.part[1] = fx;
  }
  __syncwarp();
  const double baumgarte = pr.T / pr.N;
  if (!impulse) {
    fbw_forward_kinematics(w, lane, w.q, w.v, w.a);
    if (el.cactive[FBC_DISTANCE] && lane == 1) {   // ContactDistance at the trial configuration, un-stepped slack (the last component)
      double s1 = 0.0;
      for (int i = 0; i < FB_NC; ++i) {
        if (el.active[i]) continue;
        double P[3];
        fbw_contact_point(w, i, P);
        s1 += fabs(-P[2] + w.slack[fbc_offset(FBC_DISTANCE) + i]);
      }
      w.part[0] += s1;
    }
    fbw_rnea_derivatives(w, lane, ANYMAL_GRAVITY, true, L, false);
    if (lane < FB_NU) L.IDC[6 + lane] -= w.u[lane];
  } else {
    fbw_forward_kinematics(w, lane, w.q, nullptr, w.a);
    fbw_rnea_derivatives(w, lane, 0.0, false, L, false);
    if (lane < FB_NV) w.t18[lane] = w.v[lane] + w.a[lane];
    __syncwarp();
    fbw_forward_kinematics(w, lane, w.q, w.t18, nullptr);
  }
  {
    int k = 0;
    for (int i = 0; i < FB_NC; ++i) {
      if (!el.active[i]) continue;
      if (lane == 0) {
        const int bi = 1 + ANYMAL_CONTACT_PARENT_JOINT[i];
        const double* Rf = w.R[bi];
        double P[3], vF[6], aF[6];
        fbw_contact_point(w, i, P);
        fb_pullback(Rf, P, w.ov[bi], vF);
        double* C = L.IDC + FB_NV + 3 * k;
        if (!impulse) {
          fb_pullback(Rf, P, w.oa[bi], aF);
          const double wvv = 2.0 / baumgarte, wpp = 1.0 / (baumgarte * baumgarte);
          double wxv[3];
          fb_cross(vF + 3, vF, wxv);
          for (int x = 0; x < 3; ++x) {
            const double acl = aF[x] + wxv[x];
            C[x] = fma(wpp, P[x] - el.cpoints[3 * i + x], fma(wvv, vF[x], acl));
          }
        } else {
          for (int x = 0; x < 3; ++x) C[x] = vF[x];
        }
      }
      ++k;
    }
  }
  __syncwarp();
  double pl1 = 0.0;
  if (!impulse && el.ls_sw) {
    // computeSwitchingConstraintResidual (forward_switching_constraint.hxx:57-68) at the trial point
    const double c1 = el.dt + el.ls_dt_next, c2 = el.dt * el.ls_dt_next;
    if (lane < FB_NV) w.dqv[lane] = fma(c2, w.a[lane], c1 * w.v[lane]);
    __syncwarp();
    if (lane == 0) fb_integrate(w.q, w.dqv, 1.0, w.q2);
    __syncwarp();
    fbw_forward_kinematics(w, lane, w.q2, nullptr, nullptr);
    if (lane == 0) {
      for (int i = 0; i < FB_NC; ++i) {
        if (!el.ls_imp_active[i]) continue;
        double P[3];
        fbw_contact_point(w, i, P);
        for (int x = 0; x < 3; ++x) pl1 += fabs(P[x] - el.ls_ipoints[3 * i + x]);
      }
    }
  }
  if (lane == 0) {
    double idl1 = 0.0;
    for (int j = 0; j < nvf; ++j) idl1 += fabs(L.IDC[j]);
    const double cl1 = w.part[0], fx = w.part[1];
    double viol;
    if (impulse) viol = (cl1 + fx) + idl1;
    else {
      viol = (fx + dt * idl1) + dt * cl1;
      if (el.ls_sw) viol += pl1;
    }
    Dr.ls_viol = viol;
  }
}

// totals in the reference's order (line_search.hpp:174-182): one partial sum per pass
__device__ inline void fb_ls_totals(const FbArrays& A, int b, double& cost, double& viol) {
  double c = 0.0, v = 0.0;
  for (int pass = 0; pass < 4; ++pass) {
    double cs = 0.0, vs = 0.0;
    for (int e = 0; e < A.n_elems; ++e) {
      if (!fb_in_pass(A.elems[e].kind, pass)) continue;
      const FbDir& Dr = A.dir[(size_t)A.elems[e].slot * A.B + b];
      cs += Dr.ls_cost;
      vs += Dr.ls_viol;
    }
    c = pass == 0 ? cs : c + cs;
    v = pass == 0 ? vs : v + vs;
  }
  cost = c;
  viol = v;
}
// mode 0 / 1: ls_filter_round from the fraction-to-boundary step; mode 2: publish alpha as the primal step
__global__ void k_fb_ls_filter(FbArrays A, int mode) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= A.B) return;
  if (mode == 2) {
    A.steps[2 * b] = A.ls.alpha[b];
    return;
  }
  ls_filter_round(A.ls, b, mode, A.steps[2 * b], A.ls_status, [&](double& cost, double& viol) { fb_ls_totals(A, b, cost, viol); });
}

}  // namespace idocp_b200
