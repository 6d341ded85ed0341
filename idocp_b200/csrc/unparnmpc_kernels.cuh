// unparnmpc_kernels.cuh -- batched UnParNMPCSolver: per-stage KKT inversion (coarse update) and the
// backward / forward correction sweeps.
//
//   k_parnmpc_invert            <-> SplitUnBackwardCorrection::coarseUpdate + SplitUnKKTMatrixInverter::invert
//                                   (unocp/split_unbackward_correction.hxx:37-62, split_unkkt_matrix_inverter.hxx:40-79)
//   k_parnmpc_backward_serial   <-> backwardCorrectionSerial   (split_unbackward_correction.hxx:71-79)
//   k_parnmpc_backward_parallel <-> backwardCorrectionParallel (:82-90)
//   k_parnmpc_forward_serial    <-> forwardCorrectionSerial    (:93-101)
//   k_parnmpc_forward_parallel  <-> forwardCorrectionParallel + auxMat + computeDirection (:104-121;
//                                   src/unocp/unbackward_correction.cpp:114-133)
//   k_parnmpc_init_aux          <-> UnBackwardCorrection::initAuxMat (src/unocp/unbackward_correction.cpp:55-64)
//
// The stage linearisation is k_linearize<.., BACKWARD_EULER = true> (unocp_kernels.cuh); the condensed
// direction, step sizes and the update are k_expand<true> / k_update.
//
// Stages 1..N of the reference are stored at index 0..N-1.  KKT system of a stage, unknown order
// [dlmd, dgmm | da, dq, dv], matrix [[0, F],[F^T, Q]], F = [[0,-I,dt I],[dt I,0,-I]], Q in block order (a,q,v).
// Notation for the blocks of the 35x35 inverse: TL = inv[0:14,0:14] = -S^-1, TR = inv[0:14,14:35],
// BL = TR^T, BR = inv[14:35,14:35].
#pragma once
#include "unocp_kernels.cuh"
#include "warp_llt.cuh"

namespace idocp_b200 {

constexpr int NX2 = 2 * NV;   // 14
constexpr int NQ3 = 3 * NV;   // 21
constexpr int NKKT = 5 * NV;  // 35

// s_new of the backward correction: [N stages]
enum SNSlot { SN_LMD = 0, SN_GMM, SN_A, SN_Q, SN_V, SN_NUM = 5 };
// x_res of the correction sweeps (head, tail): [N stages]
enum XRSlot { XR_H = 0, XR_T, XR_NUM = 2 };
// Blocks of the KKT inverse that the corrections use, stored for mat-vecs "lane = row, slot = column":
// slot (c, rb) = first + c * nrb + rb holds rows 7 rb .. 7 rb + 6 of column c of the block.
//   BS: inv[0:14, 21:35]   (14 x 14)  backwardCorrectionSerial      BP: inv[14:35, 21:35] (21 x 14)  ...Parallel
//   FS: inv[21:35, 0:14]   (14 x 14)  forwardCorrectionSerial       FP: inv[0:21, 0:14]   (21 x 14)  ...Parallel
enum KISlot { KI_BS = 0, KI_BP = 28, KI_FS = 70, KI_FP = 98, KI_NUM = 140 };
// aux_mat (14 x 14), slot (c, rb) = c * 2 + rb: [N stages] (index 0 is never used)
constexpr int AUX_NUM = 28;

struct ParNMPCLayout {
  double* SN = nullptr;
  double* XR = nullptr;
  double* KI = nullptr;
  double* AUX = nullptr;
};

template <typename Alloc>
inline int parnmpc_alloc(ParNMPCLayout& PL, int N, int Bp, Alloc alloc) {
  const size_t G = static_cast<size_t>(Bp) / 4, n = static_cast<size_t>(N);
  int rc = 0;
  rc |= alloc(&PL.SN, n * G * SN_NUM * SLOT);
  rc |= alloc(&PL.XR, n * G * XR_NUM * SLOT);
  rc |= alloc(&PL.KI, n * G * KI_NUM * SLOT);
  rc |= alloc(&PL.AUX, n * G * AUX_NUM * SLOT);
  return rc;
}

// ---------------------------------------------------------------------------------------------
// k_parnmpc_init_aux: every aux_mat = Hessian of the terminal cost = diag(qf_weight, vf_weight)
// ---------------------------------------------------------------------------------------------
// TASK = true: + the (dense) Gauss-Newton Hessian of the terminal task-space cost at s[N-1]
// (TerminalUnParNMPC::computeTerminalCostHessian, terminal_unparnmpc.hxx:230-241); IREF = true: the instance's task table
template <bool TASK, bool IREF = false>
__global__ void __launch_bounds__(CTA_THREADS) k_parnmpc_init_aux(const DevProblem* __restrict__ Pp, Layout L,
                                                                  ParNMPCLayout PL) {
  IDOCP_DYN_SMEM(double, smem);
  const DevProblem& P = *Pp;
  const int lane = lane_in_octet();
  const StageTask t = stage_task(L, L.N);
  double* A = rec_ptr(PL.AUX, AUX_NUM, L.G, t.stage, t.g);
  double col[NV];   // aux(lane, c), c = 0..6: row `lane` of the q-q block
#pragma unroll
  for (int c = 0; c < NV; ++c) col[c] = (lane == c) ? P.qf_weight[lane] : 0.0;
  if (TASK) {
    double* tile = smem + (threadIdx.x >> 3) * (OCT * PAIR_TILE);
    const bool act = lane < NV;
    const double* X = rec_ptr(L.X, X_NUM, L.G, L.N - 1, t.g);
    double R[9];
    V3 p;
    chain_fk(lane, act ? X[X_Q * SLOT] : 0.0, P.model + lane * MODEL_STRIDE, R, p);
    TaskEval te;
    task_evaluate<true>(R, p, P.ee, task_ref_row<IREF>(L, L.N - 1, t.g * 4 + ((threadIdx.x >> 3) & 3)), te, P.task_enabled);
    task_share_columns(lane, te, tile);
    double gf, hf[NV];
    task_gradient_hessian(te, P.task_wf6, tile, gf, hf);
    __syncwarp();
    // transpose through the tile: lane j needs H(j, c), owned by lane c as hf[j]
    double* mine = tile + lane * PAIR_TILE;
#pragma unroll
    for (int r = 0; r < NV; ++r) mine[r] = hf[r];
    __syncwarp();
    const int ln = act ? lane : 0;
#pragma unroll
    for (int c = 0; c < NV; ++c) col[c] += tile[c * PAIR_TILE + ln];
    if (!act) {
#pragma unroll
      for (int c = 0; c < NV; ++c) col[c] = 0.0;
    }
  }
#pragma unroll
  for (int c = 0; c < NX2; ++c) {
    A[(c * 2 + 0) * SLOT] = c < NV ? col[c] : 0.0;
    A[(c * 2 + 1) * SLOT] = (c >= NV && lane == c - NV) ? P.vf_weight[lane] : 0.0;
  }
}

// ---------------------------------------------------------------------------------------------
// k_parnmpc_invert: one WARP per (instance, stage); one CTA = the 4 instances of a group.
// All matrices live in shared memory (column-major, odd column strides: conflict-free for
// "lane = row" accesses) or, column per lane, in registers.  Every element is produced by the
// same ascending-index fma chain as in the oracle (invert_unkkt), so the result is bit-identical.
// ---------------------------------------------------------------------------------------------
constexpr int INV_LDQ = NQ3;       // 21 (odd)
constexpr int INV_LDX = NX2 + 1;   // 15 (odd)
// per-warp shared memory (doubles); every offset is even, so that element e of an array is 16-byte aligned iff e is even
// (the broadcast operand loads of the factorisations and products are issued two doubles at a time, inv_ld2)
constexpr int INV_OFF_A = 0;                           // Q -> L (21 x 21, column k of L contiguous), later Qinv -> BR
constexpr int INV_OFF_LT = INV_OFF_A + 442;            // L^T: row r of L contiguous (backward substitution); LLT(S)^T later
constexpr int INV_OFF_RD = INV_OFF_LT + 442;           // reciprocal pivots (21)
constexpr int INV_OFF_FQ = INV_OFF_RD + 24;            // FQinv (14 x 21), column stride 15
// S (14 x 14; first used as staging of aux_next) lives in the upper part of the L^T region: L^T of Q is dead when S is formed,
// LLT(S)^T takes LT[0, 210) only, and S * TR is parked over FQinv (dead once TR exists) -- 15.97 -> 14.29 KB per warp, which is
// what lets a fourth CTA onto the SM
constexpr int INV_OFF_S = INV_OFF_LT + 220;
constexpr int INV_OFF_LS = INV_OFF_FQ + 316;           // LLT(S), then TL = -S^-1 in place (14 x 14)
constexpr int INV_OFF_TL = INV_OFF_LS;
constexpr int INV_OFF_TR = INV_OFF_TL + NX2 * INV_LDX; // TR (14 x 21)
constexpr int INV_OFF_RES = INV_OFF_TR + 316;          // residual (35)
constexpr int INV_SMEM_PER_WARP = INV_OFF_RES + 36;
constexpr int INV_SMEM_BYTES = WARPS_PER_CTA * INV_SMEM_PER_WARP * static_cast<int>(sizeof(double));
static_assert(INV_OFF_LT % 2 == 0 && INV_OFF_FQ % 2 == 0 && INV_OFF_S % 2 == 0 && INV_OFF_LS % 2 == 0 && INV_OFF_TR % 2 == 0 &&
              INV_SMEM_PER_WARP % 2 == 0, "16-byte alignment of the even elements");
static_assert(INV_OFF_S + NX2 * INV_LDX <= INV_OFF_RD && NX2 * INV_LDX <= 220, "S and LLT(S)^T share the L^T region");
static_assert(4 * (INV_SMEM_BYTES + 1024) <= 228 * 1024, "four CTAs per SM");

// moves `nslots` slots of this warp's instance between a (stage, group) record and a per-lane
// functor, 4 slots per warp instruction (lane = 8 * sub + j): all global accesses of the loop are
// issued back to back (full unroll), i.e. one memory latency per record
template <int nslots, typename F>
__device__ __forceinline__ void warp_load_slots(const double* __restrict__ rec, int wl, F&& f) {
  const int sub = wl >> 3, j8 = wl & 7;
  double val[(nslots + 3) / 4];
#pragma unroll
  for (int k = 0; k < (nslots + 3) / 4; ++k) {
    const int slot = 4 * k + sub;
    val[k] = slot < nslots ? rec[slot * SLOT + j8] : 0.0;
  }
#pragma unroll
  for (int k = 0; k < (nslots + 3) / 4; ++k) {
    const int slot = 4 * k + sub;
    if (slot < nslots && j8 < NV) f(slot, j8, val[k]);
  }
}

// ---- the three dense products of the inversion on the FP64 tensor cores ----
// mma.sync.aligned.m8n8k4.f64 is bit-identical to the ascending fma chain (tools/dmma_probe.cu, DESIGN.md section 5), so
// C = A B by ONE warp in 8 x 16 strips (two tiles sharing the A fragment), accumulators chained over k from -0.0 (the first
// fma is then the plain product), ragged edges zero-padded, equals the per-element chain of the oracle.  Operands in shared
// memory with arbitrary strides; every element goes to `store(i, j, value)`.  Fragments: a = A[g][t], b = B[t][g],
// c = C[g][2 t + {0, 1}], g = lane / 4, t = lane % 4.
__device__ __forceinline__ void inv_dmma(double& d0, double& d1, double a, double b) {
#ifndef IDOCP_B200_EMU
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
#else
  emu_dmma_m8n8k4(d0, d1, a, b);
#endif
}
template <int M, int N, int K, class Store>
__device__ __forceinline__ void inv_mm_dmma(int lane, const double* __restrict__ A, int ars, int acs, const double* __restrict__ B, int brs,
                                            int bcs, Store store) {
  const int g = lane >> 2, t = lane & 3;
  constexpr int TM = (M + 7) / 8, TN = (N + 15) / 16;
#pragma unroll
  for (int s = 0; s < TM * TN; ++s) {
    const int i0 = (s / TN) * 8, j0 = (s % TN) * 16;
    const int row = i0 + g, ca = j0 + 2 * t, cb = ca + 8, ba = j0 + g, bb = ba + 8;
    const bool rok = row < M, baok = ba < N, bbok = bb < N;
    double c00 = -0.0, c01 = -0.0, c10 = -0.0, c11 = -0.0;
    const double* ap = A + (rok ? row : 0) * ars + t * acs;
    const double* bpa = B + (baok ? ba : 0) * bcs + t * brs;
    const double* bpb = B + (bbok ? bb : 0) * bcs + t * brs;
#pragma unroll
    for (int l = 0; l < K; l += 4) {
      const bool kin = l + t < K;
      const double a = (rok && kin) ? ap[l * acs] : 0.0;
      const double b0 = (baok && kin) ? bpa[l * brs] : 0.0, b1 = (bbok && kin) ? bpb[l * brs] : 0.0;
      inv_dmma(c00, c01, a, b0);
      if (j0 + 8 < N) inv_dmma(c10, c11, a, b1);
    }
    if (rok) {
      if (ca < N) store(row, ca, c00);
      if (ca + 1 < N) store(row, ca + 1, c01);
      if (cb < N) store(row, cb, c10);
      if (cb + 1 < N) store(row, cb + 1, c11);
    }
  }
}

constexpr int INV_MINB = 4;   // 128 registers without spills (164 at three CTAs per SM), 14.3 KB of shared memory per warp

__global__ void __launch_bounds__(CTA_THREADS, INV_MINB) k_parnmpc_invert(const DevProblem* __restrict__ Pp,
                                                                          Layout L, ParNMPCLayout PL) {
  IDOCP_DYN_SMEM(double, smem);
  const DevProblem& P = *Pp;
  const int wl = threadIdx.x & 31;           // lane in the warp
  const int inst = threadIdx.x >> 5;         // instance of the group = warp of the CTA
  const int i = blockIdx.x / L.G;            // stage index
  const int g = blockIdx.x % L.G;
  const int N = L.N;
  const double dt = P.dt;
  double* sm = smem + inst * INV_SMEM_PER_WARP;
  double* A = sm + INV_OFF_A;
  double* LT = sm + INV_OFF_LT;
  double* rd = sm + INV_OFF_RD;
  double* FQ = sm + INV_OFF_FQ;
  double* S = sm + INV_OFF_S;
  double* LS = sm + INV_OFF_LS;
  double* TL = sm + INV_OFF_TL;
  double* TR = sm + INV_OFF_TR;
  double* res = sm + INV_OFF_RES;
  // this warp's view of a (stage, group) record: element (slot, j) of its instance
  const size_t go = static_cast<size_t>(inst) * OCT;
  const int sub = wl >> 3, j8 = wl & 7;      // 4 slots are moved per warp instruction

  // ---- aux_mat of the next stage (none for the last stage) -> staging in S: aux(R, C) = S[C * 15 + R] ----
  const bool has_aux = (i < N - 1);
  if (has_aux) {
    warp_load_slots<AUX_NUM>(PL.AUX + (static_cast<size_t>(i + 1) * L.G + g) * (AUX_NUM * SLOT) + go, wl,
                             [&](int slot, int j, double val) { S[(slot >> 1) * INV_LDX + (slot & 1) * NV + j] = val; });
  }
  __syncwarp();
  // ---- Q (lower triangle, as SplitUnBackwardCorrection::coarseUpdate leaves it: Qxx += aux_next, then
  //      Qvq = Qqv^T and Qxa = Qax^T) and the residual [Fq, Fv, la, lq, lv] ----
  warp_load_slots<KQ_NUM>(L.KQ + (static_cast<size_t>(i) * L.G + g) * (KQ_NUM * SLOT) + go, wl,
                          [&](int slot, int c, double val) {
    if (slot >= KQ_FQ) { res[(slot - KQ_FQ) * NV + c] = val; return; }
    const int blk = slot / NV, r = slot - blk * NV;
    switch (blk) {
      case 0: if (r >= c) A[c * INV_LDQ + r] = val; break;                                  // aa
      case 1: A[r * INV_LDQ + NV + c] = val; break;                                         // qa = aq^T
      case 2: A[r * INV_LDQ + 2 * NV + c] = val; break;                                     // va = av^T
      case 3: if (r >= c) A[(NV + c) * INV_LDQ + NV + r] = has_aux ? val + S[c * INV_LDX + r] : val; break;
      case 4: A[(NV + r) * INV_LDQ + 2 * NV + c] = has_aux ? val + S[(NV + c) * INV_LDX + r] : val; break;  // vq = qv^T
      default: if (r >= c) A[(2 * NV + c) * INV_LDQ + 2 * NV + r] = has_aux ? val + S[(NV + c) * INV_LDX + NV + r] : val; break;
    }
  });
  __syncwarp();

  // ---- llt_Q_.compute(Q); Qinv = llt_Q_.solve(I): lane c computes column c, then parks it over L (dead) ----
  int fail = warp_llt<NQ3, INV_LDQ>(A, LT, rd, wl);
  const int cq = wl < NQ3 ? wl : 0;
  {
    double y[NQ3];
    warp_llt_solve_unit<NQ3, INV_LDQ>(A, LT, rd, cq, y);
    __syncwarp();   // every lane is done reading L
    if (wl < NQ3) {
#pragma unroll
      for (int r = 0; r < NQ3; ++r) A[wl * INV_LDQ + r] = y[r];
      // FQinv (14 x 21): rows Fq = -Qinv[q rows] + dt Qinv[v rows]; rows Fv = dt Qinv[a rows] - Qinv[v rows]
#pragma unroll
      for (int r = 0; r < NV; ++r) {
        FQ[wl * INV_LDX + r] = fma(dt, y[2 * NV + r], -y[NV + r]);
        FQ[wl * INV_LDX + NV + r] = fma(dt, y[r], -y[2 * NV + r]);
      }
    }
  }
  __syncwarp();
  // ---- S = FQinv F^T (14 x 14) ----
#pragma unroll
  for (int e0 = 0; e0 < NX2 * NX2; e0 += 32) {
    const int e = e0 + wl;
    if (e < NX2 * NX2) {
      const int cc = e / NX2, r = e - cc * NX2;
      double sv;
      if (cc < NV) sv = fma(dt, FQ[(2 * NV + cc) * INV_LDX + r], -FQ[(NV + cc) * INV_LDX + r]);
      else sv = fma(dt, FQ[(cc - NV) * INV_LDX + r], -FQ[(NV + cc) * INV_LDX + r]);
      S[cc * INV_LDX + r] = sv;
      LS[cc * INV_LDX + r] = sv;
    }
  }
  __syncwarp();
  // ---- llt_S_.compute(S); TL = -llt_S_.solve(I), written over the factor once every lane has solved ----
  fail |= warp_llt<NX2, INV_LDX>(LS, LT, rd, wl);
  {
    double z[NX2];
    const int cs = wl < NX2 ? wl : 0;
    warp_llt_solve_unit<NX2, INV_LDX>(LS, LT, rd, cs, z);
    __syncwarp();
    if (wl < NX2) {
#pragma unroll
      for (int r = 0; r < NX2; ++r) TL[wl * INV_LDX + r] = -z[r];
    }
  }
  __syncwarp();
  // ---- TR = -(TL FQinv) (14 x 21), ST = S TR (14 x 21, parked over the dead FQinv), BR = Qinv - TR^T ST (21 x 21, in place over
  //      the parked Qinv): three warp-level DMMA products, every element the oracle's ascending chain ----
  {
    double* ST = FQ;   // FQinv is dead once TR exists
    inv_mm_dmma<NX2, NQ3, NX2>(wl, TL, 1, INV_LDX, FQ, 1, INV_LDX, [=](int r, int c, double v) { TR[c * INV_LDX + r] = -v; });
    __syncwarp();
    inv_mm_dmma<NX2, NQ3, NX2>(wl, S, 1, INV_LDX, TR, 1, INV_LDX, [=](int r, int c, double v) { ST[c * INV_LDX + r] = v; });
    __syncwarp();
    inv_mm_dmma<NQ3, NQ3, NX2>(wl, TR, INV_LDX, 1, ST, 1, INV_LDX, [=](int r, int c, double v) { A[c * INV_LDQ + r] -= v; });
  }
  __syncwarp();

  // ---- d = KKT^-1 residual; s_new = s - d (lmd, gmm, a, q, v): lane = row, two passes (35 rows) ----
  const double* X = L.X + (static_cast<size_t>(i) * L.G + g) * (X_NUM * SLOT) + go;
  double* SN = PL.SN + (static_cast<size_t>(i) * L.G + g) * (SN_NUM * SLOT) + go;
#pragma unroll
  for (int pass = 0; pass < 2; ++pass) {
    const int R = pass * 32 + wl;
    if (R < NKKT) {
      const int f = R / NV, jj = R - f * NV;   // f: 0 lmd 1 gmm 2 a 3 q 4 v
      const int xs = f == 0 ? X_LMD : (f == 1 ? X_GMM : (f == 2 ? X_A : (f == 3 ? X_Q : X_V)));
      const double sx = X[xs * SLOT + jj];
      double acc = 0.0;
      if (R < NX2) {
#pragma unroll
        for (int c = 0; c < NX2; ++c) acc = fma(TL[c * INV_LDX + R], res[c], acc);
#pragma unroll
        for (int c = 0; c < NQ3; ++c) acc = fma(TR[c * INV_LDX + R], res[NX2 + c], acc);
      } else {
        const int rr = R - NX2;
#pragma unroll
        for (int c = 0; c < NX2; ++c) acc = fma(TR[rr * INV_LDX + c], res[c], acc);
#pragma unroll
        for (int c = 0; c < NQ3; ++c) acc = fma(A[c * INV_LDQ + rr], res[NX2 + c], acc);
      }
      SN[f * SLOT + jj] = sx - acc;
    }
  }

  // ---- blocks of the inverse for the correction sweeps (pad lanes are written as zeros) ----
  double* KI = PL.KI + (static_cast<size_t>(i) * L.G + g) * (KI_NUM * SLOT) + go;
  const bool real = j8 < NV;
#pragma unroll
  for (int k = 0; k < KI_BP / 4; ++k) {           // BS: inv[7 rb + j][21 + c] = TR(7 rb + j, 7 + c)
    const int slot = 4 * k + sub, c = slot >> 1, rb = slot & 1;
    KI[(KI_BS + slot) * SLOT + j8] = real ? TR[(NV + c) * INV_LDX + rb * NV + j8] : 0.0;
  }
#pragma unroll
  for (int k = 0; k < (KI_FS - KI_BP + 3) / 4; ++k) {   // BP: inv[14 + 7 rb + j][21 + c] = BR(7 rb + j, 7 + c)
    const int slot = 4 * k + sub, c = slot / 3, rb = slot - c * 3;
    if (slot < KI_FS - KI_BP) KI[(KI_BP + slot) * SLOT + j8] = real ? A[(NV + c) * INV_LDQ + rb * NV + j8] : 0.0;
  }
#pragma unroll
  for (int k = 0; k < (KI_FP - KI_FS) / 4; ++k) {  // FS: inv[21 + 7 rb + j][c] = TR(c, 7 + 7 rb + j)
    const int slot = 4 * k + sub, c = slot >> 1, rb = slot & 1;
    KI[(KI_FS + slot) * SLOT + j8] = real ? TR[(NV + rb * NV + j8) * INV_LDX + c] : 0.0;
  }
#pragma unroll
  for (int k = 0; k < (KI_NUM - KI_FP + 3) / 4; ++k) {  // FP: inv[7 rb + j][c] = TL(7 rb + j, c) | TR(c, j)
    const int slot = 4 * k + sub, c = slot / 3, rb = slot - c * 3;
    if (slot < KI_NUM - KI_FP)
      KI[(KI_FP + slot) * SLOT + j8] = real ? (rb < 2 ? TL[c * INV_LDX + rb * NV + j8] : TR[j8 * INV_LDX + c]) : 0.0;
  }
  if (fail && wl == 0) {
    const int b = g * 4 + inst;
    if (b < L.B) L.status[b] |= 1;
  }
}

// y[rb] = sum_c M[c][rb][lane] * xr[c], c ascending (xr[c] = head for c < 7, tail otherwise): the
// "lane = row, slot = column" mat-vec of the correction sweeps
template <int NRB>
__device__ __forceinline__ void oct_matvec14(const double* __restrict__ M, double xh, double xt, double (&y)[NRB]) {
#pragma unroll
  for (int rb = 0; rb < NRB; ++rb) y[rb] = 0.0;
#pragma unroll
  for (int c = 0; c < NX2; ++c) {
    const double xc = oct_bcast(c < NV ? xh : xt, c < NV ? c : c - NV);
#pragma unroll
    for (int rb = 0; rb < NRB; ++rb) y[rb] = fma(M[(c * NRB + rb) * SLOT], xc, y[rb]);
  }
}

// ask the L2 for slots [first_slot, first_slot + nslots) of the (stage, group) record `rec` points into (this thread's
// rec_ptr): the serial sweeps below would otherwise pay one DRAM round trip per stage.  No effect on results.
__device__ __forceinline__ void warp_prefetch_slots(const double* rec, int first_slot, int nslots) {
#ifndef IDOCP_B200_EMU
  const int lane = threadIdx.x & 31;
  const char* c = reinterpret_cast<const char*>(rec - lane + first_slot * SLOT);
  for (int o = lane * 128; o < nslots * SLOT * static_cast<int>(sizeof(double)); o += 32 * 128)
    asm volatile("prefetch.global.L2 [%0];" ::"l"(c + o));
#endif
}
// stages ahead of the one being corrected; distances 4 and 8 measured slower (profiles/r2zs_variant_pf*.json)
constexpr int PARNMPC_PREFETCH_DISTANCE = 2;

// ---------------------------------------------------------------------------------------------
// k_parnmpc_backward_serial: i = N-2 .. 0:  x_res = s_new[i+1].(lmd,gmm) - s[i+1].(lmd,gmm);
// s_new[i].(lmd,gmm) -= inv_i[0:14, 21:35] x_res.  One octet per instance.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) k_parnmpc_backward_serial(Layout L, ParNMPCLayout PL) {
  const int g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
  if (g >= L.G) return;   // read-modify-write kernel: tail warps must not redo a group (whole warps exit)
  const int N = L.N;
  const size_t xs = static_cast<size_t>(L.G) * (X_NUM * SLOT), ss = static_cast<size_t>(L.G) * (SN_NUM * SLOT);
  const size_t ks = static_cast<size_t>(L.G) * (KI_NUM * SLOT), rs = static_cast<size_t>(L.G) * (XR_NUM * SLOT);
  const double* X = rec_ptr(L.X, X_NUM, L.G, N - 1, g);
  double* SN = rec_ptr(PL.SN, SN_NUM, L.G, N - 1, g);
  const double* KI = rec_ptr(PL.KI, KI_NUM, L.G, N - 1, g);
  double* XR = rec_ptr(PL.XR, XR_NUM, L.G, N - 1, g);
  double nl = SN[SN_LMD * SLOT], ng = SN[SN_GMM * SLOT];   // corrected s_new of stage i + 1
  for (int i = N - 2; i >= 0; --i) {
    const double xh = nl - X[X_LMD * SLOT];
    const double xt = ng - X[X_GMM * SLOT];
    X -= xs; SN -= ss; KI -= ks; XR -= rs;
    if (i >= PARNMPC_PREFETCH_DISTANCE) {
      warp_prefetch_slots(KI - PARNMPC_PREFETCH_DISTANCE * ks, KI_BS, KI_BP - KI_BS);
      warp_prefetch_slots(SN - PARNMPC_PREFETCH_DISTANCE * ss, SN_LMD, 2);
      warp_prefetch_slots(X - (PARNMPC_PREFETCH_DISTANCE - 1) * xs, X_LMD, 2);
    }
    XR[XR_H * SLOT] = xh;
    XR[XR_T * SLOT] = xt;
    double y[2];
    oct_matvec14<2>(KI + KI_BS * SLOT, xh, xt, y);
    nl = SN[SN_LMD * SLOT] - y[0];
    ng = SN[SN_GMM * SLOT] - y[1];
    SN[SN_LMD * SLOT] = nl;
    SN[SN_GMM * SLOT] = ng;
  }
}

// k_parnmpc_backward_parallel: stages 0..N-2: s_new.(a,q,v) -= inv_i[14:35, 21:35] x_res
__global__ void __launch_bounds__(CTA_THREADS) k_parnmpc_backward_parallel(Layout L, ParNMPCLayout PL) {
  if (static_cast<long>(blockIdx.x) * WARPS_PER_CTA + (threadIdx.x >> 5) >= static_cast<long>(L.N - 1) * L.G) return;
  const StageTask t = stage_task(L, L.N - 1);
  double* SN = rec_ptr(PL.SN, SN_NUM, L.G, t.stage, t.g);
  const double* KI = rec_ptr(PL.KI, KI_NUM, L.G, t.stage, t.g);
  const double* XR = rec_ptr(PL.XR, XR_NUM, L.G, t.stage, t.g);
  double y[3];
  oct_matvec14<3>(KI + KI_BP * SLOT, XR[XR_H * SLOT], XR[XR_T * SLOT], y);
  SN[SN_A * SLOT] -= y[0];
  SN[SN_Q * SLOT] -= y[1];
  SN[SN_V * SLOT] -= y[2];
}

// ---------------------------------------------------------------------------------------------
// k_parnmpc_forward_serial: i = 1 .. N-1:  x_res = s_new[i-1].(q,v) - s[i-1].(q,v);
// s_new[i].(q,v) -= inv_i[21:35, 0:14] x_res.  One octet per instance.
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) k_parnmpc_forward_serial(Layout L, ParNMPCLayout PL) {
  const int g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
  if (g >= L.G) return;   // read-modify-write kernel: tail warps must not redo a group (whole warps exit)
  const int N = L.N;
  const size_t xs = static_cast<size_t>(L.G) * (X_NUM * SLOT), ss = static_cast<size_t>(L.G) * (SN_NUM * SLOT);
  const size_t ks = static_cast<size_t>(L.G) * (KI_NUM * SLOT), rs = static_cast<size_t>(L.G) * (XR_NUM * SLOT);
  const double* X = rec_ptr(L.X, X_NUM, L.G, 0, g);
  double* SN = rec_ptr(PL.SN, SN_NUM, L.G, 0, g);
  const double* KI = rec_ptr(PL.KI, KI_NUM, L.G, 0, g);
  double* XR = rec_ptr(PL.XR, XR_NUM, L.G, 0, g);
  double nq = SN[SN_Q * SLOT], nv = SN[SN_V * SLOT];       // corrected s_new of stage i - 1
  for (int i = 1; i < N; ++i) {
    const double xh = nq - X[X_Q * SLOT];
    const double xt = nv - X[X_V * SLOT];
    X += xs; SN += ss; KI += ks; XR += rs;
    if (i + PARNMPC_PREFETCH_DISTANCE < N) {
      warp_prefetch_slots(KI + PARNMPC_PREFETCH_DISTANCE * ks, KI_FS, KI_FP - KI_FS);
      warp_prefetch_slots(SN + PARNMPC_PREFETCH_DISTANCE * ss, SN_Q, 2);
      warp_prefetch_slots(X + (PARNMPC_PREFETCH_DISTANCE - 1) * xs, X_Q, 2);
    }
    XR[XR_H * SLOT] = xh;
    XR[XR_T * SLOT] = xt;
    double y[2];
    oct_matvec14<2>(KI + KI_FS * SLOT, xh, xt, y);
    nq = SN[SN_Q * SLOT] - y[0];
    nv = SN[SN_V * SLOT] - y[1];
    SN[SN_Q * SLOT] = nq;
    SN[SN_V * SLOT] = nv;
  }
}

// ---------------------------------------------------------------------------------------------
// k_parnmpc_forward_parallel: stages 1..N-1: s_new.(lmd,gmm,a) -= inv_i[0:21, 0:14] x_res and
// aux_mat[i] = -inv_i[0:14, 0:14]; every stage: d = s_new - s (computeDirection).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) k_parnmpc_forward_parallel(Layout L, ParNMPCLayout PL) {
  if (static_cast<long>(blockIdx.x) * WARPS_PER_CTA + (threadIdx.x >> 5) >= static_cast<long>(L.N) * L.G) return;
  const StageTask t = stage_task(L, L.N);
  const int i = t.stage;
  const double* X = rec_ptr(L.X, X_NUM, L.G, i, t.g);
  double* SN = rec_ptr(PL.SN, SN_NUM, L.G, i, t.g);
  double* D = rec_ptr(L.D, D_NUM, L.G, i, t.g);
  double nl = SN[SN_LMD * SLOT], ng = SN[SN_GMM * SLOT], na = SN[SN_A * SLOT];
  if (i > 0) {
    const double* KI = rec_ptr(PL.KI, KI_NUM, L.G, i, t.g);
    const double* XR = rec_ptr(PL.XR, XR_NUM, L.G, i, t.g);
    double* AX = rec_ptr(PL.AUX, AUX_NUM, L.G, i, t.g);
    double y[3];
    oct_matvec14<3>(KI + KI_FP * SLOT, XR[XR_H * SLOT], XR[XR_T * SLOT], y);
    nl -= y[0];
    ng -= y[1];
    na -= y[2];
#pragma unroll
    for (int c = 0; c < NX2; ++c) {
      AX[(c * 2 + 0) * SLOT] = -KI[(KI_FP + c * 3 + 0) * SLOT];
      AX[(c * 2 + 1) * SLOT] = -KI[(KI_FP + c * 3 + 1) * SLOT];
    }
  }
  D[D_LMD * SLOT] = nl - X[X_LMD * SLOT];
  D[D_GMM * SLOT] = ng - X[X_GMM * SLOT];
  D[D_A * SLOT] = na - X[X_A * SLOT];
  D[D_Q * SLOT] = SN[SN_Q * SLOT] - X[X_Q * SLOT];
  D[D_V * SLOT] = SN[SN_V * SLOT] - X[X_V * SLOT];
}

}  // namespace idocp_b200
