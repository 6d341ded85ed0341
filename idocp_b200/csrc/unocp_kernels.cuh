// unocp_kernels.cuh -- the batched Newton step of idocp's UnOCPSolver (fixed base, no contacts).
//
//   k_linearize   <-> SplitUnOCP::linearizeOCP / computeKKTResidual + squaredNormKKTResidual
//                     (reference include/idocp/unocp/split_unocp.hxx:69-99,141-174); one octet per
//                     (instance, stage), fully parallel
//   k_riccati     <-> UnRiccatiRecursion backward + forward recursion (src/unocp/unriccati_
//                     recursion.cpp:39-65, unocp/split_unriccati_factorizer.hxx:30-57,
//                     backward_unriccati_recursion_factorizer.hxx:29-89); one octet per instance,
//                     serial over the horizon
//   k_expand      <-> computeCostateDirection + SplitUnOCP::computeCondensedDirection +
//                     max{Primal,Dual}StepSize (unocp_solver.cpp:103-113); one octet per
//                     (instance, stage), fully parallel
//   k_update      <-> min over stages + updatePrimal / updateDual (unocp_solver.cpp:114-133)
//   k_kkt_sum     <-> UnOCPSolver::KKTError (unocp_solver.cpp:190-202)
//   k_init_constraints <-> UnOCPSolver::initConstraints (unocp_solver.cpp:59-70)
//
// Lane l < 7 of an octet owns joint l (all cost / constraint / state-equation algebra is lane
// local) and column l of every 7x7 block.  One warp = one GROUP of 4 instances (common.cuh).
#pragma once
#include "chain_dynamics.cuh"
#include "pdipm.cuh"
#include "task_space_cost.cuh"
#include "tma.cuh"

namespace idocp_b200 {

constexpr int LIN_MINB = 2;          // min resident CTAs/SM of k_linearize (register cap = 65536 / (128 * MINB))
constexpr int UL_CTAS_PER_SM = 2;    // persistent k_update_linearize: resident CTAs per SM (97 KB of shared memory each)
constexpr int RIC_MINB = 2;
constexpr int EXP_MINB = 3;          // k_expand holds its whole W record in registers (166): 3 warps per scheduler, 12 per SM
constexpr int WARPS_PER_CTA = 4;
constexpr int OCTETS_PER_CTA = 4 * WARPS_PER_CTA;  // 16 octets, 128 threads
constexpr int CTA_THREADS = 32 * WARPS_PER_CTA;

// ---------------------------------------------------------------------------------------------
// constraints: primal-dual interior point rows of the six joint-limit components.
// Per lane: one row of each component (its joint).  comp: 0 pos-lo 1 pos-up 2 vel-lo 3 vel-up
// 4 trq-lo 5 trq-up.  (constraints/pdipm.hxx, src/constraints/joint_*_limit.cpp)
// ---------------------------------------------------------------------------------------------
struct LaneLimits {
  double qmin, qmax, vmax, umax;
};

__device__ __forceinline__ double con_residual(int comp, const LaneLimits& L, double q, double v, double u,
                                               double slack) {
  switch (comp) {
    case 0: return L.qmin - q + slack;
    case 1: return q - L.qmax + slack;
    case 2: return (-L.vmax) - v + slack;
    case 3: return v - L.vmax + slack;
    case 4: return (-L.umax) - u + slack;
    default: return u - L.umax + slack;
  }
}
__device__ __forceinline__ double con_margin(int comp, const LaneLimits& L, double q, double v, double u) {
  switch (comp) {
    case 0: return q - L.qmin;
    case 1: return L.qmax - q;
    case 2: return v - (-L.vmax);
    case 3: return L.vmax - v;
    case 4: return u - (-L.umax);
    default: return L.umax - u;
  }
}
// slack / dual direction of joint-limit row comp for the primal direction (dq, dv, du) (e.g. joint_torques_upper_limit.cpp:75-80)
__device__ __forceinline__ void con_direction(int comp, const LaneLimits& L, double q, double v, double u, double dq, double dv,
                                              double du, double slack, double dual, double barrier, double& dslack, double& ddual) {
  const double r = con_residual(comp, L, q, v, u, slack);
  const double dty = slack * dual - barrier;
  const double dx = comp < 2 ? dq : (comp < 4 ? dv : du);
  dslack = ((comp & 1) ? -dx : dx) - r;
  ddual = pdipm_dual_direction(slack, dual, dty, dslack);
}
__device__ __forceinline__ bool comp_active(int comp, int time_stage) {
  return comp < 2 ? pos_active(time_stage) : (comp < 4 ? vel_active(time_stage) : true);
}

__device__ __forceinline__ LaneLimits load_limits(const DevProblem& P, int lane) {
  return LaneLimits{P.q_min[lane], P.q_max[lane], P.v_max[lane], P.u_max[lane]};
}

// The two acceleration-limit components (JointAccelerationLowerLimit / UpperLimit, joint_acceleration_*_limit.cpp): rows of
// this lane's joint, k = 0 lower (residual amin - a + slack), k = 1 upper (a - amax + slack).  They are processed AFTER the
// six joint-limit components everywhere (the oracle's component order), from their own array XA.
struct AccRows {
  double sl[2], du[2], lim[2];
  bool on[2];
};
__device__ __forceinline__ AccRows acc_load(const DevProblem& P, const Layout& L, int stage, int g, int lane) {
  const double* XA = rec_ptr(L.XA, XA_NUM, L.G, stage, g);
  AccRows r;
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    r.on[k] = P.acc_enable[k] != 0;
    r.sl[k] = r.on[k] ? XA[k * SLOT] : 1.0;
    r.du[k] = r.on[k] ? XA[(2 + k) * SLOT] : 0.0;
  }
  r.lim[0] = P.a_min[lane];
  r.lim[1] = P.a_max[lane];
  return r;
}
__device__ __forceinline__ double acc_residual(const AccRows& r, int k, double a, double slack) {
  return k == 0 ? r.lim[0] - a + slack : a - r.lim[1] + slack;
}
// slack / dual direction of row k for the acceleration direction da (joint_acceleration_lower_limit.cpp:72-77)
__device__ __forceinline__ void acc_direction(const AccRows& r, int k, double a, double da, double barrier, double& dslack, double& ddual) {
  const double res = acc_residual(r, k, a, r.sl[k]);
  const double dty = r.sl[k] * r.du[k] - barrier;
  dslack = (k ? -da : da) - res;
  ddual = pdipm_dual_direction(r.sl[k], r.du[k], dty, dslack);
}

// warp-task decomposition of the per-stage kernels: task = (stage, group)
struct StageTask {
  int stage, g;
};
__device__ __forceinline__ StageTask stage_task(const Layout& L, int nstages) {
  long wt = static_cast<long>(blockIdx.x) * WARPS_PER_CTA + (threadIdx.x >> 5);
  const long ntask = static_cast<long>(nstages) * L.G;
  if (wt >= ntask) wt = ntask - 1;  // tail warps redo the last task: identical, idempotent stores
  return StageTask{static_cast<int>(wt / L.G), static_cast<int>(wt % L.G)};
}

// ---------------------------------------------------------------------------------------------
// k_init_constraints: slack and dual of every live row from its margin
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(CTA_THREADS) k_init_constraints(const DevProblem* __restrict__ Pp, Layout L,
                                                                  int stage_offset) {
  const DevProblem& P = *Pp;
  const int lane = lane_in_octet();
  const StageTask t = stage_task(L, L.N);
  double* X = rec_ptr(L.X, X_NUM, L.G, t.stage, t.g);
  const LaneLimits lim = load_limits(P, lane);
  const double q = X[X_Q * SLOT], v = X[X_V * SLOT], u = X[X_U * SLOT];
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    double sl = 0.0, du = 0.0;
    if (comp_active(c, t.stage + stage_offset) && lane < NV)
      pdipm_set_slack_and_dual_positive(con_margin(c, lim, q, v, u), P.barrier, sl, du);
    X[(X_SLACK + c) * SLOT] = sl;
    X[(X_DUAL + c) * SLOT] = du;
  }
  if (L.XA) {   // acceleration limits (time stage >= 0: every stage with controls)
    double* XA = rec_ptr(L.XA, XA_NUM, L.G, t.stage, t.g);
    const double a = X[X_A * SLOT];
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      double sl = 0.0, du = 0.0;
      if (P.acc_enable[k] && lane < NV)
        pdipm_set_slack_and_dual_positive(k == 0 ? a - P.a_min[lane] : P.a_max[lane] - a, P.barrier, sl, du);
      XA[k * SLOT] = sl;
      XA[(2 + k) * SLOT] = du;
    }
  }
}

// set one solution field of `nstages` stages from value[b][7] (broadcast: value[7])
__global__ void k_set_solution(Layout L, int field, const double* __restrict__ value, int broadcast, int nstages) {
  const long idx = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long total = static_cast<long>(nstages) * L.Bp * OCT;
  if (idx >= total) return;
  const int lane = static_cast<int>(idx & 7);
  const long t = idx >> 3;
  const int b = static_cast<int>(t % L.Bp);
  const int i = static_cast<int>(t / L.Bp);
  double val = 0.0;
  if (lane < NV && b < L.B) val = broadcast ? value[lane] : value[static_cast<size_t>(b) * NV + lane];
  L.X[elem_index(X_NUM, L.G, i, b, field, lane)] = val;
}

// ---------------------------------------------------------------------------------------------
// k_linearize
// ---------------------------------------------------------------------------------------------
// RESIDUAL_ONLY = true : computeKKTResidual + squaredNormKKTResidual (writes kkt_stage only)
// RESIDUAL_ONLY = false: linearizeOCP (writes condensed KKT blocks, residual, expansion data)
// BACKWARD_EULER = false: SplitUnOCP (forward Euler, stages 0..N-1 + terminal stage N)
// BACKWARD_EULER = true : SplitUnParNMPC / TerminalUnParNMPC (unocp/split_unparnmpc.hxx:69-101,141-174;
//                         terminal_unparnmpc.hxx:70-102,155-193): stages 1..N stored at index 0..N-1, the
//                         previous state of index 0 is the measured x0 = (q0, v0), index N-1 also carries
//                         the terminal cost; constraint masks use time stage index + 1
// TASK = true: + TimeVaryingTaskSpace6DCost (task_space_cost.cuh).  With the forward-Euler solver the kernel
//               then also covers the terminal stage N (TerminalOCP::linearizeOCP, ocp/terminal_ocp.hxx:50-66)
//               and leaves its dense Hessian / gradient in record N of KQ for k_riccati and k_expand.
// FUSED = true (UnOCPSolver, forward Euler only; k_update_linearize below): the task first applies the step of the iteration
//   that has just been expanded -- s += alpha_p d, slack += alpha_p dslack, dual += alpha_d ddual (unocp_solver.cpp:121-133) --
//   reading the old iterate / the direction from the records X, D, Xn, Dn (staged in shared memory by the TMA engine) and
//   writing the new iterate to L.X2 (ping-pong: the neighbour stage's warp still needs the OLD record of this stage), and then
//   linearises the NEW iterate for the next updateSolution call.  The linearisation does not depend on the measured state
//   (q0, v0 only enter the forward Riccati recursion), so the host keeps it until the iterate or the cost reference changes
//   (capi.cu: lin_valid).  The update's HBM stream hides under the FP64 work of the linearisation.
// X: this thread's pointer into the record of (stage i, group g) -- global memory, or the staged copy when FUSED.
// KKT (with FUSED): also leave the squared KKT norm of the NEW iterate's stage in L.kkt_stage -- the very numbers
// k_linearize<RESIDUAL_ONLY> would compute from it (same operations on the same values), so that a computeKKTResidual that
// follows the pipelined updateSolution (ocpbenchmarker::Convergence, an MPC loop that watches the KKT error) only has to sum them
// IREF: the cost references of the instance (common.cuh: cfg_ref, task_ref_row) instead of the problem's; the forward-Euler
// solver then also covers the terminal stage N and leaves diag(qf_weight), lq_N, lv_N in record N of KQ as TASK does, since
// the per-instance Riccati sweep (k_riccati<true>) takes the terminal blocks from there
template <bool RESIDUAL_ONLY, bool BACKWARD_EULER, bool TASK, bool FUSED, bool ACC = false, bool KKT = false, bool IREF = false>
__device__ __forceinline__ void linearize_task(const DevProblem& P, const Layout& L, const double* __restrict__ q0,
                                               const double* __restrict__ v0, double* tile, const int i, const int g,
                                               const double* X, const double* D, const double* Xnf, const double* Dn,
                                               const double ap, const double ad) {
  static_assert(!FUSED || (!RESIDUAL_ONLY && !BACKWARD_EULER), "the fused update exists for UnOCPSolver::updateSolution only");
  static_assert(!FUSED || !ACC, "the acceleration limits run through the literal kernel sequence");
  static_assert(!KKT || FUSED, "the KKT by-product exists for the fused update + linearisation only");
  const int lane = lane_in_octet();
  const int ts = BACKWARD_EULER ? i + 1 : i;   // time stage of the constraint masks
  const int b = g * 4 + ((threadIdx.x >> 3) & 3);
  const double dt = P.dt;
  const bool act = lane < NV;

  double q = X[X_Q * SLOT], v = X[X_V * SLOT], lmd = X[X_LMD * SLOT], gmm = X[X_GMM * SLOT];
  // the state of the fused update that the linearisation below continues with
  double fa = 0.0, fu = 0.0, fbeta = 0.0, fslack[NC], fdual[NC], fqn = 0.0, fvn = 0.0, flmdn = 0.0, fgmmn = 0.0;
  if (FUSED) {
    const int N = L.N;
    double* Xw = rec_ptr(L.X2, X_NUM, L.G, i, g);
    const double dlmd = D[D_LMD * SLOT], dgmm = D[D_GMM * SLOT], dq = D[D_Q * SLOT], dv = D[D_V * SLOT];
    double da = 0.0, du = 0.0, dbeta = 0.0, dqn = 0.0, dvn = 0.0, dlmdn = 0.0, dgmmn = 0.0;
    if (i != N) {
      fa = X[X_A * SLOT]; fu = X[X_U * SLOT]; fbeta = X[X_BETA * SLOT];
      da = D[D_A * SLOT]; du = D[D_U * SLOT]; dbeta = D[D_BETA * SLOT];
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        fslack[c] = X[(X_SLACK + c) * SLOT];
        fdual[c] = X[(X_DUAL + c) * SLOT];
      }
      fqn = Xnf[X_Q * SLOT]; fvn = Xnf[X_V * SLOT]; flmdn = Xnf[X_LMD * SLOT]; fgmmn = Xnf[X_GMM * SLOT];
      dqn = Dn[D_Q * SLOT]; dvn = Dn[D_V * SLOT]; dlmdn = Dn[D_LMD * SLOT]; dgmmn = Dn[D_GMM * SLOT];
    }
    // the padding lane keeps its (zero) record: k_update never touches it
    const double q_old = q, v_old = v, u_old = fu;
    if (act) {
      lmd = fma(ap, dlmd, lmd); gmm = fma(ap, dgmm, gmm); q = fma(ap, dq, q); v = fma(ap, dv, v);
    }
    Xw[X_LMD * SLOT] = lmd; Xw[X_GMM * SLOT] = gmm; Xw[X_Q * SLOT] = q; Xw[X_V * SLOT] = v;
    if (i != N) {
      if (act) {
        fa = fma(ap, da, fa); fu = fma(ap, du, fu); fbeta = fma(ap, dbeta, fbeta);
        fqn = fma(ap, dqn, fqn); fvn = fma(ap, dvn, fvn); flmdn = fma(ap, dlmdn, flmdn); fgmmn = fma(ap, dgmmn, fgmmn);
        const LaneLimits lim = load_limits(P, lane);
#pragma unroll
        for (int c = 0; c < NC; ++c) {
          if (!comp_active(c, i)) continue;
          const double sl = fslack[c], dl = fdual[c];
          double dslack, ddual;
          con_direction(c, lim, q_old, v_old, u_old, dq, dv, du, sl, dl, P.barrier, dslack, ddual);
          fslack[c] = fma(ap, dslack, sl);
          fdual[c] = fma(ad, ddual, dl);
        }
      }
      Xw[X_A * SLOT] = fa; Xw[X_U * SLOT] = fu; Xw[X_BETA * SLOT] = fbeta;
#pragma unroll
      for (int c = 0; c < NC; ++c) {
        Xw[(X_SLACK + c) * SLOT] = fslack[c];
        Xw[(X_DUAL + c) * SLOT] = fdual[c];
      }
    } else if (!TASK && !KKT && !IREF) {
      return;   // terminal stage: the update is all there is to do
    }
  }

  if ((RESIDUAL_ONLY || TASK || KKT || IREF) && !BACKWARD_EULER && i == L.N) {
    // TerminalOCP::linearizeOCP / computeKKTResidual + squaredNormKKTResidual (ocp/terminal_ocp.hxx:50-66,120-144)
    double lq = 0.0, lv = 0.0;
    lq += P.qf_weight[lane] * (q - cfg_ref<IREF, IREF_Q>(P, L, g, lane));
    lv += P.vf_weight[lane] * (v - cfg_ref<IREF, IREF_V>(P, L, g, lane));
    double hf[NV];
    if (TASK) {
      double R[9];
      V3 p;
      chain_fk(lane, act ? q : 0.0, P.model + lane * MODEL_STRIDE, R, p);
      TaskEval te;
      task_evaluate<true>(R, p, P.ee, task_ref_row<IREF>(L, i, b), te, P.task_enabled);
      task_share_columns(lane, te, tile);
      double gf;
      task_gradient_hessian(te, P.task_wf6, tile, gf, hf);
      lq += gf;
    }
    lq -= lmd;
    lv -= gmm;
    if (!act) { lq = 0.0; lv = 0.0; }
    if (RESIDUAL_ONLY || KKT) {
      const double e = oct_sum_ordered(lq * lq) + oct_sum_ordered(lv * lv);
      if (lane == 0) L.kkt_stage[static_cast<size_t>(i) * L.Bp + b] = e;
    }
    if (RESIDUAL_ONLY || (!TASK && !IREF)) {
      // (nothing else to do: residual only, or the fused update of a problem without a task-space cost)
    } else {
      // terminal record: rows of Qqq_N (slot = row, lane = column), lq_N, lv_N
      double* KQ = rec_ptr(L.KQ, KQ_NUM, L.G, i, g);
#pragma unroll
      for (int r = 0; r < NV; ++r) KQ[(KQ_QQ + r) * SLOT] = (r == lane ? P.qf_weight[lane] : 0.0) + (TASK && act ? hf[r] : 0.0);
      KQ[KQ_LQ * SLOT] = lq;
      KQ[KQ_LV * SLOT] = lv;
    }
    return;
  }

  const double a = FUSED ? fa : X[X_A * SLOT], u = FUSED ? fu : X[X_U * SLOT], beta = FUSED ? fbeta : X[X_BETA * SLOT];
  const bool last = BACKWARD_EULER && (i == L.N - 1);                // TerminalUnParNMPC
  const double* Xn = X + static_cast<size_t>(L.G) * (X_NUM * SLOT);  // next stage, same group
  // forward Euler: (q, v, lmd, gmm) of the next stage; backward Euler: (q, v) of the previous stage
  // (x0 for index 0) and (lmd, gmm) of the next stage (none for the last one)
  double qn, vn, lmdn = 0.0, gmmn = 0.0;
  if (FUSED) {
    qn = fqn; vn = fvn; lmdn = flmdn; gmmn = fgmmn;
  } else if (!BACKWARD_EULER) {
    qn = Xn[X_Q * SLOT]; vn = Xn[X_V * SLOT]; lmdn = Xn[X_LMD * SLOT]; gmmn = Xn[X_GMM * SLOT];
  } else {
    if (i == 0) {
      const size_t bi = static_cast<size_t>(b < L.B ? b : 0) * NV + (act ? lane : 0);
      qn = act ? q0[bi] : 0.0;
      vn = act ? v0[bi] : 0.0;
    } else {
      const double* Xp = X - static_cast<size_t>(L.G) * (X_NUM * SLOT);
      qn = Xp[X_Q * SLOT]; vn = Xp[X_V * SLOT];
    }
    if (!last) { lmdn = Xn[X_LMD * SLOT]; gmmn = Xn[X_GMM * SLOT]; }
  }
  double slack[NC], dual[NC];
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    slack[c] = FUSED ? fslack[c] : X[(X_SLACK + c) * SLOT];
    dual[c] = FUSED ? fdual[c] : X[(X_DUAL + c) * SLOT];
  }
  const LaneLimits lim = load_limits(P, lane);
  AccRows acc;
  if (ACC) acc = acc_load(P, L, i, g, act ? lane : 0);

  // ---- inverse dynamics and its derivatives (UnconstrainedDynamics::linearizeInverseDynamics) ----
  JointDyn J;
  double task_g = 0.0, task_gf = 0.0;   // JJ^T W diff of the stage / terminal task-space cost (this lane's entry)
  double task_h[NV], task_hf[NV];       // rows of JJ^T W JJ (this lane's column)
  {
    double R[9];
    V3 p;
    chain_fk(lane, q, P.model + lane * MODEL_STRIDE, R, p);
    if (TASK) {
      TaskEval te;
      task_evaluate<true>(R, p, P.ee, task_ref_row<IREF>(L, i, b), te, P.task_enabled);
      task_share_columns(lane, te, tile);
      task_gradient_hessian(te, P.task_w6, tile, task_g, task_h);
      if (last) task_gradient_hessian(te, P.task_wf6, tile, task_gf, task_hf);
      __syncwarp();   // the tile is reused by chain_pair_phase
    }
    chain_world_sweep_from_fk(lane, R, p, v, a, P.model + lane * MODEL_STRIDE, P.gravity, J);
  }
  double dqc[NV], dvc[NV], Mc[NV];
  chain_pair_phase(lane, J, tile, dqc, dvc, Mc);
  const double ID = J.tau - u;

  // ---- gradient of the Lagrangian (SURVEY A.2 steps 1-4) ----
  double lq = 0.0, lv = 0.0, la = 0.0, lu = 0.0;
  lq += dt * P.q_weight[lane] * (q - cfg_ref<IREF, IREF_Q>(P, L, g, lane));
  lv += dt * P.v_weight[lane] * (v - cfg_ref<IREF, IREF_V>(P, L, g, lane));
  la += dt * P.a_weight[lane] * a;
  lu += dt * P.u_weight[lane] * (u - cfg_ref<IREF, IREF_U>(P, L, g, lane));
  if (TASK) lq += dt * task_g;
  if (last) {   // + computeTerminalCostDerivatives (terminal_unparnmpc.hxx:84)
    lq += P.qf_weight[lane] * (q - cfg_ref<IREF, IREF_Q>(P, L, g, lane));
    lv += P.vf_weight[lane] * (v - cfg_ref<IREF, IREF_V>(P, L, g, lane));
    if (TASK) lq += task_gf;
  }
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (!comp_active(c, ts)) continue;
    const double g = dt * dual[c];
    const double sg = (c & 1) ? g : -g;
    if (c < 2) lq += sg; else if (c < 4) lv += sg; else lu += sg;
  }
  if (ACC) {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (!acc.on[k]) continue;
      const double g2 = dt * acc.du[k];
      la += k ? g2 : -g2;
    }
  }
  double Fq, Fv;
  if (!BACKWARD_EULER) {
    // stateequation::linearizeForwardEuler (ocp/state_equation.hxx:11-37,210-221)
    Fq = fma(dt, v, q - qn);
    Fv = fma(dt, a, v) - vn;
    lq += lmdn - lmd;
    lv += fma(dt, lmdn, gmmn) - gmm;
    la = fma(dt, gmmn, la);
  } else {
    // stateequation::linearizeBackwardEuler[Terminal] (ocp/state_equation.hxx:111-167,224-236)
    Fq = fma(dt, v, qn - q);
    Fv = fma(dt, a, vn - v);
    if (last) {
      lq -= lmd;
      lv += fma(dt, lmd, -gmm);
    } else {
      lq += lmdn - lmd;
      lv += fma(dt, lmd, -gmm) + gmmn;
    }
    la = fma(dt, gmm, la);
  }
  {
    double tq = 0.0, tv = 0.0, ta = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const double bk = oct_bcast(beta, k);
      tq = fma(dqc[k], bk, tq);
      tv = fma(dvc[k], bk, tv);
      ta = fma(Mc[k], bk, ta);
    }
    lq = fma(dt, tq, lq);
    lv = fma(dt, tv, lv);
    la = fma(dt, ta, la);
    lu = fma(-dt, beta, lu);
  }

  if (RESIDUAL_ONLY || KKT) {
    // SplitUnOCP::squaredNormKKTResidual (split_unocp.hxx:164-174), canonical order
    double e = 0.0;
    const double z = act ? 1.0 : 0.0;
    e += oct_sum_ordered(z * (lq * lq)) + oct_sum_ordered(z * (lv * lv));
    e += oct_sum_ordered(z * (la * la));
    e += oct_sum_ordered(z * (lu * lu));
    e += oct_sum_ordered(z * (Fq * Fq)) + oct_sum_ordered(z * (Fv * Fv));
    e += dt * dt * oct_sum_ordered(z * (ID * ID));
    double c2 = 0.0;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      if (!comp_active(c, ts)) continue;
      const double r = con_residual(c, lim, q, v, u, slack[c]);
      const double dl = slack[c] * dual[c] - P.barrier;
      c2 += oct_sum_ordered(z * (r * r)) + oct_sum_ordered(z * (dl * dl));
    }
    if (ACC) {
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (!acc.on[k]) continue;
        const double r = acc_residual(acc, k, a, acc.sl[k]);
        const double dl = acc.sl[k] * acc.du[k] - P.barrier;
        c2 += oct_sum_ordered(z * (r * r)) + oct_sum_ordered(z * (dl * dl));
      }
    }
    e += dt * dt * c2;
    if (lane == 0) L.kkt_stage[static_cast<size_t>(i) * L.Bp + b] = e;
    if (RESIDUAL_ONLY) return;
  }

  // ---- Hessian diagonals + constraint condensing (steps 5-6) ----
  double Qqq_d = dt * P.q_weight[lane];
  double Qvv_d = dt * P.v_weight[lane];
  double Qaa_d = dt * P.a_weight[lane];
  double Quu_d = dt * P.u_weight[lane];
  // off-diagonal entries of the un-condensed Qqq (task-space Gauss-Newton term only), row r of this lane's column
  double Qqq_off[NV];
#pragma unroll
  for (int r = 0; r < NV; ++r) Qqq_off[r] = 0.0;
  if (TASK) {
#pragma unroll
    for (int r = 0; r < NV; ++r) {
      const double hr = dt * task_h[r];
      if (r == lane) Qqq_d += hr;
      Qqq_off[r] = hr;
    }
  }
  if (last) {   // + computeTerminalCostHessian (terminal_unparnmpc.hxx:93)
    Qqq_d += P.qf_weight[lane];
    Qvv_d += P.vf_weight[lane];
    if (TASK) {
#pragma unroll
      for (int r = 0; r < NV; ++r) {
        if (r == lane) Qqq_d += task_hf[r];
        Qqq_off[r] += task_hf[r];
      }
    }
  }
  if (act) {
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      if (!comp_active(c, ts)) continue;
      const double r = con_residual(c, lim, q, v, u, slack[c]);
      const double dl = slack[c] * dual[c] - P.barrier;
      double h, g;
      pdipm_condense(dt, slack[c], dual[c], r, dl, h, g);
      const double sg = (c & 1) ? g : -g;
      if (c < 2) { Qqq_d += h; lq += sg; }
      else if (c < 4) { Qvv_d += h; lv += sg; }
      else { Quu_d += h; lu += sg; }
    }
    if (ACC) {
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (!acc.on[k]) continue;
        const double r = acc_residual(acc, k, a, acc.sl[k]);
        const double dl = acc.sl[k] * acc.du[k] - P.barrier;
        double h2, g2;
        pdipm_condense(dt, acc.sl[k], acc.du[k], r, dl, h2, g2);
        Qaa_d += h2;
        la += k ? g2 : -g2;
      }
    }
  } else {
    Quu_d = 0.0;
  }
  // ---- eliminate u (step 7, unconstrained_dynamics.hxx:68-94) ----
  const double lu_c = act ? fma(Quu_d, ID, lu) : 0.0;
  double ulq = lq, ulv = lv, ula = la;
  {
    double tq = 0.0, tv = 0.0, ta = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const double lk = oct_bcast(lu_c, k);
      tq = fma(dqc[k], lk, tq);
      tv = fma(dvc[k], lk, tv);
      ta = fma(Mc[k], lk, ta);
    }
    ulq += tq; ulv += tv; ula += ta;
  }
  double* KQ = rec_ptr(L.KQ, KQ_NUM, L.G, i, g);
  double* W = rec_ptr(L.W, W_NUM, L.G, i, g);
  KQ[KQ_FQ * SLOT] = Fq;
  KQ[KQ_FV * SLOT] = Fv;
  KQ[KQ_LA * SLOT] = ula;
  KQ[KQ_LQ * SLOT] = ulq;
  KQ[KQ_LV * SLOT] = ulv;
  W[W_ID * SLOT] = ID;
  W[W_LU * SLOT] = lu;
  W[W_QUU * SLOT] = Quu_d;

  // exchange the columns of dID/dq, dID/dv, M through the tile: tile[lane][0..20]
  double* mine = tile + lane * PAIR_TILE;
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    mine[k] = act ? dqc[k] : 0.0;
    mine[NV + k] = act ? dvc[k] : 0.0;
    mine[2 * NV + k] = act ? Mc[k] : 0.0;
  }
  __syncwarp();
  // expansion data in ROW layout (lane r holds row r): row r, col c = tile[c][r]
  const int ln = act ? lane : 0;
#pragma unroll
  for (int c = 0; c < NV; ++c) {
    const double* o = tile + c * PAIR_TILE;
    W[(W_DQ + c) * SLOT] = o[ln];
    W[(W_DV + c) * SLOT] = o[NV + ln];
    W[(W_M + c) * SLOT] = Mc[c];
  }
  // own columns scaled by diag(Quu):  D*[k] = Quu_k * d*[k][c]
  double Dq[NV], Dv[NV], Da[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    const double qk = oct_bcast(Quu_d, k);
    Dq[k] = qk * dqc[k];
    Dv[k] = qk * dvc[k];
    Da[k] = qk * Mc[k];
  }
  // Q_xy[r][c] = sum_k d_x[k][r] * (Quu_k d_y[k][c])   (+ un-condensed diagonals)
#pragma unroll
  for (int r = 0; r < NV; ++r) {
    const double* o = tile + r * PAIR_TILE;
    double qq = 0.0, qv = 0.0, vv = 0.0, aq = 0.0, av = 0.0, aa = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const double xq = o[k], xv = o[NV + k], xa = o[2 * NV + k];
      qq = fma(xq, Dq[k], qq);
      qv = fma(xq, Dv[k], qv);
      vv = fma(xv, Dv[k], vv);
      aq = fma(xa, Dq[k], aq);
      av = fma(xa, Dv[k], av);
      aa = fma(xa, Da[k], aa);
    }
    const bool diag = (r == lane);
    KQ[(KQ_QQ + r) * SLOT] = qq + (diag ? Qqq_d : (TASK && act ? Qqq_off[r] : 0.0));
    KQ[(KQ_QV + r) * SLOT] = qv;
    KQ[(KQ_VV + r) * SLOT] = vv + (diag ? Qvv_d : 0.0);
    KQ[(KQ_AQ + r) * SLOT] = aq;
    KQ[(KQ_AV + r) * SLOT] = av;
    KQ[(KQ_AA + r) * SLOT] = aa + (diag ? Qaa_d : 0.0);
  }
}


// ACC = true: + the two acceleration-limit components (their own array L.XA; the six-component instantiations are untouched)
template <bool RESIDUAL_ONLY, bool BACKWARD_EULER, bool TASK, bool ACC = false, bool IREF = false>
__global__ void __launch_bounds__(CTA_THREADS, LIN_MINB) k_linearize(const DevProblem* __restrict__ Pp, Layout L,
                                                                     const double* __restrict__ q0,
                                                                     const double* __restrict__ v0) {
  IDOCP_DYN_SMEM(double, smem);
  double* tile = smem + (threadIdx.x >> 3) * (OCT * PAIR_TILE);
  const StageTask t = stage_task(L, ((RESIDUAL_ONLY || TASK || IREF) && !BACKWARD_EULER) ? L.N + 1 : L.N);
  linearize_task<RESIDUAL_ONLY, BACKWARD_EULER, TASK, false, ACC, false, IREF>(*Pp, L, q0, v0, tile, t.stage, t.g,
                                                             rec_ptr(L.X, X_NUM, L.G, t.stage, t.g), nullptr, nullptr, nullptr, 1.0, 1.0);
}

// ---------------------------------------------------------------------------------------------
// k_step_min + k_update_linearize: the tail of a pipelined UnOCPSolver::updateSolution.
//   k_step_min: alpha_p, alpha_d = min over the N per-stage fraction-to-boundary minima (unocp_solver.cpp:114-115), one
//     thread per instance; `primal_override` (line search) replaces the primal step when given.
//   k_update_linearize: PERSISTENT, one CTA pair per SM; a warp walks over its (stage, group) tasks and, while it works on
//     one, the TMA engine stages the records of the next one (X 19 slots, D 7 slots, the first four slots of the next
//     stage's X and D, the two step sizes of the group) into the other half of the warp's shared-memory buffer
//     (cp.async.bulk + mbarrier, tma.cuh).  The non-persistent form of this fusion was slower than k_update + k_linearize
//     (0.70 vs 0.66 ms): with 2 warps per scheduler (254 registers) the extra loads sat exposed in front of the FP64 work
//     (long scoreboard 1.6 stall cycles per issue, profiles/r2b_ncu_full_iiwa14_unocp.txt).
// ---------------------------------------------------------------------------------------------
__global__ void k_step_min(Layout L, const double* __restrict__ primal_override) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= L.Bp) return;
  const int N = L.N;
  double ap = 1.0, ad = 1.0;
  for (int s = 0; s < N; ++s) {
    ap = fmin(ap, L.smin[static_cast<size_t>(s) * L.Bp + b]);
    ad = fmin(ad, L.smin[(static_cast<size_t>(N) + s) * L.Bp + b]);
  }
  const double amax = ap;
  if (primal_override) ap = primal_override[b];
  L.steps[b] = ap;                 // primal step applied (after the line search, if any)
  L.steps[L.Bp + b] = ad;          // dual step
  L.steps[2 * L.Bp + b] = amax;    // fraction-to-boundary primal step
  if (!(ap == ap) || !(ad == ad)) L.status[b] |= 2;
}

constexpr int UL_D = X_NUM, UL_XN = UL_D + D_NUM, UL_DN = UL_XN + 4, UL_ST = UL_DN + 4, UL_SLOTS = UL_ST + 1;
constexpr int UL_WARPS = 4;   // warps per CTA of the persistent kernel (24.3 KB of shared memory each)
constexpr int UL_THREADS = 32 * UL_WARPS;
constexpr int UL_OFF_BUF = UL_WARPS * 4 * OCT * PAIR_TILE;                         // doubles, after the pair tiles
constexpr int UL_OFF_BARS = UL_OFF_BUF + UL_WARPS * 2 * UL_SLOTS * SLOT;
constexpr int UL_SMEM_DOUBLES = UL_OFF_BARS + 2 * UL_WARPS;
static_assert(X_LMD == 0 && X_GMM == 1 && X_Q == 2 && X_V == 3 && D_LMD == 0 && D_GMM == 1 && D_Q == 2 && D_V == 3,
              "the next stage's (lmd, gmm, q, v) and their directions are the first four slots of a record");
static_assert((UL_OFF_BUF * 8) % 16 == 0, "TMA destinations are 16-byte aligned");

template <bool TASK, bool KKT = false, bool IREF = false>
__global__ void __launch_bounds__(UL_THREADS, UL_CTAS_PER_SM) k_update_linearize(const DevProblem* __restrict__ Pp, Layout L) {
  IDOCP_DYN_SMEM(double, smem);
  const int warp = threadIdx.x >> 5, wl = threadIdx.x & 31;
  double* tile = smem + (threadIdx.x >> 3) * (OCT * PAIR_TILE);
  double* bufs = smem + UL_OFF_BUF + warp * (2 * UL_SLOTS * SLOT);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + UL_OFF_BARS) + 2 * warp;
  const int N = L.N;
  const long ntask = static_cast<long>(N + 1) * L.G;
  const long nwarps = static_cast<long>(gridDim.x) * UL_WARPS;
  long wt = static_cast<long>(blockIdx.x) * UL_WARPS + warp;
  if (wl == 0) {
    tma_bar_init(&bars[0], 1);
    tma_bar_init(&bars[1], 1);
  }
  __syncwarp();
  auto issue = [&](long task, int buf) {
    const int st = static_cast<int>(task / L.G), g = static_cast<int>(task % L.G);
    double* dst = bufs + buf * (UL_SLOTS * SLOT);
    const double* xr = L.X + (static_cast<size_t>(st) * L.G + g) * (X_NUM * SLOT);
    const double* dr = L.D + (static_cast<size_t>(st) * L.G + g) * (D_NUM * SLOT);
    const bool nxt = st != N;
    tma_bar_expect(&bars[buf], (X_NUM + D_NUM) * SLOT * 8 + 2 * 32 + (nxt ? 8 * SLOT * 8 : 0));
    tma_load_1d(dst, xr, X_NUM * SLOT * 8, &bars[buf]);
    tma_load_1d(dst + UL_D * SLOT, dr, D_NUM * SLOT * 8, &bars[buf]);
    if (nxt) {
      tma_load_1d(dst + UL_XN * SLOT, xr + static_cast<size_t>(L.G) * (X_NUM * SLOT), 4 * SLOT * 8, &bars[buf]);
      tma_load_1d(dst + UL_DN * SLOT, dr + static_cast<size_t>(L.G) * (D_NUM * SLOT), 4 * SLOT * 8, &bars[buf]);
    }
    tma_load_1d(dst + UL_ST * SLOT, L.steps + static_cast<size_t>(g) * 4, 32, &bars[buf]);
    tma_load_1d(dst + UL_ST * SLOT + 4, L.steps + L.Bp + static_cast<size_t>(g) * 4, 32, &bars[buf]);
  };
  if (wl == 0 && wt < ntask) issue(wt, 0);
  for (int k = 0; wt < ntask; wt += nwarps, ++k) {
    const int buf = k & 1;
    __syncwarp();   // every lane is through with the previous task: its reads of the other buffer and of the pair tile
    if (wl == 0 && wt + nwarps < ntask) issue(wt + nwarps, buf ^ 1);
    tma_bar_wait(&bars[buf], (k >> 1) & 1);
    const double* rec = bufs + buf * (UL_SLOTS * SLOT);
    const int o4 = (threadIdx.x >> 3) & 3;
    linearize_task<false, false, TASK, true, false, KKT, IREF>(*Pp, L, nullptr, nullptr, tile, static_cast<int>(wt / L.G), static_cast<int>(wt % L.G),
                                             rec + wl, rec + UL_D * SLOT + wl, rec + UL_XN * SLOT + wl, rec + UL_DN * SLOT + wl,
                                             rec[UL_ST * SLOT + o4], rec[UL_ST * SLOT + 4 + o4]);
  }
}

// ---------------------------------------------------------------------------------------------
// k_riccati: backward Riccati recursion + forward recursion.  One octet per instance (one warp =
// one group of 4 instances); lane c owns column c.  Writes the gains / Riccati matrices to W and
// (dq, dv, da) to D; everything else of the direction is expanded in parallel by k_expand.
// ---------------------------------------------------------------------------------------------
// Three [8][RIC_TILE] tiles per octet carry a stage's cross-lane traffic (tX[col * RIC_TILE + row]).  Rows 0..7 are
// shared through __syncwarp; rows 8..14 of a lane's own column hold values only that lane reads.
//   tA: Qaa | la (rows 0..7), shared for the Cholesky; the lane's Qaq column (rows RIC_STASH..) until the solve and s.
//   tB: K (Kq rows 0..6, Kv rows 7..13) from the solve to the P update; then the new Pqq (rows 0..6) and Pvv (rows
//       RIC_STASH..) for their symmetrisation.  tA is therefore free when the next stage writes Qaa.
//   tC: the stage's Pqv (rows 0..6), read transposed as Pvq = Pqv^T through the whole next stage; the lane's Qav
//       column (rows RIC_STASH..), as Qaq in tA.
// Parking Qaq / Qav there keeps them out of registers across the Cholesky, which is what leaves the sweep spill-free.
constexpr int RIC_TILE = 17;               // odd stride (doubles) -> conflict-free transposed reads
constexpr int RIC_STASH = OCT;
constexpr int RIC_SMEM_PER_OCT = 3 * OCT * RIC_TILE;
static_assert(RIC_STASH + NV <= RIC_TILE && 2 * NV <= RIC_TILE, "tile rows");
// The condensed KKT record of (stage, group) is streamed into shared memory by the TMA engine one
// stage ahead of its use, in two halves with separate barriers so that each half-buffer can be
// re-armed at the first warp sync after every lane has read it:
//   half A = a-blocks + residual (slots AA, AQ, AV | FQ..LV: 21 + 5 slots), half X = x-blocks (QQ, QV, VV)
// The forward recursion streams (rows of K, k | Fq, Fv) of the stages through a 3-deep ring in the
// same per-warp region: its body is ~100 instructions per stage, i.e. pure memory latency otherwise.
constexpr int RIC_BUFA_SLOTS = 3 * NV + 5;
constexpr int RIC_BUFX_SLOTS = 3 * NV;
constexpr int RIC_RING = 3;
constexpr int RIC_RING_SLOTS = 2 * NV + 1 + 2;                                        // Kq, Kv, k | Fq, Fv
constexpr int RIC_WARP_SLOTS = (RIC_RING * RIC_RING_SLOTS > RIC_BUFA_SLOTS + RIC_BUFX_SLOTS)
                                   ? RIC_RING * RIC_RING_SLOTS : RIC_BUFA_SLOTS + RIC_BUFX_SLOTS;
// The sweep is a serial chain per warp, so its duration is (rounds of resident warps) x (one chain): 16384 instances = 4096
// warps need 4 rounds at 8 warps / SM (3.46 waves) but 3 at 10.  Measured (profiles/r2n_variants.txt): 10 warps / SM caps the
// kernel at 168 registers (three warps on one scheduler partition) with 600-800 B of spills: 0.423 -> 0.564 ms.  Kept at 4.
constexpr int RIC_WARPS = 4;
constexpr int RIC_THREADS = 32 * RIC_WARPS;
constexpr int RIC_OFF_STREAM = 4 * RIC_WARPS * RIC_SMEM_PER_OCT;                      // doubles
constexpr int RIC_OFF_BARS = RIC_OFF_STREAM + RIC_WARPS * RIC_WARP_SLOTS * SLOT;
constexpr int RIC_NBARS = 2 + RIC_RING;
constexpr int RIC_SMEM_DOUBLES = RIC_OFF_BARS + RIC_NBARS * RIC_WARPS;
// RIC_MINB CTAs per SM, each with its 1 KB of shared memory reserved by the system, within the SM's 228 KB
static_assert(RIC_MINB * (RIC_SMEM_DOUBLES * 8 + 1024) <= 228 * 1024, "k_riccati shared memory");
static_assert(KQ_AA == 0 && KQ_QQ == 3 * NV && KQ_FQ == 6 * NV && KQ_NUM == 6 * NV + 5, "record layout");
static_assert(W_KQ == 0 && W_KV == NV && W_K == 2 * NV && KQ_FV == KQ_FQ + 1, "record layout");

// TASK = true: the terminal Hessian / gradient come from record N of KQ (k_linearize<.., true> and the per-instance reference
// instantiations, which write the cost's reference there: this sweep itself reads no reference)
template <bool TASK>
__global__ void __launch_bounds__(RIC_THREADS, RIC_MINB) k_riccati(const DevProblem* __restrict__ Pp, Layout L,
                                                   const double* __restrict__ q0,
                                                   const double* __restrict__ v0) {
  IDOCP_DYN_SMEM(double, smem);
  const DevProblem& P = *Pp;
  const int lane = lane_in_octet();
  const int oct = threadIdx.x >> 3;
  double* tA = smem + oct * RIC_SMEM_PER_OCT;         // [8][RIC_TILE]
  double* tB = tA + OCT * RIC_TILE;                   // [8][RIC_TILE]
  double* tC = tB + OCT * RIC_TILE;                   // [8][RIC_TILE]
  int g = blockIdx.x * RIC_WARPS + (threadIdx.x >> 5);
  if (g >= L.G) g = L.G - 1;     // tail warps redo the last group (identical, idempotent stores)
  const int b = g * 4 + (oct & 3);
  const bool valid = b < L.B;    // padded instances (B <= b < Bp) are computed but never reported
  const int N = L.N;
  // TMA stream of the condensed KKT records (see RIC_BUFA_SLOTS)
  const int warp = threadIdx.x >> 5, wl = threadIdx.x & 31;
  double* stream = smem + RIC_OFF_STREAM + warp * (RIC_WARP_SLOTS * SLOT);
  const double* bufA = stream + wl;
  const double* bufX = stream + RIC_BUFA_SLOTS * SLOT + wl;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + RIC_OFF_BARS) + RIC_NBARS * warp;
  const double* kq_rec = L.KQ + static_cast<size_t>(g) * (KQ_NUM * SLOT);   // + stage * kstride
  const double* w_rec = L.W + static_cast<size_t>(g) * (W_NUM * SLOT);
  const size_t kstride = static_cast<size_t>(L.G) * (KQ_NUM * SLOT);
  if (wl == 0) {
#pragma unroll
    for (int k = 0; k < RIC_NBARS; ++k) tma_bar_init(&bars[k], 1);
  }
  __syncwarp();
  // the backward sweep re-issues into the same two buffers every stage: their shared addresses are converted once
  const smem_t s_bufa = smem_addr(stream), s_bufx = smem_addr(stream + RIC_BUFA_SLOTS * SLOT);
  const smem_t s_bara = smem_addr(&bars[0]), s_barx = smem_addr(&bars[1]);
  auto issue_half_a = [&](const double* src) {   // src: the stage's KQ record
    tma_bar_expect(s_bara, RIC_BUFA_SLOTS * SLOT * 8);
    tma_load_1d(s_bufa, src + KQ_AA * SLOT, 3 * NV * SLOT * 8, s_bara);
    tma_load_1d(s_bufa + 3 * NV * SLOT * 8, src + KQ_FQ * SLOT, 5 * SLOT * 8, s_bara);
  };
  auto issue_half_x = [&](const double* src) {
    tma_bar_expect(s_barx, RIC_BUFX_SLOTS * SLOT * 8);
    tma_load_1d(s_bufx, src + KQ_QQ * SLOT, RIC_BUFX_SLOTS * SLOT * 8, s_barx);
  };
  auto issue_forward = [&](int stage) {   // ring entry stage % RIC_RING
    const int e = stage % RIC_RING;
    double* dst = stream + e * (RIC_RING_SLOTS * SLOT);
    tma_bar_expect(&bars[2 + e], RIC_RING_SLOTS * SLOT * 8);
    tma_load_1d(dst, w_rec + static_cast<size_t>(stage) * L.G * (W_NUM * SLOT) + W_KQ * SLOT, (2 * NV + 1) * SLOT * 8,
                &bars[2 + e]);
    tma_load_1d(dst + (2 * NV + 1) * SLOT, kq_rec + static_cast<size_t>(stage) * L.G * (KQ_NUM * SLOT) + KQ_FQ * SLOT,
                2 * SLOT * 8, &bars[2 + e]);
  };
  const double* kq_stage = kq_rec + static_cast<size_t>(N - 1) * kstride;   // record of the current stage
  if (wl == 0) {
    issue_half_a(kq_stage);
    issue_half_x(kq_stage);
  }
  uint32_t phase = 0;
  const double dt = P.dt;
  const double dt2 = dt * dt;
  const bool act = lane < NV;
  const int ln = act ? lane : 0;
  int chol_fail = 0;
  const size_t xstride = static_cast<size_t>(L.G) * (X_NUM * SLOT);
  const size_t wstride = static_cast<size_t>(L.G) * (W_NUM * SLOT);
  const size_t dstride = static_cast<size_t>(L.G) * (D_NUM * SLOT);

  // ---- terminal stage: P_N = diag(qf, vf), s_N = -l_N (unriccati_recursion.cpp:39-47) ----
  double Pqq[NV], Pqv[NV], Pvv[NV], sq, sv;   // Pvq = Pqv^T is read from tile C
  {
    const double* X = rec_ptr(L.X, X_NUM, L.G, N, g);
    const double q = X[X_Q * SLOT], v = X[X_V * SLOT], lmd = X[X_LMD * SLOT], gmm = X[X_GMM * SLOT];
    double lq = 0.0, lv = 0.0;
    lq += P.qf_weight[lane] * (q - P.q_ref[lane]);
    lv += P.vf_weight[lane] * (v - P.v_ref[lane]);
    lq -= lmd;
    lv -= gmm;
    sq = -lq;
    sv = -lv;
#pragma unroll
    for (int r = 0; r < NV; ++r) {
      Pqq[r] = (r == lane) ? P.qf_weight[lane] : 0.0;
      Pvv[r] = (r == lane) ? P.vf_weight[lane] : 0.0;
      Pqv[r] = 0.0;
      tC[lane * RIC_TILE + r] = 0.0;
    }
    if (TASK) {
      const double* KQN = rec_ptr(L.KQ, KQ_NUM, L.G, N, g);
#pragma unroll
      for (int r = 0; r < NV; ++r) Pqq[r] = KQN[(KQ_QQ + r) * SLOT];
      sq = -KQN[KQ_LQ * SLOT];
      sv = -KQN[KQ_LV * SLOT];
    }
    __syncwarp();
  }

  // ---- backward recursion ----
  double* W = rec_ptr(L.W, W_NUM, L.G, N - 1, g);
  for (int i = N - 1; i >= 0; --i, W -= wstride, kq_stage -= kstride, phase ^= 1) {
    tma_bar_wait(&bars[0], phase);
    // factorizeKKTMatrix, a-blocks (backward_unriccati_recursion_factorizer.hxx:44-53); the
    // x-blocks are folded into the P update below (same operation order per entry)
    double Qaa[NV];
#pragma unroll
    for (int r = 0; r < NV; ++r) {
      const double pvq = tC[r * RIC_TILE + ln];
      double qaq = bufA[(KQ_AQ + r) * SLOT], qav = bufA[(KQ_AV + r) * SLOT];
      qaq = fma(dt, pvq, qaq);
      qav = fma(dt2, pvq, qav);
      qav = fma(dt, Pvv[r], qav);
      Qaa[r] = fma(dt2, Pvv[r], bufA[(KQ_AA + r) * SLOT]);
      tA[lane * RIC_TILE + RIC_STASH + r] = qaq;
      tC[lane * RIC_TILE + RIC_STASH + r] = qav;
    }
    const double Fq = bufA[(3 * NV + 0) * SLOT], Fv = bufA[(3 * NV + 1) * SLOT];
    double la = bufA[(3 * NV + 2) * SLOT];
    const double lq = bufA[(3 * NV + 3) * SLOT], lv = bufA[(3 * NV + 4) * SLOT];
    // products of the OLD P with Fx (used by la and by the s recursion)
    double pqqF = 0.0, pvqF = 0.0, pqvF = 0.0, pvvF = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      const double fq = oct_bcast(Fq, k), fv = oct_bcast(Fv, k);
      pqqF = fma(Pqq[k], fq, pqqF);                  // (Pqq Fq)_c   (row c = column c, symmetric)
      pvqF = fma(tC[k * RIC_TILE + ln], fv, pvqF);   // (Pqv Fv)_c
      pqvF = fma(Pqv[k], fq, pqvF);                  // (Pqv^T Fq)_c
      pvvF = fma(Pvv[k], fv, pvvF);                  // (Pvv Fv)_c
    }
    if (TASK && i == N - 1) {
      // the dense terminal Pqq_N = Qqq_N (Gauss-Newton term of the task-space cost) is not bitwise symmetric:
      // (Pqq Fq)_c needs ROW c, which each lane reads from the terminal record itself
      const double* rec = L.KQ + (static_cast<size_t>(N) * L.G + g) * (KQ_NUM * SLOT) + (oct & 3) * OCT;
      pqqF = 0.0;
#pragma unroll
      for (int k = 0; k < NV; ++k) pqqF = fma(rec[(KQ_QQ + ln) * SLOT + k], oct_bcast(Fq, k), pqqF);
    }
    la = fma(dt, pqvF, la);
    la = fma(dt, pvvF, la);
    la = fma(-dt, sv, la);
    // next s (uses the OLD P): backward_unriccati_recursion_factorizer.hxx:78-88, all but the Qa^T k terms, which
    // are subtracted once k is known: two values instead of eight stay live across the Cholesky
    double nsq = sq, nsv;
    nsq -= pqqF; nsq -= pvqF;
    nsv = fma(dt, nsq, sv); nsv -= pqvF; nsv -= pvvF;
    nsq -= lq; nsv -= lv;
    // share Qaa (tile A: tA[col][row]) and la
#pragma unroll
    for (int r = 0; r < NV; ++r) tA[lane * RIC_TILE + r] = Qaa[r];
    tA[lane * RIC_TILE + NV] = la;
    __syncwarp();                              // tile A shared, half A consumed by every lane
    if (wl == 0 && i > 0) issue_half_a(kq_stage - kstride);
    // Cholesky of Qaa (lower triangle), redundantly in every lane: Lm[col][row], row >= col
    double Lm[NV][NV];
    double rdiag[NV];
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      double x = tA[k * RIC_TILE + k];
#pragma unroll
      for (int j = 0; j < k; ++j) x = fma(-Lm[j][k], Lm[j][k], x);
      if (!canon_pivot_ok(x)) chol_fail = 1;
      rdiag[k] = canon_rsqrt(x);   // the diagonal L_kk = x rdiag[k] itself is never read
#pragma unroll
      for (int r = k + 1; r < NV; ++r) {
        double y = tA[k * RIC_TILE + r];
#pragma unroll
        for (int j = 0; j < k; ++j) y = fma(-Lm[j][r], Lm[j][k], y);
        Lm[k][r] = y * rdiag[k];
      }
    }
    // K = -Qaa^-1 [Qaq Qav] (own columns), k = -Qaa^-1 la (all lanes)
    double Kq[NV], Kv[NV], kk[NV];
#pragma unroll
    for (int r = 0; r < NV; ++r) {
      double y1 = tA[lane * RIC_TILE + RIC_STASH + r], y2 = tC[lane * RIC_TILE + RIC_STASH + r], y3 = tA[r * RIC_TILE + NV];
#pragma unroll
      for (int j = 0; j < r; ++j) {
        y1 = fma(-Lm[j][r], Kq[j], y1); y2 = fma(-Lm[j][r], Kv[j], y2); y3 = fma(-Lm[j][r], kk[j], y3);
      }
      Kq[r] = y1 * rdiag[r]; Kv[r] = y2 * rdiag[r]; kk[r] = y3 * rdiag[r];
    }
#pragma unroll
    for (int r = NV - 1; r >= 0; --r) {
      double y1 = Kq[r], y2 = Kv[r], y3 = kk[r];
#pragma unroll
      for (int j = r + 1; j < NV; ++j) {
        y1 = fma(-Lm[r][j], Kq[j], y1); y2 = fma(-Lm[r][j], Kv[j], y2); y3 = fma(-Lm[r][j], kk[j], y3);
      }
      Kq[r] = y1 * rdiag[r]; Kv[r] = y2 * rdiag[r]; kk[r] = y3 * rdiag[r];
    }
#pragma unroll
    for (int r = 0; r < NV; ++r) { Kq[r] = -Kq[r]; Kv[r] = -Kv[r]; kk[r] = -kk[r]; }
    // GK = Qaa K (full Qaa, as the reference multiplies the full matrix).  Qaa is read from tile A again: without the
    // compiler barrier the Cholesky's 28 loads are reused here, which keeps them live across both solves and spills
    asm volatile("" ::: "memory");
    double GKq[NV], GKv[NV];
#pragma unroll
    for (int r = 0; r < NV; ++r) {
      double t1 = 0.0, t2 = 0.0;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const double gq = tA[k * RIC_TILE + r];
        t1 = fma(gq, Kq[k], t1);
        t2 = fma(gq, Kv[k], t2);
      }
      GKq[r] = t1; GKv[r] = t2;
    }
    // share K (tile B: tB[col][0..6] = Kq[:,col], tB[col][7..13] = Kv[:,col])
#pragma unroll
    for (int r = 0; r < NV; ++r) { tB[lane * RIC_TILE + r] = Kq[r]; tB[lane * RIC_TILE + NV + r] = Kv[r]; }
    // rest of the next s
    {
      double t5 = 0.0, t6 = 0.0;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        t5 = fma(tA[lane * RIC_TILE + RIC_STASH + k], kk[k], t5);
        t6 = fma(tC[lane * RIC_TILE + RIC_STASH + k], kk[k], t6);
      }
      nsq -= t5; nsv -= t6;
    }
    __syncwarp();                              // tile B shared
    // F-blocks of factorizeKKTMatrix (:34-43) + P = Qxx - K^T (Qaa K) (:64-75), row by row
    tma_bar_wait(&bars[1], phase);
#pragma unroll
    for (int r = 0; r < NV; ++r) {
      double Qqq = bufX[(0 * NV + r) * SLOT];
      double Qqv = bufX[(1 * NV + r) * SLOT];
      double Qvv = bufX[(2 * NV + r) * SLOT];
      Qqq += Pqq[r];
      Qqv = fma(dt, Pqq[r], Qqv);
      Qqv += Pqv[r];
      Qvv = fma(dt2, Pqq[r], Qvv);
      Qvv = fma(dt, Pqv[r], Qvv);
      Qvv = fma(dt, tC[r * RIC_TILE + ln], Qvv);
      Qvv += Pvv[r];
      double tqq = 0.0, tqv = 0.0, tvv = 0.0;
#pragma unroll
      for (int k = 0; k < NV; ++k) {
        const double kq = tB[r * RIC_TILE + k], kv = tB[r * RIC_TILE + NV + k];
        tqq = fma(kq, GKq[k], tqq);
        tqv = fma(kq, GKv[k], tqv);
        tvv = fma(kv, GKv[k], tvv);
      }
      Pqq[r] = Qqq - tqq;
      Pqv[r] = Qqv - tqv;
      Pvv[r] = Qvv - tvv;
    }
    // K in row layout for the forward pass: lane r gets Kq[r][c] = tB[c][r]
#pragma unroll
    for (int c = 0; c < NV; ++c) {
      W[(W_KQ + c) * SLOT] = tB[c * RIC_TILE + ln];
      W[(W_KV + c) * SLOT] = tB[c * RIC_TILE + NV + ln];
    }
    double k_own = kk[0];                      // kk[ln] by selects: a lane-dependent index would put kk in local memory
#pragma unroll
    for (int r = 1; r < NV; ++r) k_own = (ln == r) ? kk[r] : k_own;
    W[W_K * SLOT] = k_own;
    __syncwarp();                              // half X, K (tile B) and the old Pvq (tile C) consumed by every lane
    if (wl == 0 && i > 0) issue_half_x(kq_stage - kstride);
    // one round trip for the new P: Pqv stays in tile C as the next stage's Pvq; Pqq and Pvv are symmetrised
#pragma unroll
    for (int r = 0; r < NV; ++r) {
      tB[lane * RIC_TILE + r] = Pqq[r];
      tB[lane * RIC_TILE + RIC_STASH + r] = Pvv[r];
      tC[lane * RIC_TILE + r] = Pqv[r];
    }
    __syncwarp();
#pragma unroll
    for (int r = 0; r < NV; ++r) {
      Pqq[r] = 0.5 * (Pqq[r] + tB[r * RIC_TILE + ln]);               // (Pqq[r][c] + Pqq[c][r]) / 2
      Pvv[r] = 0.5 * (Pvv[r] + tB[r * RIC_TILE + RIC_STASH + ln]);
    }
    sq = nsq; sv = nsv;
#pragma unroll
    for (int r = 0; r < NV; ++r) {
      W[(W_PQQ + r) * SLOT] = Pqq[r];
      W[(W_PQV + r) * SLOT] = Pqv[r];
      W[(W_PVV + r) * SLOT] = Pvv[r];
    }
    W[W_SQ * SLOT] = sq;
    W[W_SV * SLOT] = sv;
  }

  // ---- forward recursion: da = K dx + k, dx+ = Fx + A dx + B da (split_unriccati_factorizer.hxx:49-57) ----
  double dq, dv;
  {
    const double* X0 = rec_ptr(L.X, X_NUM, L.G, 0, g);
    const size_t bi = static_cast<size_t>(valid ? b : 0) * NV + ln;
    dq = q0[bi] - X0[X_Q * SLOT];
    dv = v0[bi] - X0[X_V * SLOT];
    if (!act) { dq = 0.0; dv = 0.0; }
  }
  double* D = rec_ptr(L.D, D_NUM, L.G, 0, g);
  // the gains were written by this warp through the generic proxy: order those writes before the
  // TMA engine reads them back, then fill the ring
  tma_fence_global_writes();
  __syncwarp();
  if (wl == 0) {
    for (int i = 0; i < RIC_RING && i < N; ++i) issue_forward(i);
  }
  for (int i = 0; i < N; ++i) {
    const int e = i % RIC_RING;
    tma_bar_wait(&bars[2 + e], (i / RIC_RING) & 1);
    const double* ring = stream + e * (RIC_RING_SLOTS * SLOT) + wl;
    double Kr[2 * NV];
#pragma unroll
    for (int c = 0; c < 2 * NV; ++c) Kr[c] = ring[c * SLOT];
    const double kr = ring[2 * NV * SLOT];
    const double Fq = ring[(2 * NV + 1) * SLOT], Fv = ring[(2 * NV + 2) * SLOT];
    __syncwarp();                              // ring entry is in registers: refill it
    if (wl == 0 && i + RIC_RING < N) issue_forward(i + RIC_RING);
    double acc = 0.0;
#pragma unroll
    for (int c = 0; c < NV; ++c) acc = fma(Kr[c], oct_bcast(dq, c), acc);
#pragma unroll
    for (int c = 0; c < NV; ++c) acc = fma(Kr[NV + c], oct_bcast(dv, c), acc);
    const double da = acc + kr;
    D[D_Q * SLOT] = dq;
    D[D_V * SLOT] = dv;
    D[D_A * SLOT] = da;
    double ndq = Fq + dq;
    double ndv = Fv + dv;
    ndq = fma(dt, dv, ndq);
    ndv = fma(dt, da, ndv);
    dq = act ? ndq : 0.0;
    dv = act ? ndv : 0.0;
    D += dstride;
  }
  D[D_Q * SLOT] = dq;   // terminal stage
  D[D_V * SLOT] = dv;
  const int any_fail = __shfl_xor_sync(FULL, chol_fail, 1, OCT) | chol_fail;
  if (lane == 0 && valid && any_fail) L.status[b] |= 1;
  (void)xstride;
}

// ---------------------------------------------------------------------------------------------
// k_expand: per (instance, stage): costate direction dlmd, dgmm = P dx - s; condensed direction
// du = ID + dID [dq,dv,da], dbeta = (lu + Quu du)/dt; slack/dual directions; per-stage
// fraction-to-boundary minima.  Terminal stage: costate only (P_N = diag, s_N recomputed).
// ---------------------------------------------------------------------------------------------
// PARNMPC = true (UnParNMPCSolver): N stages, none terminal, the costate direction is already in D
// (k_parnmpc_forward_parallel); only the condensed direction and the step sizes are computed.
// TASK = true: the terminal P_N = Qqq_N is dense (record N of KQ)
// IREF = true: the terminal gradient from the instance's cost reference (common.cuh: cfg_ref)
constexpr int EXP_TILE = 9;   // odd stride (doubles) of the Pqv transpose tile of k_expand
template <bool PARNMPC, bool TASK, bool ACC = false, bool IREF = false>
__global__ void __launch_bounds__(CTA_THREADS, EXP_MINB) k_expand(const DevProblem* __restrict__ Pp, Layout L, int stage_offset) {
  const DevProblem& P = *Pp;
  const int lane = lane_in_octet();
  const StageTask t = stage_task(L, PARNMPC ? L.N : L.N + 1);
  const int i = t.stage;
  const int b = t.g * 4 + ((threadIdx.x >> 3) & 3);
  const int N = L.N;
  const bool act = lane < NV;
  const double* X = rec_ptr(L.X, X_NUM, L.G, i, t.g);
  double* D = rec_ptr(L.D, D_NUM, L.G, i, t.g);
  const double dq = D[D_Q * SLOT], dv = D[D_V * SLOT];
  if (!PARNMPC && i == N) {
    const double q = X[X_Q * SLOT], v = X[X_V * SLOT], lmd = X[X_LMD * SLOT], gmm = X[X_GMM * SLOT];
    double lq = 0.0, lv = 0.0;
    lq += P.qf_weight[lane] * (q - cfg_ref<IREF, IREF_Q>(P, L, t.g, lane));
    lv += P.vf_weight[lane] * (v - cfg_ref<IREF, IREF_V>(P, L, t.g, lane));
    lq -= lmd;
    lv -= gmm;
    double dlmd = P.qf_weight[lane] * dq; dlmd -= -lq;
    double dgmm = P.vf_weight[lane] * dv; dgmm -= -lv;
    if (TASK) {
      // dlmd = Pqq_N dq - sq with row `lane` of the dense Pqq_N (each lane reads its own row) and sq = -lq_N
      const double* rec = L.KQ + (static_cast<size_t>(N) * L.G + t.g) * (KQ_NUM * SLOT) + ((threadIdx.x >> 3) & 3) * OCT;
      const int row = act ? lane : 0;
      double t1 = 0.0;
#pragma unroll
      for (int k = 0; k < NV; ++k) t1 = fma(rec[(KQ_QQ + row) * SLOT + k], oct_bcast(dq, k), t1);
      dlmd = t1;
      dlmd -= -rec[KQ_LQ * SLOT + row];
      if (!act) dlmd = 0.0;
    }
    D[D_LMD * SLOT] = dlmd;
    D[D_GMM * SLOT] = dgmm;
    return;
  }
  const double* W = rec_ptr(L.W, W_NUM, L.G, i, t.g);
  const double da = D[D_A * SLOT];
  // the state / slack / dual loads go out with the W loads, before the stores through D (which would fence them)
  double xq = 0.0, xv = 0.0, xu = 0.0, slk[NC], dul[NC];
  if (act) {
    xq = X[X_Q * SLOT]; xv = X[X_V * SLOT]; xu = X[X_U * SLOT];
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const bool on = comp_active(c, i + stage_offset);
      slk[c] = on ? X[(X_SLACK + c) * SLOT] : 1.0;
      dul[c] = on ? X[(X_DUAL + c) * SLOT] : 0.0;
    }
  }
  AccRows acc;
  double xa = 0.0;
  if (ACC) { acc = acc_load(P, L, i, t.g, act ? lane : 0); xa = X[X_A * SLOT]; }
  // Every W slot of the record goes out before the first use: the kernel is a pure HBM stream, and 12 warps per SM
  // with ~60 loads in flight each (166 registers) reach 6.4 TB/s where 20 warps at 95 registers, loading as the FMA
  // chains consume, reached 5.4 TB/s (0.287 -> 0.249 ms; register CAPS of 80 / 72 for more warps: 0.36 / 0.35 ms).
  double w_pqq[NV], w_pvq[NV], w_pqv[NV], w_pvv[NV], w_dq[NV], w_dv[NV], w_m[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) {
    if (!PARNMPC) {
      w_pqq[k] = W[(W_PQQ + k) * SLOT];
      w_pqv[k] = W[(W_PQV + k) * SLOT]; w_pvv[k] = W[(W_PVV + k) * SLOT];
    }
    w_dq[k] = W[(W_DQ + k) * SLOT]; w_dv[k] = W[(W_DV + k) * SLOT]; w_m[k] = W[(W_M + k) * SLOT];
  }
  if (!PARNMPC) {
    // column c of Pvq = row c of Pqv: transposed through the octet's tile (stride 9: conflict-free both ways)
    __shared__ double pvq_tile[OCTETS_PER_CTA * OCT * EXP_TILE];
    double* tile = pvq_tile + (threadIdx.x >> 3) * (OCT * EXP_TILE);
#pragma unroll
    for (int k = 0; k < NV; ++k) tile[k * EXP_TILE + lane] = w_pqv[k];     // tile[row k][column lane]
    __syncwarp();
    const int ln = act ? lane : 0;
#pragma unroll
    for (int k = 0; k < NV; ++k) w_pvq[k] = tile[ln * EXP_TILE + k];       // Pqv[lane][k]
  }
  const double w_sq = PARNMPC ? 0.0 : W[W_SQ * SLOT], w_sv = PARNMPC ? 0.0 : W[W_SV * SLOT];
  const double w_id = W[W_ID * SLOT], w_quu = W[W_QUU * SLOT], w_lu = W[W_LU * SLOT];
  double dqk[NV], dvk[NV];
#pragma unroll
  for (int k = 0; k < NV; ++k) { dqk[k] = oct_bcast(dq, k); dvk[k] = oct_bcast(dv, k); }
  // costate direction (split_unriccati_factorizer.hxx:60-68)
  double dlmd = 0.0, dgmm = 0.0;
  if (!PARNMPC) {
    double t1 = 0.0, t2 = 0.0, t3 = 0.0, t4 = 0.0;
#pragma unroll
    for (int k = 0; k < NV; ++k) {
      t1 = fma(w_pqq[k], dqk[k], t1);
      t2 = fma(w_pvq[k], dvk[k], t2);
      t3 = fma(w_pqv[k], dqk[k], t3);
      t4 = fma(w_pvv[k], dvk[k], t4);
    }
    dlmd = t1; dlmd += t2; dlmd -= w_sq;
    dgmm = t3; dgmm += t4; dgmm -= w_sv;
  }
  // du = ID + dID/dq dq + dID/dv dv + M da ; dbeta = (lu + Quu du) / dt
  double du, dbeta;
  {
    double acc = w_id;
    double s = 0.0;
#pragma unroll
    for (int c = 0; c < NV; ++c) s = fma(w_dq[c], dqk[c], s);
    acc += s;
    s = 0.0;
#pragma unroll
    for (int c = 0; c < NV; ++c) s = fma(w_dv[c], dvk[c], s);
    acc += s;
    s = 0.0;
#pragma unroll
    for (int c = 0; c < NV; ++c) s = fma(w_m[c], oct_bcast(da, c), s);
    acc += s;
    du = acc;
    dbeta = fma(w_quu, du, w_lu) / P.dt;
  }
  if (!PARNMPC) {
    D[D_LMD * SLOT] = dlmd;
    D[D_GMM * SLOT] = dgmm;
  }
  D[D_U * SLOT] = du;
  D[D_BETA * SLOT] = dbeta;
  // slack / dual directions and fraction-to-boundary
  double min_p = 1.0, min_d = 1.0;
  if (act) {
    const LaneLimits lim = load_limits(P, lane);
    const double q = xq, v = xv, u = xu;
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      if (!comp_active(c, i + stage_offset)) continue;
      const double sl = slk[c];
      const double dl = dul[c];
      double dslack, ddual;
      con_direction(c, lim, q, v, u, dq, dv, du, sl, dl, P.barrier, dslack, ddual);
      min_p = pdipm_fraction_row(P.fraction_rate, sl, dslack, min_p);
      min_d = pdipm_fraction_row(P.fraction_rate, dl, ddual, min_d);
    }
    if (ACC) {
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        if (!acc.on[k]) continue;
        double dslack, ddual;
        acc_direction(acc, k, xa, da, P.barrier, dslack, ddual);
        min_p = pdipm_fraction_row(P.fraction_rate, acc.sl[k], dslack, min_p);
        min_d = pdipm_fraction_row(P.fraction_rate, acc.du[k], ddual, min_d);
      }
    }
  }
  min_p = oct_min(min_p);
  min_d = oct_min(min_d);
  if (lane == 0) {
    L.smin[static_cast<size_t>(i) * L.Bp + b] = min_p;
    L.smin[(static_cast<size_t>(N) + i) * L.Bp + b] = min_d;
  }
}

// ---------------------------------------------------------------------------------------------
// k_update: alpha = min over stages (unocp_solver.cpp:114-115), then s += alpha_p d,
// slack += alpha_p dslack, dual += alpha_d ddual (unocp_solver.cpp:121-133; split_solution.hxx:
// 215-239; constraints_impl.hxx:181-196).  dslack / ddual are recomputed from (s, slack, dual, d)
// instead of being stored.  `primal_override` (line search) replaces the primal step when given.
// ---------------------------------------------------------------------------------------------
// `nstages` = N + 1 with the terminal stage at index N (UnOCPSolver) or N without one (UnParNMPCSolver,
// src/unocp/unparnmpc_solver.cpp:88-101).
__global__ void __launch_bounds__(CTA_THREADS) k_update(const DevProblem* __restrict__ Pp, Layout L, int stage_offset,
                                                        const double* __restrict__ primal_override, int nstages) {
  const DevProblem& P = *Pp;
  const int lane = lane_in_octet();
  // read-modify-write kernel: tail warps must NOT redo a task (whole warps exit together)
  if (static_cast<long>(blockIdx.x) * WARPS_PER_CTA + (threadIdx.x >> 5) >= static_cast<long>(nstages) * L.G) return;
  const StageTask t = stage_task(L, nstages);
  const int i = t.stage;
  const int b = t.g * 4 + ((threadIdx.x >> 3) & 3);
  const int N = L.N;
  double* X = rec_ptr(L.X, X_NUM, L.G, i, t.g);
  const double* D = rec_ptr(L.D, D_NUM, L.G, i, t.g);
  // every load of the record is issued before the first store and before the step-size reduction (lane 7 reads its padding slot): stores through X would otherwise fence the later loads
  // (the compiler cannot prove that X and D do not overlap) and the kernel would pay one DRAM round trip per field
  const double lmd = X[X_LMD * SLOT], gmm = X[X_GMM * SLOT], q = X[X_Q * SLOT], v = X[X_V * SLOT];
  const double dlmd = D[D_LMD * SLOT], dgmm = D[D_GMM * SLOT], dq = D[D_Q * SLOT], dv = D[D_V * SLOT];
  double a = 0.0, u = 0.0, beta = 0.0, da = 0.0, du = 0.0, dbeta = 0.0, slk[NC], dul[NC];
  if (i != N) {
    a = X[X_A * SLOT]; u = X[X_U * SLOT]; beta = X[X_BETA * SLOT];
    da = D[D_A * SLOT]; du = D[D_U * SLOT]; dbeta = D[D_BETA * SLOT];
#pragma unroll
    for (int c = 0; c < NC; ++c) {
      const bool on = comp_active(c, i + stage_offset);
      slk[c] = on ? X[(X_SLACK + c) * SLOT] : 1.0;
      dul[c] = on ? X[(X_DUAL + c) * SLOT] : 0.0;
    }
  }
  // min over the N per-stage minima, lanes striding over the stages
  double ap = 1.0, ad = 1.0;
  for (int s = lane; s < N; s += OCT) {
    ap = fmin(ap, L.smin[static_cast<size_t>(s) * L.Bp + b]);
    ad = fmin(ad, L.smin[(static_cast<size_t>(N) + s) * L.Bp + b]);
  }
  ap = oct_min(ap);
  ad = oct_min(ad);
  const double amax = ap;
  if (primal_override) ap = primal_override[b];
  if (i == 0 && lane == 0) {
    L.steps[b] = ap;                 // primal step applied (after the line search, if any)
    L.steps[L.Bp + b] = ad;          // dual step
    L.steps[2 * L.Bp + b] = amax;    // fraction-to-boundary primal step
    if (!(ap == ap) || !(ad == ad)) L.status[b] |= 2;
  }
  if (lane >= NV) return;
  X[X_LMD * SLOT] = fma(ap, dlmd, lmd);
  X[X_GMM * SLOT] = fma(ap, dgmm, gmm);
  X[X_Q * SLOT] = fma(ap, dq, q);
  X[X_V * SLOT] = fma(ap, dv, v);
  if (i == N) return;
  X[X_A * SLOT] = fma(ap, da, a);
  X[X_U * SLOT] = fma(ap, du, u);
  X[X_BETA * SLOT] = fma(ap, dbeta, beta);
  const LaneLimits lim = load_limits(P, lane);
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (!comp_active(c, i + stage_offset)) continue;
    const double sl = slk[c], dl = dul[c];
    double dslack, ddual;
    con_direction(c, lim, q, v, u, dq, dv, du, sl, dl, P.barrier, dslack, ddual);
    X[(X_SLACK + c) * SLOT] = fma(ap, dslack, sl);
    X[(X_DUAL + c) * SLOT] = fma(ad, ddual, dl);
  }
  if (L.XA) {
    const AccRows acc = acc_load(P, L, i, t.g, lane);
    double* XA = rec_ptr(L.XA, XA_NUM, L.G, i, t.g);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (!acc.on[k]) continue;
      double dslack, ddual;
      acc_direction(acc, k, a, da, P.barrier, dslack, ddual);
      XA[k * SLOT] = fma(ap, dslack, acc.sl[k]);
      XA[(2 + k) * SLOT] = fma(ad, ddual, acc.du[k]);
    }
  }
}

// KKTError = sqrt(sum over stages in ascending order) (unocp_solver.cpp:190-202)
__global__ void k_kkt_sum(Layout L, int nstages) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= L.Bp) return;
  double e = 0.0;
  for (int i = 0; i < nstages; ++i) e += L.kkt_stage[static_cast<size_t>(i) * L.Bp + b];
  L.kkt_err[b] = sqrt(e);
}

}  // namespace idocp_b200
