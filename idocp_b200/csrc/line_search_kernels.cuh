// line_search_kernels.cuh -- batched filter line search of the unconstrained solvers.
//
//   UnLineSearch::computeCostAndViolation  src/line_search/unline_search.cpp:56-84
//   SplitUnOCP::stageCost / constraintViolation  include/idocp/unocp/split_unocp.hxx:177-217
//   TerminalOCP::terminalCost            include/idocp/ocp/terminal_ocp.hxx:89-95
//
// The lock-step rounds of line_search_filter.cuh:
//   k_ls_eval (stage-parallel cost / violation of the trial step)  ->  k_ls_filter (per instance)
// Finished instances drop out warp-uniformly.  Sums run over ascending stage index.
#pragma once
#include "unocp_kernels.cuh"
#include "line_search_filter.cuh"

namespace idocp_b200 {

struct LineSearchLayout {
  double* cost = nullptr;      // [N+1][Bp] per-stage cost of the current trial
  double* viol = nullptr;      // [N][Bp]   per-stage constraint violation
  LsFilter f;                  // Bp instances
};

// min over stages of the per-stage fraction-to-boundary minima (unocp_solver.cpp:114-115);
// executed by one octet (lanes stride over the stages), every lane gets the result
__device__ __forceinline__ void octet_step_sizes(const Layout& L, int b, int lane, double& ap, double& ad) {
  ap = 1.0; ad = 1.0;
  for (int s = lane; s < L.N; s += OCT) {
    ap = fmin(ap, L.smin[static_cast<size_t>(s) * L.Bp + b]);
    ad = fmin(ad, L.smin[(static_cast<size_t>(L.N) + s) * L.Bp + b]);
  }
  ap = oct_min(ap);
  ad = oct_min(ad);
}

// does instance b take part in this round?  mode 0: filter initialisation (empty filters only)
__device__ __forceinline__ bool ls_participates(const LineSearchLayout& LS, int b, int B, int mode) {
  if (b >= B) return false;
  return mode == 0 ? (LS.f.n[b] == 0) : (LS.f.state[b] == 0);
}

// ---------------------------------------------------------------------------------------------
// k_ls_eval: cost and constraint violation of s + alpha d for every (instance, stage).
// ---------------------------------------------------------------------------------------------
// TASK = true: + TimeVaryingTaskSpace6DCost::computeStageCost / computeTerminalCost
// (src/cost/time_varying_task_space_6d_cost.cpp:68-90)
// BACKWARD_EULER = true: UnParNMPCSolver (src/line_search/unline_search.cpp:87-122; split_unparnmpc.hxx:177-224,
// terminal_unparnmpc.hxx:196-227): N stages, the last one adds the terminal cost, the state-equation defect
// uses the TRIAL previous stage (x0 for index 0), the last stage's reference time is t + N dt (table row N)
// IREF = true: the instance's cost references (common.cuh: cfg_ref, task_ref_row)
template <bool TASK, bool BACKWARD_EULER, bool IREF = false>
__global__ void __launch_bounds__(CTA_THREADS) k_ls_eval(const DevProblem* __restrict__ Pp, Layout L,
                                                         LineSearchLayout LS, int mode, int stage_offset,
                                                         const double* __restrict__ q0, const double* __restrict__ v0) {
  const DevProblem& P = *Pp;
  const int lane = lane_in_octet();
  const StageTask t = stage_task(L, BACKWARD_EULER ? L.N : L.N + 1);
  const int i = t.stage;
  const int b = t.g * 4 + ((threadIdx.x >> 3) & 3);
  const bool part = ls_participates(LS, b, L.B, mode);
  if (!__any_sync(FULL, part)) return;  // warp-uniform: nothing to do for this group
  const int N = L.N;
  const double dt = P.dt;
  const bool act = lane < NV;
  const double z = act ? 1.0 : 0.0;
  const double alpha = (mode == 0 || !part) ? 0.0 : LS.f.alpha[b];
  const double* X = rec_ptr(L.X, X_NUM, L.G, i, t.g);
  const double* D = rec_ptr(L.D, D_NUM, L.G, i, t.g);
  const double q = X[X_Q * SLOT], v = X[X_V * SLOT];
  const double dq = D[D_Q * SLOT], dv = D[D_V * SLOT];
  // UnLineSearch::computeTrySolution (unline_search.hpp:125-133): q, v, a, u only
  const double qt = fma(alpha, dq, q), vt = fma(alpha, dv, v);
  if (!BACKWARD_EULER && i == N) {
    // TerminalOCP::terminalCost -> ConfigurationSpaceCost::computeTerminalCost (configuration_space_cost.cpp:259-273)
    double l = 0.0;
    l += oct_sum_ordered(z * (P.qf_weight[lane] * (qt - cfg_ref<IREF, IREF_Q>(P, L, t.g, lane)) * (qt - cfg_ref<IREF, IREF_Q>(P, L, t.g, lane))));
    l += oct_sum_ordered(z * (P.vf_weight[lane] * (vt - cfg_ref<IREF, IREF_V>(P, L, t.g, lane)) * (vt - cfg_ref<IREF, IREF_V>(P, L, t.g, lane))));
    double tc = 0.5 * l;
    if (TASK) {
      double R[9];
      V3 p;
      chain_fk(lane, act ? qt : 0.0, P.model + lane * MODEL_STRIDE, R, p);
      TaskEval te;
      task_evaluate<false>(R, p, P.ee, task_ref_row<IREF>(L, N, b), te, P.task_enabled);
      tc += 0.5 * task_weighted_sqnorm(te, P.task_wf6);
    }
    if (lane == 0 && part) LS.cost[static_cast<size_t>(N) * L.Bp + b] = tc;
    return;
  }
  const double a = X[X_A * SLOT], u = X[X_U * SLOT];
  const double da = D[D_A * SLOT], du = D[D_U * SLOT];
  const double at = fma(alpha, da, a), ut = fma(alpha, du, u);
  const size_t xs = static_cast<size_t>(L.G) * (X_NUM * SLOT), ds = static_cast<size_t>(L.G) * (D_NUM * SLOT);
  const bool last = BACKWARD_EULER && (i == N - 1);
  // neighbour state of the state equation at the trial point: next stage (forward Euler) / previous stage or
  // the measured x0 (backward Euler)
  double qnt, vnt;
  if (!BACKWARD_EULER) {
    qnt = fma(alpha, D[ds + D_Q * SLOT], X[xs + X_Q * SLOT]);
    vnt = fma(alpha, D[ds + D_V * SLOT], X[xs + X_V * SLOT]);
  } else if (i == 0) {
    const size_t bi = static_cast<size_t>(b < L.B ? b : 0) * NV + (act ? lane : 0);
    qnt = act ? q0[bi] : 0.0;
    vnt = act ? v0[bi] : 0.0;
  } else {
    qnt = fma(alpha, *(D - ds + D_Q * SLOT), *(X - xs + X_Q * SLOT));
    vnt = fma(alpha, *(D - ds + D_V * SLOT), *(X - xs + X_V * SLOT));
  }
  // ---- SplitUnOCP::stageCost (split_unocp.hxx:177-196) ----
  double l = 0.0;
  l += oct_sum_ordered(z * (P.q_weight[lane] * (qt - cfg_ref<IREF, IREF_Q>(P, L, t.g, lane)) * (qt - cfg_ref<IREF, IREF_Q>(P, L, t.g, lane))));
  l += oct_sum_ordered(z * (P.v_weight[lane] * (vt - cfg_ref<IREF, IREF_V>(P, L, t.g, lane)) * (vt - cfg_ref<IREF, IREF_V>(P, L, t.g, lane))));
  l += oct_sum_ordered(z * (P.a_weight[lane] * at * at));
  l += oct_sum_ordered(z * (P.u_weight[lane] * (ut - cfg_ref<IREF, IREF_U>(P, L, t.g, lane)) * (ut - cfg_ref<IREF, IREF_U>(P, L, t.g, lane))));
  double cost = 0.5 * dt * l;
  double R[9];
  V3 p;
  chain_fk(lane, act ? qt : 0.0, P.model + lane * MODEL_STRIDE, R, p);
  TaskEval te;
  if (TASK) {
    task_evaluate<false>(R, p, P.ee, task_ref_row<IREF>(L, last ? N : i, b), te, P.task_enabled);
    cost += 0.5 * dt * task_weighted_sqnorm(te, P.task_w6);
  }
  if (last) {   // TerminalUnParNMPC::stageCost: + computeTerminalCost
    double lf = 0.0;
    lf += oct_sum_ordered(z * (P.qf_weight[lane] * (qt - cfg_ref<IREF, IREF_Q>(P, L, t.g, lane)) * (qt - cfg_ref<IREF, IREF_Q>(P, L, t.g, lane))));
    lf += oct_sum_ordered(z * (P.vf_weight[lane] * (vt - cfg_ref<IREF, IREF_V>(P, L, t.g, lane)) * (vt - cfg_ref<IREF, IREF_V>(P, L, t.g, lane))));
    double tc = 0.5 * lf;
    if (TASK) tc += 0.5 * task_weighted_sqnorm(te, P.task_wf6);
    cost += tc;
  }
  const LaneLimits lim = load_limits(P, lane);
  double bar = 0.0, c1 = 0.0;
#pragma unroll
  for (int c = 0; c < NC; ++c) {
    if (!comp_active(c, i + stage_offset)) continue;
    const double sl = act ? X[(X_SLACK + c) * SLOT] : 1.0;
    // slack direction of the Newton step (recomputed, as in k_expand / k_update)
    const double r0 = con_residual(c, lim, q, v, u, sl);
    const double dx = c < 2 ? dq : (c < 4 ? dv : du);
    const double dslack = ((c & 1) ? -dx : dx) - r0;
    const double st = alpha > 0.0 ? fma(alpha, dslack, sl) : sl;
    // pdipm::CostBarrier (pdipm.hxx:84-87): -barrier * sum(log(slack))
    const double lg = oct_sum_ordered(z * canon_log(st));
    bar += -P.barrier * lg;
    // primal residual at the trial point with the un-stepped slack (split_unocp.hxx:208)
    const double rt = con_residual(c, lim, qt, vt, ut, sl);
    c1 += oct_sum_ordered(z * fabs(rt));
  }
  if (L.XA) {   // acceleration limits (the oracle's component order: after the six joint limits)
    const AccRows acc = acc_load(P, L, i, t.g, act ? lane : 0);
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      if (!acc.on[k]) continue;
      const double sl = act ? acc.sl[k] : 1.0;
      const double r0 = acc_residual(acc, k, a, sl);
      const double dslack = (k ? -da : da) - r0;
      const double st = alpha > 0.0 ? fma(alpha, dslack, sl) : sl;
      bar += -P.barrier * oct_sum_ordered(z * canon_log(st));
      c1 += oct_sum_ordered(z * fabs(acc_residual(acc, k, at, sl)));
    }
  }
  cost += dt * bar;
  // ---- SplitUnOCP::constraintViolation (split_unocp.hxx:199-217) ----
  const double Fq = BACKWARD_EULER ? fma(dt, vt, qnt - qt) : fma(dt, vt, qt - qnt);
  const double Fv = BACKWARD_EULER ? fma(dt, at, vnt - vt) : fma(dt, at, vt) - vnt;
  JointDyn J;
  chain_world_sweep_from_fk(lane, R, p, act ? vt : 0.0, act ? at : 0.0, P.model + lane * MODEL_STRIDE, P.gravity, J);
  const double ID = J.tau - ut;
  double viol = 0.0;
  viol += oct_sum_ordered(z * fabs(Fq)) + oct_sum_ordered(z * fabs(Fv));
  viol += dt * oct_sum_ordered(z * fabs(ID));
  viol += dt * c1;
  if (lane == 0 && part) {
    LS.cost[static_cast<size_t>(i) * L.Bp + b] = cost;
    LS.viol[static_cast<size_t>(i) * L.Bp + b] = viol;
  }
}

// sum of the per-stage values in ascending stage order (UnLineSearch::totalCosts / totalViolations)
// ncost = N + 1 (UnOCPSolver: N stages + terminal) or N (UnParNMPCSolver)
__device__ __forceinline__ void ls_totals(const Layout& L, const LineSearchLayout& LS, int b, int ncost, double& cost,
                                          double& viol) {
  double cs = 0.0, vs = 0.0;
  for (int i = 0; i < ncost; ++i) {
    cs += LS.cost[static_cast<size_t>(i) * L.Bp + b];
    if (i < L.N) vs += LS.viol[static_cast<size_t>(i) * L.Bp + b];
  }
  cost = cs; viol = vs;
}

// k_ls_filter: one thread per instance, ls_filter_round from the fraction-to-boundary step alpha_max
__global__ void k_ls_filter(Layout L, LineSearchLayout LS, int mode, int ncost) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= L.B) return;
  ls_filter_round(LS.f, b, mode, L.steps[2 * L.Bp + b], L.status,
                  [&](double& cost, double& viol) { ls_totals(L, LS, b, ncost, cost, viol); });
}

// max step sizes before the line search (stored for k_ls_filter mode 0): steps[2][b] = alpha_max
__global__ void __launch_bounds__(CTA_THREADS) k_ls_begin(Layout L) {
  const int lane = lane_in_octet();
  int g = blockIdx.x * WARPS_PER_CTA + (threadIdx.x >> 5);
  if (g >= L.G) g = L.G - 1;
  const int b = g * 4 + ((threadIdx.x >> 3) & 3);
  double ap, ad;
  octet_step_sizes(L, b, lane, ap, ad);
  if (lane == 0) L.steps[2 * L.Bp + b] = ap;
}

}  // namespace idocp_b200
