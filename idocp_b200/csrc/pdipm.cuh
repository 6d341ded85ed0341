// pdipm.cuh -- the per-row rules of the primal-dual interior point method (idocp constraints/pdipm.hxx) that every
// constraint row of both solver families follows.  A row has a slack, a dual, and per Newton step its primal residual
// and duality (slack * dual - barrier).  The kernels of both families call these; the oracle restates them on its own.
#pragma once

namespace idocp_b200 {

// pdipm::SetSlackAndDualPositive (pdipm.hxx:13-23): slack = margin pushed above the barrier in steps of the barrier,
// dual = barrier / slack.  The iteration bound keeps a margin of -inf (or a huge violation in the initial guess) from
// hanging the stream; the oracle has the same bound.
__device__ __forceinline__ void pdipm_set_slack_and_dual_positive(double margin, double barrier, double& slack, double& dual) {
  int guard = 0;
  while (margin < barrier && guard < (1 << 20)) { margin += barrier; ++guard; }
  slack = margin;
  dual = barrier / margin;
}

// pdipm::ComputeDualDirection (pdipm.hxx:76-81)
__device__ __forceinline__ double pdipm_dual_direction(double slack, double dual, double duality, double dslack) {
  return -fma(dual, dslack, duality) / slack;
}

// condenseSlackAndDual of one row (e.g. joint_position_lower_limit.cpp:64-74): Hessian term h = dt dual / slack and the
// unsigned gradient term g = dt (dual residual - duality) / slack; the two divisions share one reciprocal
__device__ __forceinline__ void pdipm_condense(double dt, double slack, double dual, double residual, double duality, double& h,
                                               double& g) {
  const double rs = 1.0 / slack;
  h = (dt * dual) * rs;
  g = (dt * fma(dual, residual, -duality)) * rs;
}

// pdipm::FractionToBoundary (pdipm.hxx:52-73) for one row: only fractions strictly inside (0, 1) count
__device__ __forceinline__ double pdipm_fraction_row(double rate, double x, double dx, double cur) {
  const double f = -rate * (x / dx);
  if (f > 0.0 && f < 1.0 && f < cur) return f;
  return cur;
}

}  // namespace idocp_b200
