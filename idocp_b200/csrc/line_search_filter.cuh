// line_search_filter.cuh -- the per-instance filter line search both solver families run.
//
//   LineSearchFilter::isAccepted / augment       src/line_search/line_search_filter.cpp:34-65
//   UnLineSearch::computeStepSize                 include/idocp/line_search/unline_search.hpp:62-91
//   LineSearch::computeStepSize                   include/idocp/line_search/line_search.hpp:62-93
//
// The reference backtracks one instance with a data-dependent trip count (alpha *= 0.75 while alpha > 0.05, at most 11
// trials from alpha = 1).  Here every instance of the batch carries its own (alpha, state, filter); the host launches a
// fixed number of lock-step rounds  (family's cost / violation kernel) -> (family's filter kernel, thread per instance)
// and finished instances drop out.  The filter kernels of both families are ls_filter_round around their own totals.
#pragma once
#include <cstddef>

#include "../../include/idocp_b200.h"

namespace idocp_b200 {

constexpr int LS_FILTER_CAP = 256;     // entries per instance (the reference's vector is unbounded)
constexpr int LS_MAX_TRIALS = 11;      // 0.75^10 > 0.05 >= 0.75^11
constexpr double LS_RATE = 0.75;       // unline_search.hpp:25
constexpr double LS_MIN_STEP = 0.05;   // unline_search.hpp:26
constexpr double LS_COST_REDUCTION = 0.005;        // line_search_filter.hpp:16
constexpr double LS_CONSTRAINTS_REDUCTION = 0.005; // line_search_filter.hpp:17

struct LsFilter {
  double* alpha = nullptr;  // [n] current / final primal step size
  int* state = nullptr;     // [n] 0 = searching, 1 = finished
  int* n = nullptr;         // [n] filter sizes
  double* cost = nullptr;   // [n][LS_FILTER_CAP]
  double* viol = nullptr;   // [n][LS_FILTER_CAP]
};

// LineSearchFilter::augment (line_search_filter.cpp:48-65)
__device__ __forceinline__ void filter_augment(const LsFilter& F, int b, double cost, double viol, int* status) {
  double* fc = F.cost + static_cast<size_t>(b) * LS_FILTER_CAP;
  double* fv = F.viol + static_cast<size_t>(b) * LS_FILTER_CAP;
  int n = F.n[b], w = 0;
  for (int i = 0; i < n; ++i) {
    if (cost <= fc[i] && viol <= fv[i]) continue;  // dominated entry erased
    fc[w] = fc[i]; fv[w] = fv[i]; ++w;
  }
  if (w < LS_FILTER_CAP) {
    fc[w] = cost - LS_COST_REDUCTION * viol;
    fv[w] = (1 - LS_CONSTRAINTS_REDUCTION) * viol;
    ++w;
  } else {
    status[b] |= IDOCP_B200_STATUS_FILTER_FULL;  // entry dropped
  }
  F.n[b] = w;
}
// LineSearchFilter::isAccepted (:34-45)
__device__ __forceinline__ bool filter_accepts(const LsFilter& F, int b, double cost, double viol) {
  const double* fc = F.cost + static_cast<size_t>(b) * LS_FILTER_CAP;
  const double* fv = F.viol + static_cast<size_t>(b) * LS_FILTER_CAP;
  const int n = F.n[b];
  for (int i = 0; i < n; ++i)
    if (cost >= fc[i] && viol >= fv[i]) return false;
  return true;
}

// one filter round of instance b; totals(cost, viol) sums the family's per-stage values of the point just evaluated
//  mode 0: augment an empty filter with the current point, then start the search at amax (finished at once if amax is
//          not above LS_MIN_STEP)
//  mode 1: one backtracking decision
template <typename Totals>
__device__ __forceinline__ void ls_filter_round(const LsFilter& F, int b, int mode, double amax, int* status, Totals totals) {
  if (mode == 0) {
    if (F.n[b] == 0) {
      double cost, viol;
      totals(cost, viol);
      filter_augment(F, b, cost, viol, status);
    }
    const bool go = amax > LS_MIN_STEP;
    F.alpha[b] = go ? amax : LS_MIN_STEP;
    F.state[b] = go ? 0 : 1;
    return;
  }
  if (F.state[b] != 0) return;
  double cost, viol;
  totals(cost, viol);
  if (filter_accepts(F, b, cost, viol)) {
    filter_augment(F, b, cost, viol, status);
    F.state[b] = 1;
    return;
  }
  const double an = F.alpha[b] * LS_RATE;
  if (an > LS_MIN_STEP) {
    F.alpha[b] = an;
  } else {
    F.alpha[b] = LS_MIN_STEP;
    F.state[b] = 1;
  }
}

// LineSearchFilter::clear of the first `count` instances
__global__ void k_ls_clear(int* n, int count) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < count) n[b] = 0;
}

}  // namespace idocp_b200
