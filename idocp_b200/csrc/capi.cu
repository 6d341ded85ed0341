// capi.cu -- C-ABI of the engine (include/idocp_b200.h): handle management, host<->device
// staging and kernel launches.  Compiled by nvcc for sm_100a into libidocp_b200.so.
// (tests/emu builds the same file with g++ against a SIMT emulator -- test infrastructure.)
#ifdef IDOCP_B200_EMU
#include "cuda_emu.h"
#else
#include <cuda_runtime.h>
#endif

#include <algorithm>
#include <array>
#include <cmath>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/idocp_b200.h"
#include "model_iiwa14.h"
#include "unocp_kernels.cuh"
#include "line_search_kernels.cuh"
#include "unparnmpc_kernels.cuh"
#include "fb_kernels.cuh"

using namespace idocp_b200;

#ifdef IDOCP_B200_EMU
#define IDOCP_LAUNCH(h, cls, kern, grid, block, smem, ...)                                   \
  do {                                                                                       \
    (h)->begin_kernel(cls);                                                                  \
    emu::launch(dim3(grid), dim3(block), (smem), [&]() { kern(__VA_ARGS__); });              \
    (h)->end_kernel(cls);                                                                    \
  } while (0)
#else
#define IDOCP_LAUNCH(h, cls, kern, grid, block, smem, ...)                                   \
  do {                                                                                       \
    (h)->begin_kernel(cls);                                                                  \
    auto kfn_ = kern;                                                                        \
    kfn_<<<(grid), (block), (smem), (h)->stream>>>(__VA_ARGS__);                             \
    (h)->end_kernel(cls);                                                                    \
  } while (0)
#endif

static thread_local std::string g_last_error;
static int fail(int code, const std::string& msg) {
  g_last_error = msg;
  return code;
}
#define CUDA_OK(expr)                                                                        \
  do {                                                                                       \
    cudaError_t e_ = (expr);                                                                 \
    if (e_ != cudaSuccess)                                                                   \
      return fail(IDOCP_B200_CUDA_ERROR, std::string(#expr) + ": " + cudaGetErrorString(e_)); \
  } while (0)

enum KernelClass { KC_LINEARIZE = 0, KC_RICCATI, KC_EXPAND, KC_UPDATE, KC_KKT, KC_MISC, KC_PARNMPC_COARSE,
                   KC_PARNMPC_CORR, KC_LINESEARCH, KC_FB_LINEARIZE, KC_FB_CONDENSE, KC_FB_RICCATI, KC_FB_FORWARD, KC_FB_EXPAND, KC_FB_UPDATE,
                   KC_FB_KKT, KC_UPDATE_LINEARIZE, KC_STEP_MIN, KC_NUM };
static const char* kKernelClassNames[KC_NUM] = {"linearize", "riccati", "expand", "update", "kkt", "misc",
                                                "parnmpc_coarse", "parnmpc_correction", "line_search", "fb_robot", "fb_condense",
                                                "fb_riccati_backward", "fb_riccati_forward", "fb_expand", "fb_update", "fb_kkt",
                                                "update_linearize", "step_min"};

// What every solver handle of both families owns: its device and stream, the device allocations, the CUDA events, the
// launch counter and the per-kernel-class event timing.  open() / release() are the one lifecycle of a handle; the
// *_sync / *_launch_count / *_stream / *_set_profiling / *_get_profile entry points of both families forward here.
struct DeviceHandle {
  int device = 0;
  cudaStream_t stream = nullptr;
  long long launches = 0;
  // profiling: 0 off, 1 = CUDA events recorded around every launch on the launching stream and
  // resolved lazily in get_profile (no host synchronisation inside the timed region)
  int profiling = 0;
  struct ProfRec { int cls; cudaEvent_t e0, e1; };
  std::vector<ProfRec> prof_recs;
  std::vector<cudaEvent_t> event_pool;
  double prof_ms[KC_NUM] = {0};
  long long prof_calls[KC_NUM] = {0};
  cudaEvent_t cur_e0 = nullptr;
  std::vector<void*> allocs;

  cudaEvent_t take_event() {
    if (!event_pool.empty()) { cudaEvent_t e = event_pool.back(); event_pool.pop_back(); return e; }
    cudaEvent_t e = nullptr;
    cudaEventCreate(&e);
    return e;
  }
  // The caller's q / v may be pinned host memory that it rewrites as soon as the call returns (the normal MPC loop): the
  // host waits for the H2D copies just enqueued (an event behind them), not for the kernels enqueued after them.
  cudaEvent_t copies_done = nullptr;
  int mark_uploads() {            // right behind the copies
    if (!copies_done && cudaEventCreate(&copies_done) != cudaSuccess) return -1;
    return cudaEventRecord(copies_done, stream) == cudaSuccess ? 0 : -1;
  }
  int wait_for_uploads() {        // after the call's kernels have been enqueued: the wait overlaps their execution
    return (copies_done && cudaEventSynchronize(copies_done) != cudaSuccess) ? -1 : 0;
  }
  void resolve_profile() {
    if (prof_recs.empty()) return;
    cudaStreamSynchronize(stream);
    for (auto& r : prof_recs) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, r.e0, r.e1);
      prof_ms[r.cls] += ms;
      prof_calls[r.cls] += 1;
      event_pool.push_back(r.e0);
      event_pool.push_back(r.e1);
    }
    prof_recs.clear();
  }
  void begin_kernel(int) {
    ++launches;
    if (profiling) {
      cur_e0 = take_event();
      cudaEventRecord(cur_e0, stream);
    }
  }
  void end_kernel(int cls) {
    if (profiling) {
      cudaEvent_t e1 = take_event();
      cudaEventRecord(e1, stream);
      prof_recs.push_back(ProfRec{cls, cur_e0, e1});
    }
  }
  template <typename T>
  int alloc(T** p, size_t count) {
    void* q = nullptr;
    if (cudaMalloc(&q, count * sizeof(T)) != cudaSuccess) return -1;
    cudaMemsetAsync(q, 0, count * sizeof(T), stream);
    allocs.push_back(q);
    *p = static_cast<T*>(q);
    return 0;
  }

  // device count and index checks, then the handle's non-blocking stream on `device`
  int open(int device) {
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev <= 0)
      return fail(IDOCP_B200_NO_DEVICE, "no CUDA device available (there is no CPU fallback)");
    if (device < 0 || device >= ndev) return fail(IDOCP_B200_INVALID_ARGUMENT, "invalid device index");
    CUDA_OK(cudaSetDevice(device));
    this->device = device;
    if (cudaStreamCreateWithFlags(&stream, cudaStreamNonBlocking) != cudaSuccess)
      return fail(IDOCP_B200_CUDA_ERROR, "cudaStreamCreate failed");
    return IDOCP_B200_OK;
  }
  // waits for the stream, then frees everything open() and the handle's calls created
  void release() {
    cudaSetDevice(device);
    if (stream) cudaStreamSynchronize(stream);
    resolve_profile();
    for (cudaEvent_t e : event_pool) cudaEventDestroy(e);
    if (copies_done) cudaEventDestroy(copies_done);
    for (void* p : allocs) cudaFree(p);
    if (stream) cudaStreamDestroy(stream);
  }

  int sync() {
    CUDA_OK(cudaSetDevice(device));
    CUDA_OK(cudaStreamSynchronize(stream));
    return IDOCP_B200_OK;
  }
  int launch_count(long long* out) const {
    *out = launches;
    return IDOCP_B200_OK;
  }
  int get_stream(void** out) const {
    *out = reinterpret_cast<void*>(stream);
    return IDOCP_B200_OK;
  }
  int set_profiling(int enabled) {
    resolve_profile();
    profiling = enabled != 0;
    for (int k = 0; k < KC_NUM; ++k) { prof_ms[k] = 0; prof_calls[k] = 0; }
    return IDOCP_B200_OK;
  }
  int get_profile(int cap, const char** names, double* ms, long long* calls) {
    resolve_profile();
    int n = 0;
    for (int k = 0; k < KC_NUM && n < cap; ++k) {
      if (prof_calls[k] == 0) continue;
      names[n] = kKernelClassNames[k];
      ms[n] = prof_ms[k];
      calls[n] = prof_calls[k];
      ++n;
    }
    return n;
  }
};

template <typename H>
static int destroy_handle(H* h) {
  if (h) {
    h->release();
    delete h;
  }
  return IDOCP_B200_OK;
}

struct idocp_b200_solver : DeviceHandle {
  idocp_b200_problem prob;
  int kind = 0;
  int B = 0, Bp = 0, N = 0;
  DevProblem* d_prob = nullptr;
  DevProblem h_prob;
  Layout L;
  double* d_q0 = nullptr;
  double* d_v0 = nullptr;
  double* d_stage = nullptr;   // staging buffer for getters / setters
  size_t stage_doubles = 0;
  // UnParNMPC extras
  ParNMPCLayout PL;
  // line search (allocated on first use)
  LineSearchLayout LS;
  bool ls_ready = false;
  // UnOCPSolver pipelining: updateSolution ends with k_linearize<.., FUSED> = update + linearisation of the NEW iterate,
  // which the next updateSolution re-uses as long as nothing changed the iterate or the cost reference in between
  bool pipelined = true;
  bool lin_valid = false;
  // KKT by-product of the fused update + linearisation (k_update_linearize<.., KKT>): switched on by the first computeKKTResidual
  // of a pipelined solver; kkt_valid = L.kkt_stage holds the stage sums of the current iterate
  bool kkt_tracking = false;
  bool kkt_valid = false;
  int sm_count = 1;            // persistent kernels launch one CTA pair per SM

  int stage_offset() const { return kind == IDOCP_B200_SOLVER_UNPARNMPC ? 1 : 0; }
};

extern "C" const char* idocp_b200_last_error(void) { return g_last_error.c_str(); }
extern "C" const char* idocp_b200_version(void) {
#ifdef IDOCP_B200_EMU
  return "idocp_b200 0.1 (SIMT emulator build -- tests only)";
#else
  return "idocp_b200 0.1 (sm_100a)";
#endif
}

extern "C" int idocp_b200_problem_default(int robot, idocp_b200_problem* p) {
  if (!p) return fail(IDOCP_B200_INVALID_ARGUMENT, "problem_default: null pointer");
  if (robot != IDOCP_B200_ROBOT_IIWA14) return fail(IDOCP_B200_UNSUPPORTED, "only the iiwa14 is supported");
  std::memset(p, 0, sizeof(*p));
  p->robot = robot;
  p->N = 20;
  p->T = 1.0;
  for (int i = 0; i < NV; ++i) {
    p->q_min[i] = IIWA14_Q_MIN[i];
    p->q_max[i] = IIWA14_Q_MAX[i];
    p->v_max[i] = IIWA14_V_MAX[i];
    p->u_max[i] = IIWA14_EFFORT_MAX[i];
  }
  p->barrier = 1.0e-04;
  p->fraction_rate = 0.995;
  return IDOCP_B200_OK;
}

static void fill_dev_problem(const idocp_b200_problem& p, DevProblem& d) {
  std::memset(&d, 0, sizeof(d));
  d.N = p.N;
  d.T = p.T;
  d.dt = p.T / p.N;
  for (int i = 0; i < NV; ++i) {
    d.q_ref[i] = p.q_ref[i]; d.v_ref[i] = p.v_ref[i]; d.u_ref[i] = p.u_ref[i];
    d.q_weight[i] = p.q_weight[i]; d.v_weight[i] = p.v_weight[i]; d.a_weight[i] = p.a_weight[i];
    d.u_weight[i] = p.u_weight[i]; d.qf_weight[i] = p.qf_weight[i]; d.vf_weight[i] = p.vf_weight[i];
    d.q_min[i] = p.q_min[i]; d.q_max[i] = p.q_max[i]; d.v_max[i] = p.v_max[i]; d.u_max[i] = p.u_max[i];
  }
  d.barrier = p.barrier;
  d.fraction_rate = p.fraction_rate;
  for (int k = 0; k < 2; ++k) d.acc_enable[k] = p.enable_acceleration_limit[k] ? 1 : 0;
  for (int i = 0; i < NV; ++i) { d.a_min[i] = p.a_min[i]; d.a_max[i] = p.a_max[i]; }
  d.gravity = IIWA14_GRAVITY;
  // TimeVaryingTaskSpace6DCost::set_q_6d_weight(position_weight, rotation_weight) stores head<3> = rotation,
  // tail<3> = position (time_varying_task_space_6d_cost.cpp:43-58) and applies them to diff_6d = [linear; angular]
  // task_enabled == 2: TaskSpace3DCost / TimeVaryingTaskSpace3DCost, the three weights apply to diff_3d as given
  d.task_enabled = p.task_enabled == 2 ? 2 : (p.task_enabled ? 1 : 0);
  for (int k = 0; k < 3; ++k) {
    if (d.task_enabled == 2) {
      d.task_w6[k] = p.task_q_weight[k];   d.task_w6[3 + k] = 0.0;
      d.task_wf6[k] = p.task_qf_weight[k]; d.task_wf6[3 + k] = 0.0;
    } else {
      d.task_w6[k] = p.task_q_weight[3 + k];  d.task_w6[3 + k] = p.task_q_weight[k];
      d.task_wf6[k] = p.task_qf_weight[3 + k]; d.task_wf6[3 + k] = p.task_qf_weight[k];
    }
  }
  for (int k = 0; k < 9; ++k) d.ee[k] = IIWA14_EE_PLACEMENT_R[k];
  for (int k = 0; k < 3; ++k) d.ee[9 + k] = IIWA14_EE_PLACEMENT_P[k];
  for (int j = 0; j < 8; ++j) {
    double* m = d.model + j * MODEL_STRIDE;
    if (j < NV) {
      for (int k = 0; k < 9; ++k) m[k] = IIWA14_PLACEMENT_R[j][k];
      for (int k = 0; k < 3; ++k) m[9 + k] = IIWA14_PLACEMENT_P[j][k];
      m[12] = IIWA14_MASS[j];
      for (int k = 0; k < 3; ++k) m[13 + k] = IIWA14_COM[j][k];
      for (int k = 0; k < 6; ++k) m[16 + k] = IIWA14_INERTIA[j][k];
    } else {
      m[0] = m[4] = m[8] = 1.0;  // padding joint: identity placement, zero mass
    }
  }
}

// grid of a per-stage kernel: one warp per (stage, group)
static int stage_grid(const idocp_b200_solver* h, int nstages) {
  const long tasks = static_cast<long>(nstages) * h->L.G;
  return static_cast<int>((tasks + WARPS_PER_CTA - 1) / WARPS_PER_CTA);
}
// grid of a per-instance kernel: one warp per group
static int group_grid(const idocp_b200_solver* h) { return (h->L.G + WARPS_PER_CTA - 1) / WARPS_PER_CTA; }
static int ric_grid(const idocp_b200_solver* h) { return (h->L.G + RIC_WARPS - 1) / RIC_WARPS; }
static const int kLinSmem = OCTETS_PER_CTA * OCT * PAIR_TILE * static_cast<int>(sizeof(double));
static const int kRicSmem = RIC_SMEM_DOUBLES * static_cast<int>(sizeof(double));
static const int kUlSmem = UL_SMEM_DOUBLES * static_cast<int>(sizeof(double));

static int do_init_constraints(idocp_b200_solver* h) {
  h->lin_valid = false; h->kkt_valid = false;   // slack / dual change: the kept linearisation is stale
  IDOCP_LAUNCH(h, KC_MISC, k_init_constraints, stage_grid(h, h->N), CTA_THREADS, 0, h->d_prob, h->L,
               h->stage_offset());
  CUDA_OK(cudaGetLastError());
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_create(const idocp_b200_problem* p, int solver_kind, int batch, int device,
                                 idocp_b200_solver** out) {
  if (!p || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "create: null pointer");
  *out = nullptr;
  if (p->robot != IDOCP_B200_ROBOT_IIWA14) return fail(IDOCP_B200_UNSUPPORTED, "only the iiwa14 is supported");
  if (!(p->T > 0)) return fail(IDOCP_B200_INVALID_ARGUMENT, "invalid value: T must be positive!");
  if (p->N <= 0) return fail(IDOCP_B200_INVALID_ARGUMENT, "invalid value: N must be positive!");
  if (batch <= 0) return fail(IDOCP_B200_INVALID_ARGUMENT, "invalid value: batch must be positive!");
  if (!(p->barrier > 0) || !(p->fraction_rate > 0) || p->fraction_rate > 1)
    return fail(IDOCP_B200_INVALID_ARGUMENT, "invalid value: barrier / fraction_rate");
  if (solver_kind != IDOCP_B200_SOLVER_UNOCP && solver_kind != IDOCP_B200_SOLVER_UNPARNMPC)
    return fail(IDOCP_B200_INVALID_ARGUMENT, "unknown solver kind");
  idocp_b200_solver* h = new idocp_b200_solver();
  const int orc = h->open(device);
  if (orc != IDOCP_B200_OK) {
    delete h;
    return orc;
  }
  h->prob = *p;
  h->kind = solver_kind;
  h->B = batch;
  h->Bp = (batch + 3) / 4 * 4;
  h->N = p->N;
  fill_dev_problem(*p, h->h_prob);
  const size_t N = h->N, Bp = h->Bp, G = Bp / 4;
  const bool par = solver_kind == IDOCP_B200_SOLVER_UNPARNMPC;
  Layout& L = h->L;
  std::memset(&L, 0, sizeof(L));
  L.B = h->B; L.Bp = h->Bp; L.G = static_cast<int>(G); L.N = h->N;
  int rc = 0;
  rc |= h->alloc(&h->d_prob, 1);
  rc |= h->alloc(&L.X, (N + 1) * G * X_NUM * SLOT);
  if (!par) rc |= h->alloc(&L.X2, (N + 1) * G * X_NUM * SLOT);
  rc |= h->alloc(&L.KQ, (N + 1) * G * KQ_NUM * SLOT);   // record N: dense terminal Hessian of the task-space cost
  rc |= h->alloc(&L.task_ref, (N + 1) * 12);
  if (p->enable_acceleration_limit[0] || p->enable_acceleration_limit[1]) {
    // JointAcceleration{Lower,Upper}Limit: their slack / dual rows live in their own array and run through the literal kernel
    // sequence with the ACC instantiations; the six-component kernels and the X record are untouched
    rc |= h->alloc(&L.XA, N * G * XA_NUM * SLOT);
    h->pipelined = false;
  }
  rc |= h->alloc(&L.W, N * G * W_NUM * SLOT);
  rc |= h->alloc(&L.D, (N + 1) * G * D_NUM * SLOT);
  rc |= h->alloc(&L.smin, 2 * N * Bp);
  rc |= h->alloc(&L.steps, 3 * Bp);
  rc |= h->alloc(&L.kkt_stage, (N + 1) * Bp);
  rc |= h->alloc(&L.kkt_err, Bp);
  rc |= h->alloc(&L.status, Bp);
  rc |= h->alloc(&h->d_q0, Bp * NV);
  rc |= h->alloc(&h->d_v0, Bp * NV);
  {
    const size_t Bz = static_cast<size_t>(h->B);
    size_t need = Bz * N * NC * NV;                              // get_constraint_data
    if (need < Bz * (N + 1) * NV) need = Bz * (N + 1) * NV;      // get_solution / get_direction / set_solution
    if (need < Bz * (441 + 35)) need = Bz * (441 + 35);          // get_unkkt
    h->stage_doubles = need;
  }
  rc |= h->alloc(&h->d_stage, h->stage_doubles);
  if (cudaFuncSetAttribute(k_riccati<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRicSmem) != cudaSuccess) rc |= -1;
  if (cudaFuncSetAttribute(k_riccati<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRicSmem) != cudaSuccess) rc |= -1;
  if (cudaFuncSetAttribute(k_update_linearize<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUlSmem) != cudaSuccess) rc |= -1;
  if (cudaFuncSetAttribute(k_update_linearize<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUlSmem) != cudaSuccess) rc |= -1;
  if (cudaFuncSetAttribute(k_update_linearize<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUlSmem) != cudaSuccess) rc |= -1;
  if (cudaFuncSetAttribute(k_update_linearize<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kUlSmem) != cudaSuccess) rc |= -1;
  {
    int dev = 0, sms = 0;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && sms > 0)
      h->sm_count = sms;
  }
  if (par) {
    rc |= parnmpc_alloc(h->PL, h->N, h->Bp, [&](double** pp, size_t n) { return h->alloc(pp, n); });
    if (cudaFuncSetAttribute(k_parnmpc_invert, cudaFuncAttributeMaxDynamicSharedMemorySize, INV_SMEM_BYTES) !=
        cudaSuccess)
      rc |= -1;
  }
  if (rc != 0) {
    idocp_b200_destroy(h);
    return fail(IDOCP_B200_CUDA_ERROR, "device memory allocation failed");
  }
  if (cudaMemcpyAsync(h->d_prob, &h->h_prob, sizeof(DevProblem), cudaMemcpyHostToDevice, h->stream) != cudaSuccess) {
    idocp_b200_destroy(h);
    return fail(IDOCP_B200_CUDA_ERROR, "problem upload failed");
  }
  {
    // until set_task_reference is called: identity placements (only read when the task-space cost is enabled)
    std::vector<double> ident((N + 1) * 12, 0.0);
    for (size_t i = 0; i <= N; ++i) ident[i * 12] = ident[i * 12 + 4] = ident[i * 12 + 8] = 1.0;
    if (cudaMemcpyAsync(L.task_ref, ident.data(), ident.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream) !=
            cudaSuccess ||
        cudaStreamSynchronize(h->stream) != cudaSuccess) {
      idocp_b200_destroy(h);
      return fail(IDOCP_B200_CUDA_ERROR, "task reference upload failed");
    }
  }
  const int irc = do_init_constraints(h);  // the reference ctor ends with initConstraints() (unocp_solver.cpp:48)
  if (irc != IDOCP_B200_OK) {
    idocp_b200_destroy(h);
    return irc;
  }
  CUDA_OK(cudaStreamSynchronize(h->stream));
  *out = h;
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_destroy(idocp_b200_solver* h) { return destroy_handle(h); }

static int field_index(const char* name) {
  if (!name) return -1;
  if (!std::strcmp(name, "lmd")) return X_LMD;
  if (!std::strcmp(name, "gmm")) return X_GMM;
  if (!std::strcmp(name, "q")) return X_Q;
  if (!std::strcmp(name, "v")) return X_V;
  if (!std::strcmp(name, "a")) return X_A;
  if (!std::strcmp(name, "u")) return X_U;
  if (!std::strcmp(name, "beta")) return X_BETA;
  return -1;
}
static int dir_index(const char* name) {
  if (!name) return -1;
  if (!std::strcmp(name, "dlmd")) return D_LMD;
  if (!std::strcmp(name, "dgmm")) return D_GMM;
  if (!std::strcmp(name, "dq")) return D_Q;
  if (!std::strcmp(name, "dv")) return D_V;
  if (!std::strcmp(name, "da")) return D_A;
  if (!std::strcmp(name, "du")) return D_U;
  if (!std::strcmp(name, "dbeta")) return D_BETA;
  return -1;
}

extern "C" int idocp_b200_set_solution(idocp_b200_solver* h, const char* name, const double* value, int broadcast) {
  if (!h || !value) return fail(IDOCP_B200_INVALID_ARGUMENT, "set_solution: null pointer");
  const int f = field_index(name);
  if (f != X_Q && f != X_V && f != X_A && f != X_U)
    return fail(IDOCP_B200_INVALID_ARGUMENT, "invalid arugment: name must be q, v, a, or u!");
  CUDA_OK(cudaSetDevice(h->device));
  const size_t n = broadcast ? NV : static_cast<size_t>(h->B) * NV;
  CUDA_OK(cudaMemcpyAsync(h->d_stage, value, n * sizeof(double), cudaMemcpyHostToDevice, h->stream));
  // UnOCPSolver: all N+1 stages (a, u: harmless on the terminal slot, never read);
  // UnParNMPCSolver stores stages 1..N at index 0..N-1
  const int nst = h->kind == IDOCP_B200_SOLVER_UNPARNMPC ? h->N : h->N + 1;
  const long total = static_cast<long>(nst) * h->Bp * OCT;
  IDOCP_LAUNCH(h, KC_MISC, k_set_solution, static_cast<int>((total + 255) / 256), 256, 0, h->L, f, h->d_stage,
               broadcast ? 1 : 0, nst);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaStreamSynchronize(h->stream));  // `value` may be pageable host memory reused by the caller
  return do_init_constraints(h);
}

extern "C" int idocp_b200_init_constraints(idocp_b200_solver* h) {
  if (!h) return fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
  CUDA_OK(cudaSetDevice(h->device));
  return do_init_constraints(h);
}

static int upload_x0(idocp_b200_solver* h, const double* q, const double* v) {
  if (!q || !v) return fail(IDOCP_B200_INVALID_ARGUMENT, "q / v: null pointer");
  const size_t n = static_cast<size_t>(h->B) * NV * sizeof(double);
  CUDA_OK(cudaMemcpyAsync(h->d_q0, q, n, cudaMemcpyHostToDevice, h->stream));
  CUDA_OK(cudaMemcpyAsync(h->d_v0, v, n, cudaMemcpyHostToDevice, h->stream));
  if (h->mark_uploads() != 0) return fail(IDOCP_B200_CUDA_ERROR, "upload of q / v failed");
  return IDOCP_B200_OK;
}

static int ensure_line_search(idocp_b200_solver* h) {
  if (h->ls_ready) return IDOCP_B200_OK;
  const size_t N = h->N, Bp = h->Bp;
  int rc = 0;
  rc |= h->alloc(&h->LS.cost, (N + 1) * Bp);
  rc |= h->alloc(&h->LS.viol, N * Bp);
  rc |= h->alloc(&h->LS.alpha, Bp);
  rc |= h->alloc(&h->LS.state, Bp);
  rc |= h->alloc(&h->LS.flt_n, Bp);
  rc |= h->alloc(&h->LS.flt_cost, Bp * LS_FILTER_CAP);
  rc |= h->alloc(&h->LS.flt_viol, Bp * LS_FILTER_CAP);
  if (rc != 0) return fail(IDOCP_B200_CUDA_ERROR, "line-search buffers: device memory allocation failed");
  h->ls_ready = true;
  return IDOCP_B200_OK;
}

// UnLineSearch::computeStepSize for the whole batch: lock-step rounds, no host synchronisation
static int run_line_search(idocp_b200_solver* h, const double* d_q, const double* d_v) {
  const int rc = ensure_line_search(h);
  if (rc != IDOCP_B200_OK) return rc;
  const int off = h->stage_offset();
  const bool par = h->kind == IDOCP_B200_SOLVER_UNPARNMPC;
  const int ncost = par ? h->N : h->N + 1;
  const int fgrid = (h->B + 127) / 128;
  const bool task = h->prob.task_enabled != 0;
  IDOCP_LAUNCH(h, KC_LINESEARCH, k_ls_begin, group_grid(h), CTA_THREADS, 0, h->L);
  auto eval = [&](int mode) {
    const int grid = stage_grid(h, ncost);
    if (par) {
      if (task)
        IDOCP_LAUNCH(h, KC_LINESEARCH, (k_ls_eval<true, true>), grid, CTA_THREADS, 0, h->d_prob, h->L, h->LS, mode, off, d_q, d_v);
      else
        IDOCP_LAUNCH(h, KC_LINESEARCH, (k_ls_eval<false, true>), grid, CTA_THREADS, 0, h->d_prob, h->L, h->LS, mode, off, d_q, d_v);
    } else {
      if (task)
        IDOCP_LAUNCH(h, KC_LINESEARCH, (k_ls_eval<true, false>), grid, CTA_THREADS, 0, h->d_prob, h->L, h->LS, mode, off, d_q, d_v);
      else
        IDOCP_LAUNCH(h, KC_LINESEARCH, (k_ls_eval<false, false>), grid, CTA_THREADS, 0, h->d_prob, h->L, h->LS, mode, off, d_q, d_v);
    }
  };
  eval(0);
  IDOCP_LAUNCH(h, KC_LINESEARCH, k_ls_filter, fgrid, 128, 0, h->L, h->LS, 0, ncost);
  for (int trial = 0; trial < LS_MAX_TRIALS; ++trial) {
    eval(1);
    IDOCP_LAUNCH(h, KC_LINESEARCH, k_ls_filter, fgrid, 128, 0, h->L, h->LS, 1, ncost);
  }
  CUDA_OK(cudaGetLastError());
  return IDOCP_B200_OK;
}

// k_linearize / k_expand instantiation by the run-time problem flags (task-space cost, acceleration limits)
template <bool RES, bool BE>
static void launch_linearize(idocp_b200_solver* h, int cls, int nstages, const double* d_q, const double* d_v) {
  const bool task = h->prob.task_enabled != 0, acc = h->L.XA != nullptr;
  const int grid = stage_grid(h, nstages);
  if (task && acc) IDOCP_LAUNCH(h, cls, (k_linearize<RES, BE, true, true>), grid, CTA_THREADS, kLinSmem, h->d_prob, h->L, d_q, d_v);
  else if (task) IDOCP_LAUNCH(h, cls, (k_linearize<RES, BE, true, false>), grid, CTA_THREADS, kLinSmem, h->d_prob, h->L, d_q, d_v);
  else if (acc) IDOCP_LAUNCH(h, cls, (k_linearize<RES, BE, false, true>), grid, CTA_THREADS, kLinSmem, h->d_prob, h->L, d_q, d_v);
  else IDOCP_LAUNCH(h, cls, (k_linearize<RES, BE, false, false>), grid, CTA_THREADS, kLinSmem, h->d_prob, h->L, d_q, d_v);
}
template <bool PARNMPC>
static void launch_expand(idocp_b200_solver* h, int nstages, int stage_offset) {
  const bool task = !PARNMPC && h->prob.task_enabled != 0, acc = h->L.XA != nullptr;
  const int grid = stage_grid(h, nstages);
  if (task && acc) IDOCP_LAUNCH(h, KC_EXPAND, (k_expand<PARNMPC, !PARNMPC, true>), grid, CTA_THREADS, 0, h->d_prob, h->L, stage_offset);
  else if (task) IDOCP_LAUNCH(h, KC_EXPAND, (k_expand<PARNMPC, !PARNMPC, false>), grid, CTA_THREADS, 0, h->d_prob, h->L, stage_offset);
  else if (acc) IDOCP_LAUNCH(h, KC_EXPAND, (k_expand<PARNMPC, false, true>), grid, CTA_THREADS, 0, h->d_prob, h->L, stage_offset);
  else IDOCP_LAUNCH(h, KC_EXPAND, (k_expand<PARNMPC, false, false>), grid, CTA_THREADS, 0, h->d_prob, h->L, stage_offset);
}

static int unocp_update(idocp_b200_solver* h, const double* d_q, const double* d_v, int line_search) {
  const bool task = h->prob.task_enabled != 0;
  if (!(h->pipelined && h->lin_valid)) {
    launch_linearize<false, false>(h, KC_LINEARIZE, task ? h->N + 1 : h->N, d_q, d_v);
  }
  if (task) {
    IDOCP_LAUNCH(h, KC_RICCATI, k_riccati<true>, ric_grid(h), RIC_THREADS, kRicSmem, h->d_prob, h->L, d_q, d_v);
    launch_expand<false>(h, h->N + 1, 0);
  } else {
    IDOCP_LAUNCH(h, KC_RICCATI, k_riccati<false>, ric_grid(h), RIC_THREADS, kRicSmem, h->d_prob, h->L, d_q, d_v);
    launch_expand<false>(h, h->N + 1, 0);
  }
  const double* override_alpha = nullptr;
  if (line_search) {
    const int rc = run_line_search(h, d_q, d_v);
    if (rc != IDOCP_B200_OK) return rc;
    override_alpha = h->LS.alpha;
  }
  if (h->pipelined) {
    // step sizes, then update + linearisation of the new iterate in one persistent launch; X (old) -> X2 (new), then the
    // two swap roles
    IDOCP_LAUNCH(h, KC_STEP_MIN, k_step_min, (h->Bp + 127) / 128, 128, 0, h->L, override_alpha);
    const long ul_tasks = static_cast<long>(h->N + 1) * h->L.G;
    const int ul_grid = static_cast<int>(std::min<long>((ul_tasks + UL_WARPS - 1) / UL_WARPS, static_cast<long>(IDOCP_UL_CTAS_PER_SM) * h->sm_count));
    if (task && h->kkt_tracking)
      IDOCP_LAUNCH(h, KC_UPDATE_LINEARIZE, (k_update_linearize<true, true>), ul_grid, UL_THREADS, kUlSmem, h->d_prob, h->L);
    else if (task)
      IDOCP_LAUNCH(h, KC_UPDATE_LINEARIZE, (k_update_linearize<true, false>), ul_grid, UL_THREADS, kUlSmem, h->d_prob, h->L);
    else if (h->kkt_tracking)
      IDOCP_LAUNCH(h, KC_UPDATE_LINEARIZE, (k_update_linearize<false, true>), ul_grid, UL_THREADS, kUlSmem, h->d_prob, h->L);
    else
      IDOCP_LAUNCH(h, KC_UPDATE_LINEARIZE, (k_update_linearize<false, false>), ul_grid, UL_THREADS, kUlSmem, h->d_prob, h->L);
    std::swap(h->L.X, h->L.X2);
    h->lin_valid = true;
    h->kkt_valid = h->kkt_tracking;
  } else {
    IDOCP_LAUNCH(h, KC_UPDATE, k_update, stage_grid(h, h->N + 1), CTA_THREADS, 0, h->d_prob, h->L, 0, override_alpha,
                 h->N + 1);
  }
  CUDA_OK(cudaGetLastError());
  return IDOCP_B200_OK;
}

// UnParNMPCSolver::updateSolution (src/unocp/unparnmpc_solver.cpp:74-102)
static int parnmpc_update(idocp_b200_solver* h, double, const double* d_q, const double* d_v, int line_search) {
  const int N = h->N;
  // UnBackwardCorrection::coarseUpdate (src/unocp/unbackward_correction.cpp:67-97)
  launch_linearize<false, true>(h, KC_LINEARIZE, N, d_q, d_v);
  IDOCP_LAUNCH(h, KC_PARNMPC_COARSE, k_parnmpc_invert, N * h->L.G, CTA_THREADS, INV_SMEM_BYTES, h->d_prob, h->L, h->PL);
  // UnBackwardCorrection::backwardCorrection (:100-134)
  if (N > 1) {
    IDOCP_LAUNCH(h, KC_PARNMPC_CORR, k_parnmpc_backward_serial, group_grid(h), CTA_THREADS, 0, h->L, h->PL);
    IDOCP_LAUNCH(h, KC_PARNMPC_CORR, k_parnmpc_backward_parallel, stage_grid(h, N - 1), CTA_THREADS, 0, h->L, h->PL);
    IDOCP_LAUNCH(h, KC_PARNMPC_CORR, k_parnmpc_forward_serial, group_grid(h), CTA_THREADS, 0, h->L, h->PL);
  }
  IDOCP_LAUNCH(h, KC_PARNMPC_CORR, k_parnmpc_forward_parallel, stage_grid(h, N), CTA_THREADS, 0, h->L, h->PL);
  launch_expand<true>(h, N, 1);
  const double* override_alpha = nullptr;
  if (line_search) {
    const int rc = run_line_search(h, d_q, d_v);
    if (rc != IDOCP_B200_OK) return rc;
    override_alpha = h->LS.alpha;
  }
  IDOCP_LAUNCH(h, KC_UPDATE, k_update, stage_grid(h, N), CTA_THREADS, 0, h->d_prob, h->L, 1, override_alpha, N);
  CUDA_OK(cudaGetLastError());
  return IDOCP_B200_OK;
}

// UnParNMPCSolver::computeKKTResidual (src/unocp/unparnmpc_solver.cpp:171-192)
static int parnmpc_kkt_residual(idocp_b200_solver* h, double, const double* d_q, const double* d_v) {
  launch_linearize<true, true>(h, KC_KKT, h->N, d_q, d_v);
  IDOCP_LAUNCH(h, KC_KKT, k_kkt_sum, (h->Bp + 127) / 128, 128, 0, h->L, h->N);
  CUDA_OK(cudaGetLastError());
  return IDOCP_B200_OK;
}

// UnParNMPCSolver::initBackwardCorrection (src/unocp/unparnmpc_solver.cpp:69-71)
static int parnmpc_init_backward_correction(idocp_b200_solver* h, double) {
  if (h->prob.task_enabled)
    IDOCP_LAUNCH(h, KC_MISC, k_parnmpc_init_aux<true>, stage_grid(h, h->N), CTA_THREADS, kLinSmem, h->d_prob, h->L, h->PL);
  else
    IDOCP_LAUNCH(h, KC_MISC, k_parnmpc_init_aux<false>, stage_grid(h, h->N), CTA_THREADS, kLinSmem, h->d_prob, h->L,
                 h->PL);
  CUDA_OK(cudaGetLastError());
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_update_solution_device(idocp_b200_solver* h, double t, const double* d_q, const double* d_v,
                                                 int line_search) {
  if (!h || !d_q || !d_v) return fail(IDOCP_B200_INVALID_ARGUMENT, "update_solution: null pointer");
  (void)t;  // ConfigurationSpaceCost is time invariant
  CUDA_OK(cudaSetDevice(h->device));
  if (h->kind == IDOCP_B200_SOLVER_UNOCP) return unocp_update(h, d_q, d_v, line_search);
  return parnmpc_update(h, t, d_q, d_v, line_search);
}

extern "C" int idocp_b200_update_solution(idocp_b200_solver* h, double t, const double* q, const double* v,
                                          int line_search) {
  if (!h) return fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
  CUDA_OK(cudaSetDevice(h->device));
  int rc = upload_x0(h, q, v);
  if (rc != IDOCP_B200_OK) return rc;
  rc = idocp_b200_update_solution_device(h, t, h->d_q0, h->d_v0, line_search);
  if (h->wait_for_uploads() != 0) return fail(IDOCP_B200_CUDA_ERROR, "upload of q / v failed");
  return rc;
}

extern "C" int idocp_b200_compute_kkt_residual_device(idocp_b200_solver* h, double t, const double* d_q,
                                                      const double* d_v) {
  if (!h || !d_q || !d_v) return fail(IDOCP_B200_INVALID_ARGUMENT, "compute_kkt_residual: null pointer");
  (void)t;
  CUDA_OK(cudaSetDevice(h->device));
  if (h->kind == IDOCP_B200_SOLVER_UNPARNMPC) return parnmpc_kkt_residual(h, t, d_q, d_v);
  if (h->pipelined && h->lin_valid && h->kkt_valid) {
    // the fused update + linearisation of the last updateSolution left the stage sums of this very iterate behind
    IDOCP_LAUNCH(h, KC_KKT, k_kkt_sum, (h->Bp + 127) / 128, 128, 0, h->L, h->N + 1);
    CUDA_OK(cudaGetLastError());
    return IDOCP_B200_OK;
  }
  if (h->pipelined) h->kkt_tracking = true;   // the caller watches the KKT error: from the next updateSolution on it comes for free
  launch_linearize<true, false>(h, KC_KKT, h->N + 1, d_q, d_v);
  IDOCP_LAUNCH(h, KC_KKT, k_kkt_sum, (h->Bp + 127) / 128, 128, 0, h->L, h->N + 1);
  CUDA_OK(cudaGetLastError());
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_compute_kkt_residual(idocp_b200_solver* h, double t, const double* q, const double* v) {
  if (!h) return fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
  CUDA_OK(cudaSetDevice(h->device));
  int rc = upload_x0(h, q, v);
  if (rc != IDOCP_B200_OK) return rc;
  rc = idocp_b200_compute_kkt_residual_device(h, t, h->d_q0, h->d_v0);
  if (h->wait_for_uploads() != 0) return fail(IDOCP_B200_CUDA_ERROR, "upload of q / v failed");
  return rc;
}

extern "C" int idocp_b200_kkt_error(idocp_b200_solver* h, double* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "kkt_error: null pointer");
  CUDA_OK(cudaSetDevice(h->device));
  CUDA_OK(cudaMemcpyAsync(out, h->L.kkt_err, static_cast<size_t>(h->B) * sizeof(double), cudaMemcpyDeviceToHost,
                          h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return IDOCP_B200_OK;
}

// gather one slot of `nstage` stages: out[b][stage][7]
__global__ void k_gather(const double* __restrict__ src, int ns, int slot, int nstage, int B, int G,
                         double* __restrict__ out) {
  const long idx = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long total = static_cast<long>(B) * nstage * NV;
  if (idx >= total) return;
  const int j = static_cast<int>(idx % NV);
  const long t = idx / NV;
  const int i = static_cast<int>(t % nstage);
  const int b = static_cast<int>(t / nstage);
  out[idx] = src[elem_index(ns, G, i, b, slot, j)];
}

static int gather_to_host(idocp_b200_solver* h, const double* src, int ns, int slot, int nstage, double* out) {
  const long total = static_cast<long>(h->B) * nstage * NV;
  if (static_cast<size_t>(total) > h->stage_doubles) return fail(IDOCP_B200_INVALID_ARGUMENT, "staging buffer too small");
  IDOCP_LAUNCH(h, KC_MISC, k_gather, static_cast<int>((total + 255) / 256), 256, 0, src, ns, slot, nstage, h->B,
               h->L.G, h->d_stage);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaMemcpyAsync(out, h->d_stage, total * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return IDOCP_B200_OK;
}

static bool full_horizon(const idocp_b200_solver* h, int f) {
  return (f == X_LMD || f == X_GMM || f == X_Q || f == X_V) && h->kind == IDOCP_B200_SOLVER_UNOCP;
}

extern "C" int idocp_b200_get_solution(idocp_b200_solver* h, const char* name, double* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_solution: null pointer");
  const int f = field_index(name);
  if (f < 0) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_solution: unknown field");
  CUDA_OK(cudaSetDevice(h->device));
  return gather_to_host(h, h->L.X, X_NUM, f, full_horizon(h, f) ? h->N + 1 : h->N, out);
}

// one stage of one field: out[b][7]
__global__ void k_gather_stage(const double* __restrict__ src, int ns, int slot, int stage, int B, int G,
                               double* __restrict__ out) {
  const long idx = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  if (idx >= static_cast<long>(B) * OCT) return;
  const int j = static_cast<int>(idx & 7);
  const int b = static_cast<int>(idx >> 3);
  if (j < NV) out[static_cast<size_t>(b) * NV + j] = src[elem_index(ns, G, stage, b, slot, j)];
}

extern "C" int idocp_b200_get_stage_solution(idocp_b200_solver* h, const char* name, int stage, double* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_stage_solution: null pointer");
  const int f = field_index(name);
  if (f < 0) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_stage_solution: unknown field");
  if (stage < 0 || stage >= (full_horizon(h, f) ? h->N + 1 : h->N))
    return fail(IDOCP_B200_INVALID_ARGUMENT, "get_stage_solution: stage out of range");
  CUDA_OK(cudaSetDevice(h->device));
  const long total = static_cast<long>(h->B) * OCT;
  IDOCP_LAUNCH(h, KC_MISC, k_gather_stage, static_cast<int>((total + 255) / 256), 256, 0, h->L.X, X_NUM, f, stage,
               h->B, h->L.G, h->d_stage);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaMemcpyAsync(out, h->d_stage, static_cast<size_t>(h->B) * NV * sizeof(double), cudaMemcpyDeviceToHost,
                          h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_get_direction(idocp_b200_solver* h, const char* name, double* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_direction: null pointer");
  const int f = dir_index(name);
  if (f < 0) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_direction: unknown field");
  CUDA_OK(cudaSetDevice(h->device));
  const bool full = (f == D_LMD || f == D_GMM || f == D_Q || f == D_V) && h->kind == IDOCP_B200_SOLVER_UNOCP;
  return gather_to_host(h, h->L.D, D_NUM, f, full ? h->N + 1 : h->N, out);
}

// out[b][N][6][7]
__global__ void k_gather_constraints(const double* __restrict__ X, int first_slot, int N, int B, int G,
                                     double* __restrict__ out) {
  const long idx = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long total = static_cast<long>(B) * N * NC * NV;
  if (idx >= total) return;
  const int j = static_cast<int>(idx % NV);
  long t = idx / NV;
  const int c = static_cast<int>(t % NC);
  t /= NC;
  const int i = static_cast<int>(t % N);
  const int b = static_cast<int>(t / N);
  out[idx] = X[elem_index(X_NUM, G, i, b, first_slot + c, j)];
}

// out[b][N][2][7]: slots first_slot, first_slot + 1 of the acceleration-limit record
__global__ void k_gather_acc_rows(const double* __restrict__ XA, int first_slot, int N, int B, int G, double* __restrict__ out) {
  const long idx = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long total = static_cast<long>(B) * N * 2 * NV;
  if (idx >= total) return;
  const int j = static_cast<int>(idx % NV);
  long t = idx / NV;
  const int c = static_cast<int>(t % 2);
  t /= 2;
  const int i = static_cast<int>(t % N);
  const int b = static_cast<int>(t / N);
  out[idx] = XA[elem_index(XA_NUM, G, i, b, first_slot + c, j)];
}

extern "C" int idocp_b200_get_constraint_data(idocp_b200_solver* h, const char* name, double* out) {
  if (!h || !out || !name) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_constraint_data: null pointer");
  int first = -1;
  if (!std::strcmp(name, "slack")) first = X_SLACK;
  else if (!std::strcmp(name, "dual")) first = X_DUAL;
  else if (!std::strcmp(name, "acc_slack") || !std::strcmp(name, "acc_dual")) {
    // the two acceleration-limit components: out[batch][N][2][dimv]
    if (!h->L.XA) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_constraint_data: the acceleration limits are not enabled");
    CUDA_OK(cudaSetDevice(h->device));
    const long tot = static_cast<long>(h->B) * h->N * 2 * NV;
    IDOCP_LAUNCH(h, KC_MISC, k_gather_acc_rows, static_cast<int>((tot + 255) / 256), 256, 0, h->L.XA, name[4] == 's' ? 0 : 2, h->N,
                 h->B, h->L.G, h->d_stage);
    CUDA_OK(cudaGetLastError());
    CUDA_OK(cudaMemcpyAsync(out, h->d_stage, tot * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CUDA_OK(cudaStreamSynchronize(h->stream));
    return IDOCP_B200_OK;
  }
  else return fail(IDOCP_B200_INVALID_ARGUMENT, "get_constraint_data: name must be slack, dual, acc_slack or acc_dual");
  CUDA_OK(cudaSetDevice(h->device));
  const long total = static_cast<long>(h->B) * h->N * NC * NV;
  IDOCP_LAUNCH(h, KC_MISC, k_gather_constraints, static_cast<int>((total + 255) / 256), 256, 0, h->L.X, first, h->N,
               h->B, h->L.G, h->d_stage);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaMemcpyAsync(out, h->d_stage, total * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_get_step_sizes(idocp_b200_solver* h, double* primal, double* dual) {
  if (!h) return fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
  CUDA_OK(cudaSetDevice(h->device));
  const size_t n = static_cast<size_t>(h->B) * sizeof(double);
  if (primal) CUDA_OK(cudaMemcpyAsync(primal, h->L.steps, n, cudaMemcpyDeviceToHost, h->stream));
  if (dual) CUDA_OK(cudaMemcpyAsync(dual, h->L.steps + h->Bp, n, cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return IDOCP_B200_OK;
}

// Q[b][21*21] column-major (block order a,q,v), res[b][35]
__global__ void k_gather_unkkt(Layout L, int stage, double* __restrict__ Q, double* __restrict__ res) {
  const int b = blockIdx.x;
  if (b >= L.B) return;
  const int D = 3 * NV;
  for (int e = threadIdx.x; e < D * D; e += blockDim.x) Q[static_cast<size_t>(b) * D * D + e] = 0.0;
  __syncthreads();
  // (row-block, col-block) of the [a,q,v] ordering for the blocks AA, AQ, AV, QQ, QV, VV
  const int blk[6][2] = {{0, 0}, {0, 1}, {0, 2}, {1, 1}, {1, 2}, {2, 2}};
  for (int e = threadIdx.x; e < 6 * NV * NV; e += blockDim.x) {
    const int k = e / (NV * NV);
    const int r = (e / NV) % NV;
    const int c = e % NV;
    const double val = L.KQ[elem_index(KQ_NUM, L.G, stage, b, k * NV + r, c)];
    Q[static_cast<size_t>(b) * D * D + static_cast<size_t>(blk[k][1] * NV + c) * D + blk[k][0] * NV + r] = val;
  }
  for (int e = threadIdx.x; e < 5 * NV; e += blockDim.x)
    res[static_cast<size_t>(b) * 5 * NV + e] = L.KQ[elem_index(KQ_NUM, L.G, stage, b, KQ_FQ + e / NV, e % NV)];
}

extern "C" int idocp_b200_get_unkkt(idocp_b200_solver* h, int stage, double* Q, double* res) {
  if (!h || !Q || !res) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_unkkt: null pointer");
  if (stage < 0 || stage >= h->N) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_unkkt: stage out of range");
  CUDA_OK(cudaSetDevice(h->device));
  double* dQ = h->d_stage;
  double* dres = h->d_stage + static_cast<size_t>(h->B) * 441;
  IDOCP_LAUNCH(h, KC_MISC, k_gather_unkkt, h->B, 128, 0, h->L, stage, dQ, dres);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaMemcpyAsync(Q, dQ, static_cast<size_t>(h->B) * 441 * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(cudaMemcpyAsync(res, dres, static_cast<size_t>(h->B) * 35 * sizeof(double), cudaMemcpyDeviceToHost,
                          h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_get_status(idocp_b200_solver* h, int* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_status: null pointer");
  CUDA_OK(cudaSetDevice(h->device));
  CUDA_OK(cudaMemcpyAsync(out, h->L.status, static_cast<size_t>(h->B) * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return IDOCP_B200_OK;
}

__global__ void k_is_feasible(const DevProblem* __restrict__ Pp, Layout L, int stage_offset, int* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= L.B) return;
  const DevProblem& P = *Pp;
  int ok = 1;
  for (int i = 0; i < L.N; ++i)
    for (int j = 0; j < NV; ++j) {
      const LaneLimits lim = load_limits(P, j);
      const double q = L.X[elem_index(X_NUM, L.G, i, b, X_Q, j)];
      const double v = L.X[elem_index(X_NUM, L.G, i, b, X_V, j)];
      const double u = L.X[elem_index(X_NUM, L.G, i, b, X_U, j)];
      for (int c = 0; c < NC; ++c)
        if (comp_active(c, i + stage_offset) && con_margin(c, lim, q, v, u) < 0) ok = 0;
      if (L.XA) {   // JointAccelerationLowerLimit / UpperLimit::isFeasible (joint_acceleration_lower_limit.cpp:29-38)
        const double a = L.X[elem_index(X_NUM, L.G, i, b, X_A, j)];
        if (P.acc_enable[0] && a < P.a_min[j]) ok = 0;
        if (P.acc_enable[1] && a > P.a_max[j]) ok = 0;
      }
    }
  out[b] = ok;
}

extern "C" int idocp_b200_is_feasible(idocp_b200_solver* h, int* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "is_feasible: null pointer");
  CUDA_OK(cudaSetDevice(h->device));
  int* d = reinterpret_cast<int*>(h->d_stage);
  IDOCP_LAUNCH(h, KC_MISC, k_is_feasible, (h->B + 127) / 128, 128, 0, h->d_prob, h->L, h->stage_offset(), d);
  CUDA_OK(cudaGetLastError());
  CUDA_OK(cudaMemcpyAsync(out, d, static_cast<size_t>(h->B) * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_clear_line_search_filter(idocp_b200_solver* h) {
  if (!h) return fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
  if (!h->ls_ready) return IDOCP_B200_OK;  // never used: already empty
  CUDA_OK(cudaSetDevice(h->device));
  IDOCP_LAUNCH(h, KC_LINESEARCH, k_ls_clear, (h->B + 127) / 128, 128, 0, h->LS, h->B);
  CUDA_OK(cudaGetLastError());
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_init_backward_correction(idocp_b200_solver* h, double t) {
  if (!h) return fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
  if (h->kind != IDOCP_B200_SOLVER_UNPARNMPC)
    return fail(IDOCP_B200_INVALID_ARGUMENT, "init_backward_correction: not an UnParNMPC solver");
  CUDA_OK(cudaSetDevice(h->device));
  return parnmpc_init_backward_correction(h, t);
}

extern "C" int idocp_b200_set_task_reference(idocp_b200_solver* h, const double* table) {
  if (!h || !table) return fail(IDOCP_B200_INVALID_ARGUMENT, "set_task_reference: null pointer");
  CUDA_OK(cudaSetDevice(h->device));
  CUDA_OK(cudaMemcpyAsync(h->L.task_ref, table, static_cast<size_t>(h->N + 1) * 12 * sizeof(double),
                          cudaMemcpyHostToDevice, h->stream));
  CUDA_OK(cudaStreamSynchronize(h->stream));  // `table` may be pageable host memory reused by the caller
  h->lin_valid = false; h->kkt_valid = false;                       // the kept linearisation used the old reference
  return IDOCP_B200_OK;
}

// UnOCPSolver pipelining (default on): see k_linearize<.., FUSED>.  Off: linearise, solve, expand, update as four launches;
// get_unkkt then shows the linearisation the last direction was computed from instead of the one kept for the next call.
extern "C" int idocp_b200_set_pipelining(idocp_b200_solver* h, int enabled) {
  if (!h) return fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
  h->pipelined = enabled != 0 && h->L.XA == nullptr;   // the acceleration limits run through the literal sequence only
  h->lin_valid = false; h->kkt_valid = false;
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_sync(idocp_b200_solver* h) {
  return h ? h->sync() : fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
}
extern "C" int idocp_b200_launch_count(idocp_b200_solver* h, long long* out) {
  return h && out ? h->launch_count(out) : fail(IDOCP_B200_INVALID_ARGUMENT, "launch_count: null pointer");
}
extern "C" int idocp_b200_stream(idocp_b200_solver* h, void** out) {
  return h && out ? h->get_stream(out) : fail(IDOCP_B200_INVALID_ARGUMENT, "stream: null pointer");
}
extern "C" int idocp_b200_set_profiling(idocp_b200_solver* h, int enabled) {
  return h ? h->set_profiling(enabled) : fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
}
extern "C" int idocp_b200_get_profile(idocp_b200_solver* h, int cap, const char** names, double* ms, long long* calls) {
  return h && names && ms && calls ? h->get_profile(cap, names, ms, calls)
                                   : fail(IDOCP_B200_INVALID_ARGUMENT, "get_profile: null pointer");
}

#include "derivative_checker.inc"
#include "hybrid_capi.inc"
#include "fb_capi.inc"
#include "sharded_capi.inc"
