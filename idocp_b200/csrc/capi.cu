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
#include <type_traits>
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

// f(std::true_type) if `flag` else f(std::false_type): turns a run-time problem flag into a kernel template argument
template <typename F>
static void with_flag(bool flag, F f) {
  if (flag) f(std::true_type());
  else f(std::false_type());
}

enum KernelClass { KC_LINEARIZE = 0, KC_RICCATI, KC_EXPAND, KC_UPDATE, KC_KKT, KC_MISC, KC_PARNMPC_COARSE,
                   KC_PARNMPC_CORR, KC_LINESEARCH, KC_FB_LINEARIZE, KC_FB_CONDENSE, KC_FB_RICCATI, KC_FB_FORWARD, KC_FB_EXPAND, KC_FB_UPDATE,
                   KC_FB_KKT, KC_UPDATE_LINEARIZE, KC_STEP_MIN, KC_NUM };
static const char* kKernelClassNames[KC_NUM] = {"linearize", "riccati", "expand", "update", "kkt", "misc",
                                                "parnmpc_coarse", "parnmpc_correction", "line_search", "fb_robot", "fb_condense",
                                                "fb_riccati_backward", "fb_riccati_forward", "fb_expand", "fb_update", "fb_kkt",
                                                "update_linearize", "step_min"};

// What every solver handle of both families owns: its device and stream, the device allocations, the CUDA events, the
// launch counter, the per-kernel-class event timing, the staging buffer, the initial state and the copies between the
// caller's host arrays and the device.  open() / release() are the one lifecycle of a handle; the *_sync /
// *_launch_count / *_stream / *_set_profiling / *_get_profile entry points of both families forward here.
struct DeviceHandle {
  int device = 0;
  cudaStream_t stream = nullptr;
  long long launches = 0;
  double* d_stage = nullptr;   // staging buffer of the getters / setters; each family sizes it at create time
  size_t stage_doubles = 0;
  double* d_q0 = nullptr;      // initial state of the batch (upload_state)
  double* d_v0 = nullptr;
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
  // copies whichever of q and v is non-null to d_q0 / d_v0 and records copies_done right behind the copies
  int upload_state(const double* q, size_t q_doubles, const double* v, size_t v_doubles) {
    if (q) CUDA_OK(cudaMemcpyAsync(d_q0, q, q_doubles * sizeof(double), cudaMemcpyHostToDevice, stream));
    if (v) CUDA_OK(cudaMemcpyAsync(d_v0, v, v_doubles * sizeof(double), cudaMemcpyHostToDevice, stream));
    if (!q && !v) return IDOCP_B200_OK;
    if ((!copies_done && cudaEventCreate(&copies_done) != cudaSuccess) || cudaEventRecord(copies_done, stream) != cudaSuccess)
      return fail(IDOCP_B200_CUDA_ERROR, "upload of q / v failed");
    return IDOCP_B200_OK;
  }
  int wait_for_uploads() {        // after the call's kernels have been enqueued: the wait overlaps their execution
    return (copies_done && cudaEventSynchronize(copies_done) != cudaSuccess) ? -1 : 0;
  }
  // Blocking copies: `src` of upload may be pageable host memory that the caller reuses as soon as the call returns, and
  // download returns once `dst` holds the device's data (both wait for everything enqueued on the stream before them).
  int upload(void* dst, const void* src, size_t bytes) {
    CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, stream));
    CUDA_OK(cudaStreamSynchronize(stream));
    return IDOCP_B200_OK;
  }
  int download(void* dst, const void* src, size_t bytes) {
    CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, stream));
    CUDA_OK(cudaStreamSynchronize(stream));
    return IDOCP_B200_OK;
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
  // the line-search filter of n instances (line_search_filter.cuh)
  int alloc_filter(LsFilter* F, size_t n) {
    int rc = 0;
    rc |= alloc(&F->alpha, n);
    rc |= alloc(&F->state, n);
    rc |= alloc(&F->n, n);
    rc |= alloc(&F->cost, n * LS_FILTER_CAP);
    rc |= alloc(&F->viol, n * LS_FILTER_CAP);
    return rc;
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
  // per-instance cost references (idocp_b200_set_instance_reference / _task_reference): L.iref / L.itask point at these
  // allocations while the mode is on (nullptr in shared mode); the allocations outlive a clear for the next set
  double* d_iref = nullptr;
  double* d_itask = nullptr;
  std::vector<double> iref_host;   // [B][IREF_NUM][7]: the configuration references of every instance in the caller's layout

  int stage_offset() const { return kind == IDOCP_B200_SOLVER_UNPARNMPC ? 1 : 0; }
  bool iref() const { return L.iref || L.itask; }   // kernels: the IREF instantiations
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
  for (int task = 0; task < 2; ++task)
    for (int kkt = 0; kkt < 2; ++kkt)
      for (int iref = 0; iref < 2; ++iref)
        with_flag(task, [&](auto T) { with_flag(kkt, [&](auto K) { with_flag(iref, [&](auto IR) {
          if (cudaFuncSetAttribute(k_update_linearize<decltype(T)::value, decltype(K)::value, decltype(IR)::value>,
                                   cudaFuncAttributeMaxDynamicSharedMemorySize, kUlSmem) != cudaSuccess)
            rc |= -1;
        }); }); });
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
  if (h->upload(h->d_prob, &h->h_prob, sizeof(DevProblem)) != IDOCP_B200_OK) {
    idocp_b200_destroy(h);
    return fail(IDOCP_B200_CUDA_ERROR, "problem upload failed");
  }
  {
    // until set_task_reference is called: identity placements (only read when the task-space cost is enabled)
    std::vector<double> ident((N + 1) * 12, 0.0);
    for (size_t i = 0; i <= N; ++i) ident[i * 12] = ident[i * 12 + 4] = ident[i * 12 + 8] = 1.0;
    if (h->upload(L.task_ref, ident.data(), ident.size() * sizeof(double)) != IDOCP_B200_OK) {
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

// The named fields of the slot-major arrays (elem_index): `nslot` slots from `slot0` of every record of `array`
// (`ns` slots per record).  `full`: UnOCPSolver keeps the field on N + 1 stages; every other field, and every field of
// UnParNMPCSolver, has N.
struct Field {
  const char* name;
  double* Layout::*array;
  int ns, slot0, nslot;
  bool full;
};
static const Field kFields[] = {
    {"lmd", &Layout::X, X_NUM, X_LMD, 1, true},        {"gmm", &Layout::X, X_NUM, X_GMM, 1, true},
    {"q", &Layout::X, X_NUM, X_Q, 1, true},            {"v", &Layout::X, X_NUM, X_V, 1, true},
    {"a", &Layout::X, X_NUM, X_A, 1, false},           {"u", &Layout::X, X_NUM, X_U, 1, false},
    {"beta", &Layout::X, X_NUM, X_BETA, 1, false},
    {"dlmd", &Layout::D, D_NUM, D_LMD, 1, true},       {"dgmm", &Layout::D, D_NUM, D_GMM, 1, true},
    {"dq", &Layout::D, D_NUM, D_Q, 1, true},           {"dv", &Layout::D, D_NUM, D_V, 1, true},
    {"da", &Layout::D, D_NUM, D_A, 1, false},          {"du", &Layout::D, D_NUM, D_U, 1, false},
    {"dbeta", &Layout::D, D_NUM, D_BETA, 1, false},
    {"slack", &Layout::X, X_NUM, X_SLACK, NC, false},  {"dual", &Layout::X, X_NUM, X_DUAL, NC, false},
    {"acc_slack", &Layout::XA, XA_NUM, 0, 2, false},   {"acc_dual", &Layout::XA, XA_NUM, 2, 2, false},
};
static const Field* find_field(const char* name) {
  if (name)
    for (const Field& f : kFields)
      if (!std::strcmp(name, f.name)) return &f;
  return nullptr;
}
// the fields of getSolution / getStageSolution: one slot of X
static const Field* solution_field(const char* name) {
  const Field* f = find_field(name);
  return f && f->array == &Layout::X && f->nslot == 1 ? f : nullptr;
}
static int field_stages(const idocp_b200_solver* h, const Field& f) {
  return f.full && h->kind == IDOCP_B200_SOLVER_UNOCP ? h->N + 1 : h->N;
}

extern "C" int idocp_b200_set_solution(idocp_b200_solver* h, const char* name, const double* value, int broadcast) {
  if (!h || !value) return fail(IDOCP_B200_INVALID_ARGUMENT, "set_solution: null pointer");
  const Field* fld = solution_field(name);
  const int f = fld ? fld->slot0 : -1;
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

static int ensure_line_search(idocp_b200_solver* h) {
  if (h->ls_ready) return IDOCP_B200_OK;
  const size_t N = h->N, Bp = h->Bp;
  int rc = 0;
  rc |= h->alloc(&h->LS.cost, (N + 1) * Bp);
  rc |= h->alloc(&h->LS.viol, N * Bp);
  rc |= h->alloc_filter(&h->LS.f, Bp);
  if (rc != 0) return fail(IDOCP_B200_CUDA_ERROR, "line-search buffers: device memory allocation failed");
  h->ls_ready = true;
  return IDOCP_B200_OK;
}

// The filter line search of both families for the whole batch, without host synchronisation: eval(mode) enqueues the
// family's cost / violation kernel (mode 0: the current point, 1: the trial point), filter(mode) its filter round
template <typename Eval, typename Filter>
static void enqueue_line_search_rounds(Eval eval, Filter filter) {
  eval(0);
  filter(0);
  for (int trial = 0; trial < LS_MAX_TRIALS; ++trial) {
    eval(1);
    filter(1);
  }
}

// UnLineSearch::computeStepSize for the whole batch
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
    with_flag(task, [&](auto T) { with_flag(par, [&](auto PAR) { with_flag(h->iref(), [&](auto IR) {
      IDOCP_LAUNCH(h, KC_LINESEARCH, (k_ls_eval<decltype(T)::value, decltype(PAR)::value, decltype(IR)::value>), grid, CTA_THREADS, 0,
                   h->d_prob, h->L, h->LS, mode, off, d_q, d_v);
    }); }); });
  };
  enqueue_line_search_rounds(eval, [&](int mode) {
    IDOCP_LAUNCH(h, KC_LINESEARCH, k_ls_filter, fgrid, 128, 0, h->L, h->LS, mode, ncost);
  });
  CUDA_OK(cudaGetLastError());
  return IDOCP_B200_OK;
}

// k_linearize / k_expand instantiation by the run-time problem flags (task-space cost, acceleration limits, per-instance references)
template <bool RES, bool BE>
static void launch_linearize(idocp_b200_solver* h, int cls, int nstages, const double* d_q, const double* d_v) {
  const int grid = stage_grid(h, nstages);
  with_flag(h->prob.task_enabled != 0, [&](auto task) { with_flag(h->L.XA != nullptr, [&](auto acc) { with_flag(h->iref(), [&](auto iref) {
    IDOCP_LAUNCH(h, cls, (k_linearize<RES, BE, decltype(task)::value, decltype(acc)::value, decltype(iref)::value>), grid, CTA_THREADS,
                 kLinSmem, h->d_prob, h->L, d_q, d_v);
  }); }); });
}
template <bool PARNMPC>
static void launch_expand(idocp_b200_solver* h, int nstages, int stage_offset) {
  // UnParNMPCSolver has no terminal stage, the only place k_expand reads a reference
  const int grid = stage_grid(h, nstages);
  with_flag(!PARNMPC && h->prob.task_enabled != 0, [&](auto task) { with_flag(h->L.XA != nullptr, [&](auto acc) {
    with_flag(!PARNMPC && h->iref(), [&](auto iref) {
      IDOCP_LAUNCH(h, KC_EXPAND, (k_expand<PARNMPC, decltype(task)::value, decltype(acc)::value, decltype(iref)::value>), grid,
                   CTA_THREADS, 0, h->d_prob, h->L, stage_offset);
    });
  }); });
}

// the persistent update + linearisation (k_update_linearize) of the run-time flags
static void launch_update_linearize(idocp_b200_solver* h, int grid) {
  with_flag(h->prob.task_enabled != 0, [&](auto task) { with_flag(h->kkt_tracking, [&](auto kkt) { with_flag(h->iref(), [&](auto iref) {
    IDOCP_LAUNCH(h, KC_UPDATE_LINEARIZE, (k_update_linearize<decltype(task)::value, decltype(kkt)::value, decltype(iref)::value>), grid,
                 UL_THREADS, kUlSmem, h->d_prob, h->L);
  }); }); });
}

static int unocp_update(idocp_b200_solver* h, const double* d_q, const double* d_v, int line_search) {
  // the terminal blocks come from record N of KQ with a task-space cost or per-instance references (k_riccati<true>)
  const bool task = h->prob.task_enabled != 0 || h->iref();
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
    override_alpha = h->LS.f.alpha;
  }
  if (h->pipelined) {
    // step sizes, then update + linearisation of the new iterate in one persistent launch; X (old) -> X2 (new), then the
    // two swap roles
    IDOCP_LAUNCH(h, KC_STEP_MIN, k_step_min, (h->Bp + 127) / 128, 128, 0, h->L, override_alpha);
    const long ul_tasks = static_cast<long>(h->N + 1) * h->L.G;
    const int ul_grid = static_cast<int>(std::min<long>((ul_tasks + UL_WARPS - 1) / UL_WARPS, static_cast<long>(UL_CTAS_PER_SM) * h->sm_count));
    launch_update_linearize(h, ul_grid);
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
    override_alpha = h->LS.f.alpha;
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
  if (h->prob.task_enabled && h->L.itask)
    IDOCP_LAUNCH(h, KC_MISC, (k_parnmpc_init_aux<true, true>), stage_grid(h, h->N), CTA_THREADS, kLinSmem, h->d_prob, h->L, h->PL);
  else if (h->prob.task_enabled)
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
  if (!q || !v) return fail(IDOCP_B200_INVALID_ARGUMENT, "q / v: null pointer");
  int rc = h->upload_state(q, static_cast<size_t>(h->B) * NV, v, static_cast<size_t>(h->B) * NV);
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
  if (!q || !v) return fail(IDOCP_B200_INVALID_ARGUMENT, "q / v: null pointer");
  int rc = h->upload_state(q, static_cast<size_t>(h->B) * NV, v, static_cast<size_t>(h->B) * NV);
  if (rc != IDOCP_B200_OK) return rc;
  rc = idocp_b200_compute_kkt_residual_device(h, t, h->d_q0, h->d_v0);
  if (h->wait_for_uploads() != 0) return fail(IDOCP_B200_CUDA_ERROR, "upload of q / v failed");
  return rc;
}

extern "C" int idocp_b200_kkt_error(idocp_b200_solver* h, double* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "kkt_error: null pointer");
  CUDA_OK(cudaSetDevice(h->device));
  return h->download(out, h->L.kkt_err, static_cast<size_t>(h->B) * sizeof(double));
}

// out[b][i][c][j] = src[elem_index(ns, G, stage0 + i, b, slot0 + c, j)] for b < B, i < nstage, c < nslot, j < NV
__global__ void k_gather(const double* __restrict__ src, int ns, int G, int B, int stage0, int nstage, int slot0, int nslot,
                         double* __restrict__ out) {
  const long idx = static_cast<long>(blockIdx.x) * blockDim.x + threadIdx.x;
  const long total = static_cast<long>(B) * nstage * nslot * NV;
  if (idx >= total) return;
  const int j = static_cast<int>(idx % NV);
  long t = idx / NV;
  const int c = static_cast<int>(t % nslot);
  t /= nslot;
  const int i = static_cast<int>(t % nstage);
  const int b = static_cast<int>(t / nstage);
  out[idx] = src[elem_index(ns, G, stage0 + i, b, slot0 + c, j)];
}

// field f of stages stage0 .. stage0 + nstage - 1 of the whole batch: out[b][stage][slot][7]
static int gather_to_host(idocp_b200_solver* h, const Field& f, int stage0, int nstage, double* out) {
  const long total = static_cast<long>(h->B) * nstage * f.nslot * NV;
  if (static_cast<size_t>(total) > h->stage_doubles) return fail(IDOCP_B200_INVALID_ARGUMENT, "staging buffer too small");
  CUDA_OK(cudaSetDevice(h->device));
  IDOCP_LAUNCH(h, KC_MISC, k_gather, static_cast<int>((total + 255) / 256), 256, 0, h->L.*f.array, f.ns, h->L.G, h->B, stage0,
               nstage, f.slot0, f.nslot, h->d_stage);
  CUDA_OK(cudaGetLastError());
  return h->download(out, h->d_stage, total * sizeof(double));
}

extern "C" int idocp_b200_get_solution(idocp_b200_solver* h, const char* name, double* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_solution: null pointer");
  const Field* f = solution_field(name);
  if (!f) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_solution: unknown field");
  return gather_to_host(h, *f, 0, field_stages(h, *f), out);
}

// one stage of one field: out[b][7]
extern "C" int idocp_b200_get_stage_solution(idocp_b200_solver* h, const char* name, int stage, double* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_stage_solution: null pointer");
  const Field* f = solution_field(name);
  if (!f) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_stage_solution: unknown field");
  if (stage < 0 || stage >= field_stages(h, *f))
    return fail(IDOCP_B200_INVALID_ARGUMENT, "get_stage_solution: stage out of range");
  return gather_to_host(h, *f, stage, 1, out);
}

extern "C" int idocp_b200_get_direction(idocp_b200_solver* h, const char* name, double* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_direction: null pointer");
  const Field* f = find_field(name);
  if (!f || f->array != &Layout::D) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_direction: unknown field");
  return gather_to_host(h, *f, 0, field_stages(h, *f), out);
}

// out[b][N][6][7] (slack, dual: the six joint-limit components) or out[b][N][2][7] (acc_slack, acc_dual: the two
// acceleration-limit components)
extern "C" int idocp_b200_get_constraint_data(idocp_b200_solver* h, const char* name, double* out) {
  if (!h || !out || !name) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_constraint_data: null pointer");
  const Field* f = find_field(name);
  if (!f || f->nslot == 1)
    return fail(IDOCP_B200_INVALID_ARGUMENT, "get_constraint_data: name must be slack, dual, acc_slack or acc_dual");
  if (!(h->L.*f->array)) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_constraint_data: the acceleration limits are not enabled");
  return gather_to_host(h, *f, 0, h->N, out);
}

extern "C" int idocp_b200_get_step_sizes(idocp_b200_solver* h, double* primal, double* dual) {
  if (!h) return fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
  CUDA_OK(cudaSetDevice(h->device));
  const size_t n = static_cast<size_t>(h->B) * sizeof(double);
  const int rc = primal ? h->download(primal, h->L.steps, n) : IDOCP_B200_OK;
  return rc == IDOCP_B200_OK && dual ? h->download(dual, h->L.steps + h->Bp, n) : rc;
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
  const int rc = h->download(Q, dQ, static_cast<size_t>(h->B) * 441 * sizeof(double));
  return rc == IDOCP_B200_OK ? h->download(res, dres, static_cast<size_t>(h->B) * 35 * sizeof(double)) : rc;
}

extern "C" int idocp_b200_get_status(idocp_b200_solver* h, int* out) {
  if (!h || !out) return fail(IDOCP_B200_INVALID_ARGUMENT, "get_status: null pointer");
  CUDA_OK(cudaSetDevice(h->device));
  return h->download(out, h->L.status, static_cast<size_t>(h->B) * sizeof(int));
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
  return h->download(out, d, static_cast<size_t>(h->B) * sizeof(int));
}

extern "C" int idocp_b200_clear_line_search_filter(idocp_b200_solver* h) {
  if (!h) return fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
  if (!h->ls_ready) return IDOCP_B200_OK;  // never used: already empty
  CUDA_OK(cudaSetDevice(h->device));
  IDOCP_LAUNCH(h, KC_LINESEARCH, k_ls_clear, (h->B + 127) / 128, 128, 0, h->LS.f.n, h->B);
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
  h->lin_valid = false; h->kkt_valid = false;                       // the kept linearisation used the old reference
  return h->upload(h->L.task_ref, table, static_cast<size_t>(h->N + 1) * 12 * sizeof(double));
}

// Per-instance cost references.  Every set / clear invalidates the kept linearisation (it was made with the old references);
// the line-search filter is left as it is, as on a change of the shared references.  Padded instances (B <= b < Bp) repeat
// the last instance: they are computed but never reported.
extern "C" int idocp_b200_set_instance_reference(idocp_b200_solver* h, const char* name, const double* value) {
  if (!h || !name || !value) return fail(IDOCP_B200_INVALID_ARGUMENT, "set_instance_reference: null pointer");
  const int field = !std::strcmp(name, "q_ref") ? IREF_Q : !std::strcmp(name, "v_ref") ? IREF_V : !std::strcmp(name, "u_ref") ? IREF_U : -1;
  if (field < 0) return fail(IDOCP_B200_INVALID_ARGUMENT, "invalid argument: name must be q_ref, v_ref, or u_ref!");
  CUDA_OK(cudaSetDevice(h->device));
  const size_t B = h->B, Bp = h->Bp, G = h->L.G;
  if (!h->d_iref && h->alloc(&h->d_iref, G * IREF_NUM * SLOT) != 0)
    return fail(IDOCP_B200_CUDA_ERROR, "set_instance_reference: device memory allocation failed");
  if (!h->L.iref) {   // entering per-instance mode: the fields not set yet start as copies of the problem's
    h->iref_host.assign(B * IREF_NUM * NV, 0.0);
    for (size_t b = 0; b < B; ++b)
      for (int j = 0; j < NV; ++j) {
        h->iref_host[(b * IREF_NUM + IREF_Q) * NV + j] = h->prob.q_ref[j];
        h->iref_host[(b * IREF_NUM + IREF_V) * NV + j] = h->prob.v_ref[j];
        h->iref_host[(b * IREF_NUM + IREF_U) * NV + j] = h->prob.u_ref[j];
      }
  }
  for (size_t b = 0; b < B; ++b)
    for (int j = 0; j < NV; ++j) h->iref_host[(b * IREF_NUM + field) * NV + j] = value[b * NV + j];
  // [b][field][j] -> [group][field][b & 3][lane], padding lane 7 zero as DevProblem's
  std::vector<double> dev(G * IREF_NUM * SLOT, 0.0);
  for (size_t b = 0; b < Bp; ++b)
    for (int f = 0; f < IREF_NUM; ++f)
      for (int j = 0; j < NV; ++j)
        dev[elem_index(IREF_NUM, static_cast<int>(G), 0, static_cast<int>(b), f, j)] = h->iref_host[((b < B ? b : B - 1) * IREF_NUM + f) * NV + j];
  const int rc = h->upload(h->d_iref, dev.data(), dev.size() * sizeof(double));
  if (rc != IDOCP_B200_OK) return rc;
  h->L.iref = h->d_iref;
  h->lin_valid = false; h->kkt_valid = false;
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_set_instance_task_reference(idocp_b200_solver* h, const double* table) {
  if (!h || !table) return fail(IDOCP_B200_INVALID_ARGUMENT, "set_instance_task_reference: null pointer");
  if (!h->prob.task_enabled)
    return fail(IDOCP_B200_INVALID_ARGUMENT, "invalid argument: set_instance_task_reference needs a task-space cost (task_enabled == 0)!");
  CUDA_OK(cudaSetDevice(h->device));
  const size_t B = h->B, Bp = h->Bp, rows = static_cast<size_t>(h->N) + 1;
  if (!h->d_itask && h->alloc(&h->d_itask, rows * Bp * 12) != 0)
    return fail(IDOCP_B200_CUDA_ERROR, "set_instance_task_reference: device memory allocation failed");
  // [b][row][12] -> [row][b][12]: the four instances of a (stage, group) task are 48 contiguous doubles
  std::vector<double> dev(rows * Bp * 12);
  for (size_t i = 0; i < rows; ++i)
    for (size_t b = 0; b < Bp; ++b)
      std::memcpy(&dev[(i * Bp + b) * 12], table + ((b < B ? b : B - 1) * rows + i) * 12, 12 * sizeof(double));
  const int rc = h->upload(h->d_itask, dev.data(), dev.size() * sizeof(double));
  if (rc != IDOCP_B200_OK) return rc;
  h->L.itask = h->d_itask;
  h->lin_valid = false; h->kkt_valid = false;
  return IDOCP_B200_OK;
}

extern "C" int idocp_b200_clear_instance_references(idocp_b200_solver* h) {
  if (!h) return fail(IDOCP_B200_INVALID_ARGUMENT, "null handle");
  h->L.iref = nullptr;
  h->L.itask = nullptr;
  h->lin_valid = false; h->kkt_valid = false;
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
