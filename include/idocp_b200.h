/*
 * idocp_b200.h -- C-ABI of the B200-native batched optimal-control engine.
 *
 * Drop-in boundary for idocp's data-parallel Newton-step hot path.  The reference
 * (mayataka/idocp) has no FFI; its "operator API" for this path is the public C++ interface
 * of its solver classes.  Each entry point below replaces one of those methods for a BATCH
 * of independent OCP instances (the reference solves one instance per solver object), and the
 * C++ host classes in include/idocp_b200/ (*.hpp) re-create the reference's class API on top.
 *
 * Conventions
 *  - plain pointers and sizes, no torch / Eigen types;
 *  - every function returns 0 on success, a negative idocp_b200_status on error, and never
 *    exits the process (the reference prints + std::exit, unocp_solver.cpp:33-47); the text of
 *    the last error of the calling thread is returned by idocp_b200_last_error();
 *  - host arrays are row-major [batch][...]; `dimv` = 7 for the iiwa14;
 *  - one handle = one CUDA device + one stream; calls on a handle are serialised, asynchronous
 *    with respect to the host until a getter / idocp_b200_sync();
 *  - there is NO CPU fallback: creation fails when no CUDA device is usable.
 */
#ifndef IDOCP_B200_H_
#define IDOCP_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

#define IDOCP_B200_DIMV 7          /* iiwa14: nq = nv = nu */
#define IDOCP_B200_NUM_CONSTRAINTS 6 /* JointConstraintsFactory: pos/vel/torque x lower/upper */

typedef enum {
  IDOCP_B200_OK = 0,
  IDOCP_B200_INVALID_ARGUMENT = -1,
  IDOCP_B200_CUDA_ERROR = -2,
  IDOCP_B200_NO_DEVICE = -3,
  IDOCP_B200_UNSUPPORTED = -4
} idocp_b200_status;

/* per-instance numerical status bits (idocp_b200_get_status) -- the reference only asserts in
 * Debug builds (split_unriccati_factorizer.hxx:38,41-42) */
#define IDOCP_B200_STATUS_CHOL_FAIL 1  /* a Cholesky pivot was <= 0 or NaN */
#define IDOCP_B200_STATUS_NAN       2  /* a step size / KKT error was NaN */
#define IDOCP_B200_STATUS_FILTER_FULL 4  /* the line-search filter held its 256 entries: a new entry was dropped */

typedef enum {
  IDOCP_B200_ROBOT_IIWA14 = 0
} idocp_b200_robot;

typedef enum {
  IDOCP_B200_SOLVER_UNOCP = 0,     /* idocp::UnOCPSolver      (include/idocp/unocp/unocp_solver.hpp:25-188)   */
  IDOCP_B200_SOLVER_UNPARNMPC = 1  /* idocp::UnParNMPCSolver  (include/idocp/unocp/unparnmpc_solver.hpp:37-171) */
} idocp_b200_solver_kind;

/*
 * Problem descriptor = the closed, POD form of what the reference builds from plug-ins:
 *   Robot limits             robot/robot.hxx:699-709, Robot::setJointEffortLimit/VelocityLimit
 *   ConfigurationSpaceCost   src/cost/configuration_space_cost.cpp:241-396
 *   JointConstraintsFactory  src/utils/joint_constraints_factory.cpp:22-37 (six joint-limit
 *                            components, barrier / fraction-to-boundary of
 *                            constraints/joint_position_lower_limit.hpp:19-20)
 *   TimeVaryingTaskSpace6DCost (optional) src/cost/time_varying_task_space_6d_cost.cpp:68-195
 */
typedef struct {
  int robot;                /* idocp_b200_robot */
  int N;                    /* number of horizon stages  (UnOCPSolver ctor argument N) */
  double T;                 /* horizon length            (ctor argument T)             */
  double q_ref[IDOCP_B200_DIMV], v_ref[IDOCP_B200_DIMV], u_ref[IDOCP_B200_DIMV];
  double q_weight[IDOCP_B200_DIMV], v_weight[IDOCP_B200_DIMV], a_weight[IDOCP_B200_DIMV];
  double u_weight[IDOCP_B200_DIMV], qf_weight[IDOCP_B200_DIMV], vf_weight[IDOCP_B200_DIMV];
  double q_min[IDOCP_B200_DIMV], q_max[IDOCP_B200_DIMV];
  double v_max[IDOCP_B200_DIMV], u_max[IDOCP_B200_DIMV];
  double barrier;           /* 1e-4  */
  double fraction_rate;     /* 0.995 */
  int task_enabled;         /* task-space cost on the end-effector frame (frame id 22 of examples/iiwa14/task_space_ocp.cpp:67):
                               0 none; 1 TimeVaryingTaskSpace6DCost / TaskSpace6DCost (log6 pose error);
                               2 TimeVaryingTaskSpace3DCost / TaskSpace3DCost (src/cost/task_space_3d_cost.cpp: position error;
                               task_q_weight[0..2] = q_3d_weight, the reference table's rotation entries are ignored) */
  double task_q_weight[6], task_qf_weight[6]; /* [position xyz, rotation xyz] = the arguments of
                               set_q_6d_weight / set_qf_6d_weight (time_varying_task_space_6d_cost.cpp:43-58) */
  double task_center[3], task_radius, task_t0, task_tf; /* reserved (the reference is a host-sampled table) */
  double task_rot_ref[9];
  /* JointAccelerationLowerLimit / JointAccelerationUpperLimit (src/constraints/joint_acceleration_*_limit.cpp) with their
   * constructor arguments amin / amax: [0] lower, [1] upper.  While one is enabled the solver runs the literal kernel
   * sequence (no pipelining) with the kernel instantiations that carry the two extra components. */
  int enable_acceleration_limit[2];
  double a_min[IDOCP_B200_DIMV], a_max[IDOCP_B200_DIMV];
} idocp_b200_problem;

typedef struct idocp_b200_solver idocp_b200_solver; /* opaque */

/* fills robot limits (URDF), barrier 1e-4, fraction 0.995, N = 20, T = 1, zero weights */
int idocp_b200_problem_default(int robot, idocp_b200_problem* p);

/* UnOCPSolver::UnOCPSolver(robot, cost, constraints, T, N, nthreads) / UnParNMPCSolver ctor
 * (src/unocp/unocp_solver.cpp:11-49).  `nthreads` has no meaning on the GPU and is not taken.
 * Like the reference ctor it ends with initConstraints() on the zero solution. */
int idocp_b200_create(const idocp_b200_problem* p, int solver_kind, int batch, int device,
                      idocp_b200_solver** out);
int idocp_b200_destroy(idocp_b200_solver* h);

/* UnOCPSolver::setSolution(name, value) (unocp_solver.cpp:157-181): name in {"q","v","a","u"};
 * broadcast != 0: value[dimv] is written to every stage of every instance (the reference call);
 * broadcast == 0: value[batch][dimv] gives each instance its own vector (all stages).
 * Ends with initConstraints() like the reference. */
int idocp_b200_set_solution(idocp_b200_solver* h, const char* name, const double* value, int broadcast);
/* UnOCPSolver::initConstraints() (unocp_solver.cpp:59-70) */
int idocp_b200_init_constraints(idocp_b200_solver* h);
/* UnParNMPCSolver::initBackwardCorrection(t) (src/unocp/unparnmpc_solver.cpp:69-71) */
int idocp_b200_init_backward_correction(idocp_b200_solver* h, double t);

/* UnOCPSolver::updateSolution(t, q, v, line_search) (unocp_solver.cpp:73-134), one SQP
 * iteration of every instance.  q, v: HOST arrays [batch][dimv] (initial state per instance), pageable or pinned: the
 * call returns once q and v have been copied (an event behind the H2D copies), so the caller may rewrite them at once;
 * the kernels of the iteration are still running then (asynchronous until idocp_b200_sync or a getter).  The same
 * holds for compute_kkt_residual and the idocp_b200_fb_* twins. */
int idocp_b200_update_solution(idocp_b200_solver* h, double t, const double* q, const double* v,
                               int line_search);
/* same, q and v already resident in device memory ([batch][dimv] doubles on the handle's device) */
int idocp_b200_update_solution_device(idocp_b200_solver* h, double t, const double* d_q,
                                      const double* d_v, int line_search);
/* UnOCPSolver::computeKKTResidual(t, q, v) (unocp_solver.cpp:205-225) */
int idocp_b200_compute_kkt_residual(idocp_b200_solver* h, double t, const double* q, const double* v);
int idocp_b200_compute_kkt_residual_device(idocp_b200_solver* h, double t, const double* d_q,
                                           const double* d_v);
/* UnOCPSolver::KKTError() (unocp_solver.cpp:190-202): out[batch]; reads the residual buffers of
 * the last computeKKTResidual, exactly like the reference. */
int idocp_b200_kkt_error(idocp_b200_solver* h, double* out);

/* UnOCPSolver::getSolution(name) (unocp_solver.cpp:240-264): name in
 * {"q","v","lmd","gmm"} -> out[batch][N+1][dimv]; {"a","u","beta"} -> out[batch][N][dimv]
 * (UnParNMPC: N stages for every field). */
int idocp_b200_get_solution(idocp_b200_solver* h, const char* name, double* out);
/* UnOCPSolver::getSolution(int stage) (unocp_solver.cpp:137-141), one field of one stage:
 * out[batch][dimv] */
int idocp_b200_get_stage_solution(idocp_b200_solver* h, const char* name, int stage, double* out);
/* Newton direction of the last updateSolution ({"dq","dv","dlmd","dgmm"}: N+1 stages;
 * {"da","du","dbeta"}: N stages) -- for parity tests; the reference keeps it in d_ */
int idocp_b200_get_direction(idocp_b200_solver* h, const char* name, double* out);
/* ConstraintComponentData fields {"slack","dual"}: out[batch][N][6][dimv] (inactive rows 0) */
int idocp_b200_get_constraint_data(idocp_b200_solver* h, const char* name, double* out);
/* primal / dual step sizes of the last updateSolution, out arrays [batch] (either may be NULL) */
int idocp_b200_get_step_sizes(idocp_b200_solver* h, double* primal, double* dual);
/* condensed KKT data of the last linearisation for one stage (parity tests):
 * Q[batch][21*21] column-major in block order (a,q,v) as SplitUnKKTMatrix, lower blocks
 * (qa, va) left zero; res[batch][35] = [Fq,Fv,la,lq,lv] as SplitUnKKTResidual */
int idocp_b200_get_unkkt(idocp_b200_solver* h, int stage, double* Q, double* res);
int idocp_b200_get_status(idocp_b200_solver* h, int* out);
/* UnOCPSolver::isCurrentSolutionFeasible() (unocp_solver.cpp:228-237): out[batch] 0/1 */
int idocp_b200_is_feasible(idocp_b200_solver* h, int* out);
/* UnOCPSolver::clearLineSearchFilter() (unocp_solver.cpp:185-187) */
int idocp_b200_clear_line_search_filter(idocp_b200_solver* h);

/* TimeVaryingTaskSpace6DRefBase::compute_q_6d_ref(t, SE3&) (cost/time_varying_task_space_6d_cost.hpp:39-40)
 * is a user-derived host virtual: the host layer samples it at the time of every stage index and hands the
 * samples over as table[N+1][12] = [R_ref row-major (9), p_ref (3)]:
 *   UnOCPSolver     row i = t + i dt (i < N), row N = t + T        (unocp_solver.cpp:80-93)
 *   UnParNMPCSolver row i = t + (i+1) dt (i < N-1), row N-1 = t + T (unbackward_correction.cpp:73-95), row N unused
 * Call it before updateSolution / computeKKTResidual / initBackwardCorrection whenever t changes. */
int idocp_b200_set_task_reference(idocp_b200_solver* h, const double* table);

/* Per-instance cost references: the counterpart of one reference solver object per instance, each with its own
 * ConfigurationSpaceCost::set_q_ref / set_v_ref / set_u_ref and its own task-space reference.  A handle starts in shared mode
 * (the problem's q_ref / v_ref / u_ref, the table of idocp_b200_set_task_reference for every instance).
 *   set_instance_reference: name in {"q_ref", "v_ref", "u_ref"}, value[batch][7].  The first call switches the
 *     configuration-space cost to per-instance references; the two other fields start as copies of the problem's.
 *   set_instance_task_reference: table[batch][N+1][12] = [R row-major (9), p (3)], rows as idocp_b200_set_task_reference
 *     (a constant target: every row the same).  Switches the task-space cost to per-instance tables; the shared table that
 *     idocp_b200_set_task_reference keeps writing is stored but not read until the clear.  Needs task_enabled != 0.
 *   clear_instance_references: back to the problem's references and the last shared table.
 * Every call invalidates the linearisation a pipelined UnOCPSolver keeps for its next updateSolution.  The line-search
 * filter is NOT cleared, as on a change of the shared references; call idocp_b200_clear_line_search_filter for a fresh
 * start.  Instance b gives the bits of a shared-mode handle whose problem / table hold instance b's references.  The
 * DerivativeChecker (idocp_b200_check_cost_derivatives) always uses the shared references. */
int idocp_b200_set_instance_reference(idocp_b200_solver* h, const char* name, const double* value);
int idocp_b200_set_instance_task_reference(idocp_b200_solver* h, const double* table);
int idocp_b200_clear_instance_references(idocp_b200_solver* h);

/* Device-side analogue of idocp::DerivativeChecker (include/idocp/utils/derivative_checker.hpp:14-66,
 * src/utils/derivative_checker.cpp:47-312) for the cost of this handle's problem: for n samples of a split solution
 * (q, v, a, u rows [n][7], host pointers) the kernel evaluates the cost with the device functions of the line search and its
 * gradient / Hessian with those of the lineariser, and forms the forward differences the reference compares them with
 * (step finite_diff).  kind 0: stage cost (includes dt = T / N), 1: terminal cost; the task-space reference is row `stage`
 * of the table of idocp_b200_set_task_reference.  out[n][IDOCP_B200_DC_DOUBLES]:
 *   [0] cost | [1..28] lq, lv, la, lu | [29..56] their forward differences | [57..105] Qqq (row-major 7 x 7) |
 *   [106..126] diagonals of Qvv, Qaa, Quu | [127..175], [176..224], [225..273], [274..322] forward differences of the
 *   gradient: Qqq, Qvv, Qaa, Quu (row-major, column i = coordinate i moved).
 * The comparison itself (Eigen's isApprox with the test tolerance) is the host classes' (DerivativeChecker in
 * include/idocp_b200/idocp_b200.hpp and idocp_b200/solvers.py). */
#define IDOCP_B200_DC_DOUBLES 323
int idocp_b200_check_cost_derivatives(idocp_b200_solver* h, int kind, int stage, int n, const double* q, const double* v,
                                      const double* a, const double* u, double finite_diff, double* out);

int idocp_b200_sync(idocp_b200_solver* h);
/* number of kernels this handle has launched since creation (bench.py "gpu_launches") */
int idocp_b200_launch_count(idocp_b200_solver* h, long long* out);
/* CUDA stream of the handle as an opaque pointer (for event timing on the launching stream) */
int idocp_b200_stream(idocp_b200_solver* h, void** out);
/* per-kernel-class device time: while profiling is enabled every launch is bracketed by CUDA
 * events on the launching stream (no host sync inside the timed region); get_profile resolves them:
 * names[i], total ms[i], calls[i]; returns the number of entries (<= cap) */
/* UnOCPSolver only, default enabled = 1: updateSolution applies its step and linearises the NEW iterate in one launch
 * (the linearisation does not depend on the measured state), and the next updateSolution re-uses it unless setSolution /
 * initConstraints / set_task_reference intervened.  Results are bit-identical either way; with enabled = 0 the call is the
 * reference's literal sequence linearise, Riccati, expand, update (unocp_solver.cpp:73-134) and get_unkkt shows the
 * linearisation the last direction came from. */
int idocp_b200_set_pipelining(idocp_b200_solver* h, int enabled);
int idocp_b200_set_profiling(idocp_b200_solver* h, int enabled);
int idocp_b200_get_profile(idocp_b200_solver* h, int cap, const char** names, double* ms, long long* calls);

/* ------------------------------------------------------------------------------------------------------------
 * One solver object over several GPUs of one node (SURVEY.md section 8e: the batch of independent OCP instances is
 * split into contiguous shards, one device + stream per shard, NO collective on the hot path).  The reference's
 * counterpart is the `nthreads` argument of its solver constructors (OpenMP over stages, unocp_solver.cpp:11-49):
 * here the parallel resource is the list of devices.  Every call forwards to the shards with the caller's
 * [batch][...] arrays offset to each shard's first instance; the per-shard calls only enqueue work, so all GPUs
 * run concurrently; getters and sync wait for every shard.  Results are those of one idocp_b200_solver over the
 * whole batch, instance by instance (tests/test_sharded_solver.py).
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct idocp_b200_sharded idocp_b200_sharded; /* opaque */
int idocp_b200_create_sharded(const idocp_b200_problem* p, int solver_kind, int batch, const int* devices,
                              int n_devices, idocp_b200_sharded** out);
int idocp_b200_sharded_destroy(idocp_b200_sharded* s);
/* number of shards and (first != NULL) the first instance of every shard, first[n] = batch */
int idocp_b200_sharded_num_shards(const idocp_b200_sharded* s, int* n, int* first);
/* the single-device solver behind shard `index` (borrowed; for the device-pointer entry points and the profile) */
int idocp_b200_sharded_shard(idocp_b200_sharded* s, int index, idocp_b200_solver** out);
int idocp_b200_sharded_set_solution(idocp_b200_sharded* s, const char* name, const double* value, int broadcast);
int idocp_b200_sharded_init_constraints(idocp_b200_sharded* s);
int idocp_b200_sharded_init_backward_correction(idocp_b200_sharded* s, double t);
int idocp_b200_sharded_set_task_reference(idocp_b200_sharded* s, const double* table);
int idocp_b200_sharded_set_instance_reference(idocp_b200_sharded* s, const char* name, const double* value /* [batch][7] */);
int idocp_b200_sharded_set_instance_task_reference(idocp_b200_sharded* s, const double* table /* [batch][N+1][12] */);
int idocp_b200_sharded_clear_instance_references(idocp_b200_sharded* s);
int idocp_b200_sharded_update_solution(idocp_b200_sharded* s, double t, const double* q, const double* v, int line_search);
int idocp_b200_sharded_compute_kkt_residual(idocp_b200_sharded* s, double t, const double* q, const double* v);
int idocp_b200_sharded_kkt_error(idocp_b200_sharded* s, double* out /* [batch] */);
int idocp_b200_sharded_get_solution(idocp_b200_sharded* s, const char* name, double* out /* [batch][stages][dimv] */);
int idocp_b200_sharded_get_stage_solution(idocp_b200_sharded* s, const char* name, int stage, double* out /* [batch][dimv] */);
int idocp_b200_sharded_get_step_sizes(idocp_b200_sharded* s, double* primal, double* dual);
int idocp_b200_sharded_get_status(idocp_b200_sharded* s, int* out);
int idocp_b200_sharded_clear_line_search_filter(idocp_b200_sharded* s);
int idocp_b200_sharded_sync(idocp_b200_sharded* s);

/* ------------------------------------------------------------------------------------------------------------
 * Host-side contact schedule of the hybrid OCP (SURVEY.md section 8, row a13; implementation
 * include/idocp_b200/hybrid.hpp; no device work).  Contact activity arrays are int[max_point_contacts] (0/1),
 * contact points double[max_point_contacts][3] (may be NULL = zeros).
 * ------------------------------------------------------------------------------------------------------------ */
typedef struct idocp_b200_contact_sequence idocp_b200_contact_sequence; /* opaque */
/* ContactSequence::ContactSequence(robot, max_num_events) (hybrid/contact_sequence.hxx:10-29): starts with one
 * phase without active contacts */
int idocp_b200_contact_sequence_create(int max_point_contacts, int max_num_events, idocp_b200_contact_sequence** out);
int idocp_b200_contact_sequence_destroy(idocp_b200_contact_sequence* cs);
/* setContactStatusUniformly (:50-54) */
int idocp_b200_contact_sequence_set_uniform(idocp_b200_contact_sequence* cs, const int* is_active,
                                            const double* contact_points);
/* push_back(contact_status, event_time) (:56-110): the event (impulse if a contact becomes active, else lift;
 * hybrid/discrete_event.hxx:78-104) between the last phase and the new status; errors carry the reference's text */
int idocp_b200_contact_sequence_push_back(idocp_b200_contact_sequence* cs, const int* is_active,
                                          const double* contact_points, double event_time);
int idocp_b200_contact_sequence_pop_back(idocp_b200_contact_sequence* cs);   /* :113-132 */
int idocp_b200_contact_sequence_pop_front(idocp_b200_contact_sequence* cs);  /* :135-154 */
/* updateImpulseTime / updateLiftTime (:157-240) */
int idocp_b200_contact_sequence_update_event_time(idocp_b200_contact_sequence* cs, int is_impulse, int index, double time);
/* setContactPoints(contact_phase, contact_points) (:243-262) */
int idocp_b200_contact_sequence_set_contact_points(idocp_b200_contact_sequence* cs, int contact_phase,
                                                   const double* contact_points);
/* numContactPhases / numImpulseEvents / numLiftEvents (:265-282); any pointer may be NULL */
int idocp_b200_contact_sequence_counts(const idocp_b200_contact_sequence* cs, int* num_contact_phases,
                                       int* num_impulse_events, int* num_lift_events);
/* contactStatus(contact_phase) / impulseStatus(impulse_index) + impulseTime / liftTime (:285-316) */
int idocp_b200_contact_sequence_get_phase(const idocp_b200_contact_sequence* cs, int contact_phase, int* is_active,
                                          double* contact_points);
int idocp_b200_contact_sequence_get_impulse(const idocp_b200_contact_sequence* cs, int impulse_index, int* is_active,
                                            double* contact_points, double* time);
int idocp_b200_contact_sequence_get_lift_time(const idocp_b200_contact_sequence* cs, int lift_index, double* time);

#define IDOCP_B200_MAX_GRID 1024   /* capacity of the tables below: N <= 1024 grid stages, <= 64 events */
#define IDOCP_B200_MAX_EVENTS 64
/* one row of the flattened schedule, in the order the Riccati recursion visits the stages
 * (src/ocp/riccati_recursion_solver.cpp:48-107): kind 0 grid, 1 impulse, 2 aux, 3 lift, 4 terminal */
typedef struct {
  int kind, index;
  double t, dt;
  int contact_phase;      /* ContactSequence::contactStatus(contact_phase) is active on the stage */
  int constraint_stage;   /* constraints mask index: grid index; 0 for aux / lift; -1 impulse (ocp_linearizer.cpp:40-68) */
  int before_impulse;     /* the switching constraint of impulse `switching_impulse` is imposed on this grid stage */
  int switching_impulse;
} idocp_b200_scheduled_stage;
/* OCPDiscretizer after discretizeOCP(contact_sequence, t) (hybrid/ocp_discretizer.hxx:61-72, getters :75-202) */
typedef struct {
  int well_defined;       /* isWellDefined() and every event inside the horizon found its stage */
  int N, N_impulse, N_lift;
  double t[IDOCP_B200_MAX_GRID + 1], dt[IDOCP_B200_MAX_GRID + 1];
  int contact_phase[IDOCP_B200_MAX_GRID + 1];
  int impulse_index_after_time_stage[IDOCP_B200_MAX_GRID + 1], lift_index_after_time_stage[IDOCP_B200_MAX_GRID + 1];
  int time_stage_before_impulse[IDOCP_B200_MAX_EVENTS], time_stage_before_lift[IDOCP_B200_MAX_EVENTS];
  double t_impulse[IDOCP_B200_MAX_EVENTS], t_lift[IDOCP_B200_MAX_EVENTS];
  double dt_aux[IDOCP_B200_MAX_EVENTS], dt_lift[IDOCP_B200_MAX_EVENTS];
  int num_stages;         /* = N + 1 + 2 N_impulse + N_lift when well defined */
  idocp_b200_scheduled_stage stages[IDOCP_B200_MAX_GRID + 1 + 3 * IDOCP_B200_MAX_EVENTS];
} idocp_b200_ocp_discretization;
int idocp_b200_discretize_ocp(const idocp_b200_contact_sequence* cs, double T, int N, double t,
                              idocp_b200_ocp_discretization* out);

/* ------------------------------------------------------------------------------------------------------------
 * OCPSolver for the floating-base robot (ANYmal: free-flyer + 12 joints, 4 point contacts), SURVEY.md section 8 row a12.
 * One handle = a batch of independent OCP instances that share the problem and the contact schedule and differ in the
 * initial state, in their iterates and, optionally, in the cost reference.  Mirrors
 *   OCPSolver(robot, cost, constraints, T, N, max_num_impulse, nthreads)   src/ocp/ocp_solver.cpp:10-48
 *   setSolution / initConstraints / updateSolution / computeKKTResidual / KKTError / getSolution
 *                                                                          src/ocp/ocp_solver.cpp:60-92,96-213,244-280
 * The contact schedule (setContactStatusUniformly, pushBackContactStatus, popBack/popFront, setContactPoints:
 * ocp_solver.cpp:173-194) is the idocp_b200_contact_sequence above; the handle borrows it and re-discretises it at
 * the t of every call.
 * Cost = configuration-space cost with a time-varying reference + contact-force cost:
 *   ConfigurationSpaceCost / TrottingConfigurationSpaceCost / TimeVaryingConfigurationSpaceCost
 *       (src/cost/trotting_configuration_space_cost.cpp:241-375): weights below, q_ref(t) / v_ref sampled by the host at
 *       the time of every stage (idocp_b200_fb_set_cost_reference), like the 6D reference of the iiwa14 path;
 *   ContactForceCost (src/cost/contact_force_cost.cpp:121-228): f_weight / f_ref, fi_weight / fi_ref (impulses).
 * Constraints = JointConstraintsFactory's six joint limits on the 12 actuated joints + LinearizedFrictionCone +
 * LinearizedImpulseFrictionCone (src/constraints/ *.cpp), enable[] in the order below; cone_nonlinear[0 / 1] selects
 * FrictionCone / ImpulseFrictionCone (friction_cone.cpp, impulse_friction_cone.cpp: two rows per contact, normal force and
 * fx^2 + fy^2 - mu^2 fz^2 <= 0) for the enabled cone; enable_acceleration_limit[0 / 1] adds JointAccelerationLowerLimit /
 * JointAccelerationUpperLimit (joint_acceleration_*_limit.cpp) with the bounds a_min / a_max on the 12 joint accelerations;
 * enable_contact_distance adds ContactDistance (contact_distance.cpp): the contact frames of the legs in the air stay above z = 0.
 * ------------------------------------------------------------------------------------------------------------ */
#define IDOCP_B200_FB_NQ 19
#define IDOCP_B200_FB_NV 18
#define IDOCP_B200_FB_NU 12
#define IDOCP_B200_FB_MAXF 12
enum idocp_b200_fb_constraint {
  IDOCP_B200_FB_POSITION_LOWER = 0, IDOCP_B200_FB_POSITION_UPPER, IDOCP_B200_FB_VELOCITY_LOWER, IDOCP_B200_FB_VELOCITY_UPPER,
  IDOCP_B200_FB_TORQUES_LOWER, IDOCP_B200_FB_TORQUES_UPPER, IDOCP_B200_FB_FRICTION_CONE, IDOCP_B200_FB_IMPULSE_FRICTION_CONE,
  IDOCP_B200_FB_NUM_CONSTRAINTS
};
typedef struct {
  double T;
  int N, max_num_impulse;
  double q_weight[18], v_weight[18], a_weight[18], qf_weight[18], vf_weight[18], qi_weight[18], vi_weight[18], dvi_weight[18];
  double f_weight[12], f_ref[12], fi_weight[12], fi_ref[12];   /* [contact][xyz] */
  double q_min[12], q_max[12], v_max[12], u_max[12];           /* Robot::*JointPositionLimit etc. (robot.hxx:699-709) */
  double mu, barrier, fraction_rate;                           /* friction coefficient; PDIPM barrier, fraction-to-boundary */
  int enable[IDOCP_B200_FB_NUM_CONSTRAINTS];
  int cone_nonlinear[2];                                       /* [0] FrictionCone, [1] ImpulseFrictionCone */
  int enable_acceleration_limit[2];                            /* [0] lower, [1] upper */
  double a_min[12], a_max[12];
  int enable_contact_distance;                                 /* ContactDistance (contact_distance.cpp): 0 off; 1 the reference literally
                                                                  (gradient rows = row 2 of the LOCAL frame Jacobian, robot.hxx:182-188: not
                                                                  the derivative of the height, the iteration diverges on a trot); 2 the
                                                                  consistent variant, rows = d z / d q */
} idocp_b200_fb_problem;
typedef struct idocp_b200_fb_solver idocp_b200_fb_solver; /* opaque */

int idocp_b200_fb_create(const idocp_b200_fb_problem* problem, const idocp_b200_contact_sequence* contact_sequence, int batch,
                         int device, idocp_b200_fb_solver** out);
int idocp_b200_fb_destroy(idocp_b200_fb_solver* h);
/* setSolution(name, value): name in q v a f u; value[dim] broadcast (per_instance = 0) or value[batch][dim]; "f" takes
 * one 3-vector that is given to every contact */
int idocp_b200_fb_set_solution(idocp_b200_fb_solver* h, const char* name, const double* value, int per_instance);
/* cost reference of one slot: kind 0 grid stage (index = time stage, N = terminal), 1 impulse, 2 aux, 3 lift */
int idocp_b200_fb_set_cost_reference(idocp_b200_fb_solver* h, int kind, int index, const double* q_ref, const double* v_ref);
/* Per-instance cost references: the counterpart of one reference OCPSolver per instance, each with its own q_ref(t) / v_ref.
 * A handle starts in shared mode (the references of idocp_b200_fb_set_cost_reference for every instance).
 *   set_instance_cost_reference: q_ref[batch][19], v_ref[batch][18] of the slot (kind, index), same kind / index rules as
 *     idocp_b200_fb_set_cost_reference.  The first call after creation or a clear switches to per-instance references and
 *     starts every slot of every instance from the shared references, so the slots never set keep the shared values.
 *     idocp_b200_fb_set_cost_reference keeps writing the shared references, which are not read until the clear.
 *   clear_instance_cost_references: back to the shared references.
 * The host keeps the table and copies the slots that changed at the next initConstraints / updateSolution /
 * computeKKTResidual, so a reference that does not change between calls is copied once.  Neither call clears the
 * line-search filter, as on a change of the shared references.  Instance b gives the bits of a shared-mode handle whose
 * references are instance b's. */
int idocp_b200_fb_set_instance_cost_reference(idocp_b200_fb_solver* h, int kind, int index, const double* q_ref, const double* v_ref);
int idocp_b200_fb_clear_instance_cost_references(idocp_b200_fb_solver* h);
/* the chain of stages at time t in the order of the Riccati recursion; arrays of capacity cap (may be NULL;
 * active is [cap][4], the contact / impulse status of the stage); returns the number of stages.
 * dimi > 0: the switching constraint of the coming impulse is imposed on that stage */
int idocp_b200_fb_discretize(idocp_b200_fb_solver* h, double t, int cap, int* kind, int* index, double* stage_t, double* dt,
                             int* dimf, int* dimi, int* active);
int idocp_b200_fb_init_constraints(idocp_b200_fb_solver* h, double t);
/* OCPDiscretizer::discretizeOCP asserts isWellDefined() (ocp_discretizer.hxx:62-72,231-244).  strict = 1 (default): a
 * schedule that cannot be discretised at t (an event before t, two events in one grid interval, impulses after
 * consecutive stages) makes initConstraints / updateSolution / computeKKTResidual / discretize return
 * IDOCP_B200_INVALID_ARGUMENT before anything is launched.  strict = 0: run on like a Release build of the reference. */
int idocp_b200_fb_set_strict_discretization(idocp_b200_fb_solver* h, int strict);
/* q[batch][19], v[batch][18] host buffers; NULL keeps the initial states already resident on the device */
int idocp_b200_fb_update_solution(idocp_b200_fb_solver* h, double t, const double* q, const double* v, int line_search);
int idocp_b200_fb_compute_kkt_residual(idocp_b200_fb_solver* h, double t, const double* q, const double* v);
int idocp_b200_fb_kkt_error(idocp_b200_fb_solver* h, double* out /* [batch] */);
int idocp_b200_fb_clear_line_search_filter(idocp_b200_fb_solver* h);   /* clearLineSearchFilter() ocp_solver.cpp:197-199 */
int idocp_b200_fb_get_step_sizes(idocp_b200_fb_solver* h, double* out /* [batch][2]: primal, dual */);
/* one field of one stage of the current chain: out[batch][dim], returns dim (see fb_capi.inc for the field names) */
int idocp_b200_fb_get(idocp_b200_fb_solver* h, int stage, const char* name, double* out);
int idocp_b200_fb_sync(idocp_b200_fb_solver* h);
int idocp_b200_fb_launch_count(idocp_b200_fb_solver* h, long long* out);
int idocp_b200_fb_stream(idocp_b200_fb_solver* h, void** out);
int idocp_b200_fb_set_profiling(idocp_b200_fb_solver* h, int enabled);
int idocp_b200_fb_get_profile(idocp_b200_fb_solver* h, int cap, const char** names, double* ms, long long* calls);
int idocp_b200_fb_record_bytes(void);
/* host-side model facts of ANYmal (the reference's Robot is a host object) */
int idocp_b200_fb_problem_default(idocp_b200_fb_problem* problem);   /* URDF joint limits, barrier 1e-4, rate 0.995 */
double idocp_b200_fb_total_weight(void);                               /* Robot::totalWeight (robot.hxx:746-748) */
/* Robot::updateFrameKinematics(q) + getContactPoints (robot.hxx:233-238,737-743): out[4][3] */
int idocp_b200_fb_contact_frame_positions(const double* q, double* out);

/* The hybrid OCPSolver over several GPUs of one node (twin of idocp_b200_create_sharded): one single-device solver per entry
 * of `devices`, the batch split contiguously, the contact sequence shared; every entry point has the signature of its
 * idocp_b200_fb_* counterpart with the caller's arrays covering the WHOLE batch.  Bit-identical to one solver over the whole
 * batch (tests/test_sharded_solver.py). */
typedef struct idocp_b200_fb_sharded idocp_b200_fb_sharded; /* opaque */
int idocp_b200_fb_create_sharded(const idocp_b200_fb_problem* problem, const idocp_b200_contact_sequence* contact_sequence, int batch,
                                 const int* devices, int n_devices, idocp_b200_fb_sharded** out);
int idocp_b200_fb_sharded_destroy(idocp_b200_fb_sharded* s);
int idocp_b200_fb_sharded_num_shards(const idocp_b200_fb_sharded* s, int* n, int* first);
/* the single-device solver behind shard `index` (borrowed), as idocp_b200_sharded_shard */
int idocp_b200_fb_sharded_shard(idocp_b200_fb_sharded* s, int index, idocp_b200_fb_solver** out);
int idocp_b200_fb_sharded_set_solution(idocp_b200_fb_sharded* s, const char* name, const double* value, int per_instance);
int idocp_b200_fb_sharded_set_cost_reference(idocp_b200_fb_sharded* s, int kind, int index, const double* q_ref, const double* v_ref);
int idocp_b200_fb_sharded_set_instance_cost_reference(idocp_b200_fb_sharded* s, int kind, int index, const double* q_ref /* [batch][19] */,
                                                      const double* v_ref /* [batch][18] */);
int idocp_b200_fb_sharded_clear_instance_cost_references(idocp_b200_fb_sharded* s);
int idocp_b200_fb_sharded_discretize(idocp_b200_fb_sharded* s, double t, int cap, int* kind, int* index, double* stage_t, double* dt,
                                     int* dimf, int* dimi, int* active);
int idocp_b200_fb_sharded_init_constraints(idocp_b200_fb_sharded* s, double t);
int idocp_b200_fb_sharded_set_strict_discretization(idocp_b200_fb_sharded* s, int strict);
int idocp_b200_fb_sharded_update_solution(idocp_b200_fb_sharded* s, double t, const double* q, const double* v, int line_search);
int idocp_b200_fb_sharded_compute_kkt_residual(idocp_b200_fb_sharded* s, double t, const double* q, const double* v);
int idocp_b200_fb_sharded_kkt_error(idocp_b200_fb_sharded* s, double* out /* [batch] */);
int idocp_b200_fb_sharded_clear_line_search_filter(idocp_b200_fb_sharded* s);
int idocp_b200_fb_sharded_get_step_sizes(idocp_b200_fb_sharded* s, double* out /* [batch][2] */);
int idocp_b200_fb_sharded_get(idocp_b200_fb_sharded* s, int stage, const char* name, double* out);
int idocp_b200_fb_sharded_sync(idocp_b200_fb_sharded* s);
int idocp_b200_fb_sharded_launch_count(idocp_b200_fb_sharded* s, long long* out);

const char* idocp_b200_last_error(void);
const char* idocp_b200_version(void);

#ifdef __cplusplus
}
#endif
#endif /* IDOCP_B200_H_ */
