"""Host-side mirror of idocp's solver interface for a BATCH of instances.

Same method names, argument meaning and call order as the reference classes
(include/idocp/unocp/unocp_solver.hpp:37-170, unparnmpc_solver.hpp:37-171); every vector argument
gains a leading batch dimension.  The C++ twin of these classes is include/idocp_b200/*.hpp.
All arithmetic happens in the CUDA library behind the C-ABI; nothing here computes.
"""
import ctypes as C

import numpy as np

from . import capi
from .capi import DIMV, NUM_CONSTRAINTS, SOLVER_UNOCP, SOLVER_UNPARNMPC, Idocp_b200Error, Problem, dptr

__all__ = ["UnOCPSolver", "UnParNMPCSolver", "DerivativeChecker", "benchmark_problem", "config_space_problem", "task_space_problem",
           "task_space_circle_ref", "Problem"]


def _fill(arr, value):
    value = np.broadcast_to(np.asarray(value, dtype=np.float64), (len(arr),))
    for i in range(len(arr)):
        arr[i] = float(value[i])


def benchmark_problem(lib=None, N=20, T=1.0):
    """examples/iiwa14/unocp_benchmark.cpp:22-46 (BASELINE.json configs[2], the metric config)."""
    lib = lib or capi.default_library()
    p = lib.default_problem()
    p.N, p.T = N, T
    _fill(p.u_max, 200.0)
    _fill(p.q_ref, -5.0)
    _fill(p.v_ref, -9.0)
    _fill(p.q_weight, 10.0)
    _fill(p.qf_weight, 10.0)
    _fill(p.v_weight, 0.1)
    _fill(p.vf_weight, 0.1)
    _fill(p.a_weight, 0.01)
    _fill(p.u_weight, 0.0)
    return p


def config_space_problem(lib=None):
    """examples/iiwa14/config_space_ocp.cpp:26-61 (BASELINE.json configs[0])."""
    lib = lib or capi.default_library()
    p = lib.default_problem()
    p.N, p.T = 60, 3.0
    _fill(p.u_max, 50.0)
    _fill(p.v_max, np.pi / 2)
    _fill(p.q_ref, [0, np.pi / 2, 0, np.pi / 2, 0, np.pi / 2, 0])
    _fill(p.q_weight, 10.0)
    _fill(p.qf_weight, 10.0)
    _fill(p.v_weight, 0.01)
    _fill(p.vf_weight, 0.01)
    _fill(p.a_weight, 0.01)
    return p


def task_space_problem(lib=None, N=120, T=6.0):
    """examples/iiwa14/task_space_ocp.cpp:55-84 (BASELINE.json configs[1] problem): joint limits 50 / pi/2,
    ConfigurationSpaceCost (v, a weights 0.01) + TimeVaryingTaskSpace6DCost with weights 1000."""
    lib = lib or capi.default_library()
    p = lib.default_problem()
    p.N, p.T = N, T
    _fill(p.u_max, 50.0)
    _fill(p.v_max, np.pi / 2)
    _fill(p.v_weight, 0.01)
    _fill(p.vf_weight, 0.01)
    _fill(p.a_weight, 0.01)
    p.task_enabled = 1
    _fill(p.task_q_weight, 1000.0)
    _fill(p.task_qf_weight, 1000.0)
    return p


def task_space_3d_problem(lib=None, N=30, T=1.5):
    """TaskSpace3DCost / TimeVaryingTaskSpace3DCost (src/cost/task_space_3d_cost.cpp) on the task_space_ocp robot set-up:
    position error of the end-effector frame, weights 1000 (task_enabled = 2; task_q_weight[0..2] = q_3d_weight)."""
    p = task_space_problem(lib, N, T)
    p.task_enabled = 2
    for k in range(3, 6):
        p.task_q_weight[k] = 0.0
        p.task_qf_weight[k] = 0.0
    for i in range(7):          # a 3D position cost has rank 3 in q: a small posture weight keeps the stage Hessian definite
        p.q_weight[i] = 0.1     # (UnParNMPC factorises the full 21 x 21 stage Hessian)
        p.qf_weight[i] = 0.1
    return p


def task_space_circle_ref(t):
    """TimeVaryingTaskSpace6DRef::compute_q_6d_ref of examples/iiwa14/task_space_ocp.cpp:21-46
    -> [R_ref row-major (9), p_ref (3)]."""
    return np.array([0.0, 0.0, 1.0, 0.0, 1.0, 0.0, -1.0, 0.0, 0.0,
                     0.546, 0.1 * np.sin(np.pi * t), 0.76 + 0.1 * np.cos(np.pi * t)])


class _BatchSolver:
    kind = None

    def __init__(self, problem, batch, device=0, lib=None, devices=None):
        """devices = [d0, d1, ...]: the batch sharded over several GPUs of this node by ONE solver object
        (idocp_b200_create_sharded: contiguous split, one device + stream per shard, no collective); `first` then holds the
        first instance of every shard.  Entry points without a sharded twin raise on such a solver."""
        self.lib = lib or capi.default_library()
        self.batch = int(batch)
        self.N = int(problem.N)
        self.problem = problem
        self._h = C.c_void_p()
        self._sharded = devices is not None
        if self._sharded:
            devs = (C.c_int * len(devices))(*[int(d) for d in devices])
            self.lib.check(self.lib.L.idocp_b200_create_sharded(C.byref(problem), self.kind, self.batch, devs, len(devices),
                                                                C.byref(self._h)))
            first = (C.c_int * (len(devices) + 1))()
            self.lib.check(self._f("num_shards")(self._h, C.byref(C.c_int()), first))
            self.first = list(first)
        else:
            self.lib.check(self.lib.L.idocp_b200_create(C.byref(problem), self.kind, self.batch, device, C.byref(self._h)))

    def _f(self, name):
        """The C-ABI entry point `name` of this solver: idocp_b200_<name> or its sharded twin."""
        return self.lib.entry("", name, self._sharded)

    def close(self):
        if getattr(self, "_h", None):
            self._f("destroy")(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- reference API -----------------------------------------------------------------------
    def _x(self, a):
        a = np.ascontiguousarray(np.asarray(a, dtype=np.float64))
        if a.shape == (DIMV,):
            a = np.ascontiguousarray(np.broadcast_to(a, (self.batch, DIMV)))
        if a.shape != (self.batch, DIMV):
            raise ValueError("expected an array of shape (%d, %d) or (%d,)" % (self.batch, DIMV, DIMV))
        return a

    def setSolution(self, name, value):
        """UnOCPSolver::setSolution: value (dimv,) is written to all stages of all instances;
        value (batch, dimv) gives every instance its own vector."""
        value = np.ascontiguousarray(np.asarray(value, dtype=np.float64))
        if value.shape == (DIMV,):
            bc = 1
        elif value.shape == (self.batch, DIMV):
            bc = 0
        else:
            raise ValueError("setSolution: bad shape %s" % (value.shape,))
        self.lib.check(self._f("set_solution")(self._h, name.encode(), dptr(value), bc))

    def initConstraints(self):
        self.lib.check(self._f("init_constraints")(self._h))

    def stageTimes(self, t):
        """Time at which every stage index is linearised (unocp_solver.cpp:80-93 / unbackward_correction.cpp:73-95)."""
        dt = self.problem.T / self.N
        if self.kind == SOLVER_UNOCP:
            return [t + i * dt for i in range(self.N)] + [t + self.problem.T]
        return [t + (i + 1) * dt for i in range(self.N - 1)] + [t + self.problem.T, t + self.N * dt]

    def setTaskReference(self, ref, t=0.0):
        """TimeVaryingTaskSpace6DCost reference: `ref` is the user's compute_q_6d_ref(t) -> 12 doubles
        (R row-major, p), sampled here on the host at every stage time, or an (N+1, 12) table."""
        table = np.array([ref(x) for x in self.stageTimes(t)]) if callable(ref) else np.asarray(ref, dtype=np.float64)
        table = np.ascontiguousarray(table, dtype=np.float64)
        if table.shape != (self.N + 1, 12):
            raise ValueError("task reference table must have shape (%d, 12)" % (self.N + 1))
        self.lib.check(self._f("set_task_reference")(self._h, dptr(table)))

    def updateSolution(self, t, q, v, line_search=False):
        q, v = self._x(q), self._x(v)
        self.lib.check(self._f("update_solution")(self._h, float(t), dptr(q), dptr(v), int(line_search)))

    def updateSolutionDevice(self, t, q_ptr, v_ptr, line_search=False):
        """q_ptr / v_ptr: device addresses (e.g. torch.Tensor.data_ptr()) of (batch, dimv) float64."""
        self.lib.check(self._f("update_solution_device")(self._h, float(t), C.c_void_p(q_ptr), C.c_void_p(v_ptr),
                                                         int(line_search)))

    def computeKKTResidual(self, t, q, v):
        q, v = self._x(q), self._x(v)
        self.lib.check(self._f("compute_kkt_residual")(self._h, float(t), dptr(q), dptr(v)))

    def computeKKTResidualDevice(self, t, q_ptr, v_ptr):
        self.lib.check(self._f("compute_kkt_residual_device")(self._h, float(t), C.c_void_p(q_ptr), C.c_void_p(v_ptr)))

    def KKTError(self):
        out = np.zeros(self.batch)
        self.lib.check(self._f("kkt_error")(self._h, dptr(out)))
        return out

    def _nstages(self, name, full_names):
        return self.N + 1 if (name in full_names and self.kind == SOLVER_UNOCP) else self.N

    def getSolution(self, name):
        out = np.zeros((self.batch, self._nstages(name, ("q", "v", "lmd", "gmm")), DIMV))
        self.lib.check(self._f("get_solution")(self._h, name.encode(), dptr(out)))
        return out

    def getStageSolution(self, name, stage, out=None):
        """UnOCPSolver::getSolution(int stage), one field: (batch, dimv)."""
        if out is None:
            out = np.zeros((self.batch, DIMV))
        self.lib.check(self._f("get_stage_solution")(self._h, name.encode(), int(stage), dptr(out)))
        return out

    def saveSolution(self, path_to_file, name, instance=0):
        """UnOCPSolver::saveSolution (unocp_solver.cpp:312-352): one stage per line, every coefficient followed by a
        blank, the stream's default formatting (%g); `instance` selects the member of the batch."""
        with open(path_to_file, "w") as f:
            if name in ("q", "v", "a", "u"):
                for row in self.getSolution(name)[instance]:
                    f.write("".join("%g " % x for x in row) + "\n")

    def clearLineSearchFilter(self):
        self.lib.check(self._f("clear_line_search_filter")(self._h))

    def isCurrentSolutionFeasible(self):
        out = np.zeros(self.batch, dtype=np.int32)
        self.lib.check(self._f("is_feasible")(self._h, out.ctypes.data_as(C.POINTER(C.c_int))))
        return out.astype(bool)

    # -- additions for parity tests / measurement ----------------------------------------------
    def getDirection(self, name):
        out = np.zeros((self.batch, self._nstages(name, ("dq", "dv", "dlmd", "dgmm")), DIMV))
        self.lib.check(self._f("get_direction")(self._h, name.encode(), dptr(out)))
        return out

    def getConstraintData(self, name):
        # "slack" / "dual": the six joint-limit components; "acc_slack" / "acc_dual": the two acceleration limits
        out = np.zeros((self.batch, self.N, 2 if name.startswith("acc_") else NUM_CONSTRAINTS, DIMV))
        self.lib.check(self._f("get_constraint_data")(self._h, name.encode(), dptr(out)))
        return out

    def getStepSizes(self):
        p, d = np.zeros(self.batch), np.zeros(self.batch)
        self.lib.check(self._f("get_step_sizes")(self._h, dptr(p), dptr(d)))
        return p, d

    def setPipelining(self, enabled):
        """UnOCPSolver: fuse the update with the linearisation of the new iterate (default on; idocp_b200_set_pipelining)."""
        self.lib.check(self._f("set_pipelining")(self._h, int(bool(enabled))))

    def getUnKKT(self, stage):
        Q = np.zeros((self.batch, 21, 21))
        res = np.zeros((self.batch, 35))
        self.lib.check(self._f("get_unkkt")(self._h, int(stage), dptr(Q), dptr(res)))
        return np.ascontiguousarray(Q.transpose(0, 2, 1)), res   # column-major -> [row, col]

    def getStatus(self):
        out = np.zeros(self.batch, dtype=np.int32)
        self.lib.check(self._f("get_status")(self._h, out.ctypes.data_as(C.POINTER(C.c_int))))
        return out

    def sync(self):
        self.lib.check(self._f("sync")(self._h))

    def launchCount(self):
        n = C.c_longlong(0)
        self.lib.check(self._f("launch_count")(self._h, C.byref(n)))
        return n.value

    def stream(self):
        s = C.c_void_p()
        self.lib.check(self._f("stream")(self._h, C.byref(s)))
        return s.value or 0

    def setProfiling(self, enabled):
        self.lib.check(self._f("set_profiling")(self._h, int(enabled)))

    def getProfile(self):
        cap = 16
        names = (C.c_char_p * cap)()
        ms = np.zeros(cap)
        calls = (C.c_longlong * cap)()
        n = self.lib.check(self._f("get_profile")(self._h, cap, names, dptr(ms), calls))
        return {names[i].decode(): (ms[i], calls[i]) for i in range(n)}


class UnOCPSolver(_BatchSolver):
    """Batched idocp::UnOCPSolver (Riccati recursion)."""
    kind = SOLVER_UNOCP


def _is_approx(a, b, prec):
    """Eigen's a.isApprox(b, prec): |a - b|^2 <= prec^2 min(|a|^2, |b|^2) (Frobenius norms)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.sum((a - b) ** 2)) <= prec * prec * min(float(np.sum(a * a)), float(np.sum(b * b)))


class DerivativeChecker:
    """idocp::DerivativeChecker (include/idocp/utils/derivative_checker.hpp:14-66, src/utils/derivative_checker.cpp:47-312)
    for the cost of a fixed-base Problem, evaluated ON THE DEVICE (idocp_b200_check_cost_derivatives): at `samples` random split
    solutions the analytic gradient of the lineariser's device functions is compared with forward differences of the cost
    value of the line search's device functions (first order), and the analytic Hessian with forward differences of the
    gradient (second order), block by block with Eigen's isApprox like the reference.  The reference takes one cost
    component and draws ONE sample; here the problem carries the cost (configuration-space + optional task-space term) and
    every sample has to pass.  `last_failure` names the block that failed, as the reference's message does."""

    def __init__(self, problem, finite_diff=1.0e-08, test_tol=1.0e-04, samples=8, seed=0, lib=None, task_ref=None, t=0.0):
        self.finite_diff, self.test_tol = float(finite_diff), float(test_tol)
        self.samples = int(samples)
        self._solver = UnOCPSolver(problem, self.samples, lib=lib)
        if task_ref is not None:
            self._solver.setTaskReference(task_ref, t)
        self._rng = np.random.default_rng(seed)
        self.last_failure = None

    def setFiniteDifference(self, finite_diff=1.0e-08):
        self.finite_diff = float(finite_diff)

    def setTestTolerance(self, test_tol=1.0e-04):
        self.test_tol = float(test_tol)

    def evaluate(self, terminal=False, stage=0):
        """The raw numbers of one device pass over fresh random samples (SplitSolution::Random: uniform in [-1, 1])."""
        s = self._solver
        x = [np.ascontiguousarray(self._rng.uniform(-1.0, 1.0, (self.samples, DIMV))) for _ in range(4)]
        out = np.zeros((self.samples, capi.DC_DOUBLES))
        s.lib.check(s.lib.L.idocp_b200_check_cost_derivatives(s._h, int(bool(terminal)), int(stage), self.samples, dptr(x[0]), dptr(x[1]),
                                                             dptr(x[2]), dptr(x[3]), self.finite_diff, dptr(out)))
        n = DIMV
        r = dict(cost=out[:, 0], q=x[0], v=x[1], a=x[2], u=x[3])
        for k, name in enumerate(("lq", "lv", "la", "lu")):
            r[name] = out[:, 1 + k * n:1 + (k + 1) * n]
            r[name + "_ref"] = out[:, 29 + k * n:29 + (k + 1) * n]
        r["Qqq"] = out[:, 57:106].reshape(-1, n, n)
        for k, name in enumerate(("Qvv", "Qaa", "Quu")):
            r[name] = np.stack([np.diag(d) for d in out[:, 106 + k * n:106 + (k + 1) * n]])
        for k, name in enumerate(("Qqq", "Qvv", "Qaa", "Quu")):
            r[name + "_ref"] = out[:, 127 + 49 * k:127 + 49 * (k + 1)].reshape(-1, n, n)
        return r

    def _check(self, names, terminal):
        r = self.evaluate(terminal)
        for b in range(self.samples):
            for name in names:
                if not _is_approx(r[name][b], r[name + "_ref"][b], self.test_tol):
                    self.last_failure = "%s is not correct! sample %d, %s - %s_ref = %s" % (name, b, name, name,
                                                                                             (r[name][b] - r[name + "_ref"][b]).ravel())
                    return False
        self.last_failure = None
        return True

    def checkFirstOrderStageCostDerivatives(self):
        return self._check(("lq", "lv", "la", "lu"), False)

    def checkSecondOrderStageCostDerivatives(self):
        return self._check(("Qqq", "Qvv", "Qaa", "Quu"), False)

    def checkFirstOrderTerminalCostDerivatives(self):
        return self._check(("lq", "lv"), True)

    def checkSecondOrderTerminalCostDerivatives(self):
        return self._check(("Qqq", "Qvv"), True)


class UnParNMPCSolver(_BatchSolver):
    """Batched idocp::UnParNMPCSolver (ParNMPC backward correction)."""
    kind = SOLVER_UNPARNMPC

    def initBackwardCorrection(self, t):
        self.lib.check(self._f("init_backward_correction")(self._h, float(t)))


class ShardedSolver(_BatchSolver):
    """One UnOCPSolver / UnParNMPCSolver (`kind`) over several GPUs of one node: the batch is split into contiguous shards,
    one device + stream per shard, no collective.  Same methods and argument shapes as the single-device classes; arrays
    are (batch, ...) over the WHOLE batch."""

    def __init__(self, problem, batch, devices, kind=SOLVER_UNOCP, lib=None):
        self.kind = kind
        super().__init__(problem, batch, lib=lib, devices=devices)

    initBackwardCorrection = UnParNMPCSolver.initBackwardCorrection
