"""Host-side mirror of idocp::OCPSolver for a batch of instances (floating-base ANYmal), marshalling only.

Reference interface: include/idocp/ocp/ocp_solver.hpp (setSolution, initConstraints, updateSolution,
computeKKTResidual, KKTError, getSolution, setContactStatusUniformly, pushBackContactStatus, popBack/popFront...).
Everything numerical happens in libidocp_b200.so (idocp_b200_fb_* of include/idocp_b200.h)."""
import ctypes as C

import numpy as np

from . import capi
from .hybrid import ContactSequence

KIND_GRID, KIND_IMPULSE, KIND_AUX, KIND_LIFT, KIND_TERMINAL = range(5)
NQ, NV, NU = 19, 18, 12

_FIELD_DIMS = dict(ls_cost=1, ls_viol=1, q=19, f=12, mu=12, nu_passive=6, xi=12, u=12, du=12, daf=30, dbetamu=30, dnu_passive=6, dxi=12, lu=12,
                   lu_passive=6, P=12, Qxx=36 * 36, Qxu=36 * 18, Quu=18 * 18, Fvq=324, Fvv=324, Fvu=216, Fqq6=36, Fqv6=36,
                   Fqq_prev_inv=36, MJtJinv=900, MJ_dIDC=30 * 36, MJ_IDC=30, Qafqv=30 * 36, Qafu=30 * 18, laf=30, K=12 * 36, k=12,
                   Pqq=324, Pqv=324, Pvv=324, Phix=12 * 36, Phiu=144, cM=12 * 36, cm=12, kkt=1, info=1, max_primal=1, max_dual=1,
                   slack=140, dual=140, residual=140, duality=140, dslack=140, ddual=140)


class OCPSolver:
    """OCPSolver(robot, cost, constraints, T, N, max_num_impulse, nthreads) for `batch` instances.

    `problem` is a capi.FbProblem (cost weights, limits, friction); `q_ref(t)` returns the (q_ref, v_ref) pair of the
    configuration-space cost at time t (the reference's update_q_ref, a host-side function of time)."""

    def __init__(self, problem, batch, q_ref=None, device=0, lib=None, max_num_events=None, devices=None):
        """devices = [d0, d1, ...]: the batch sharded over several GPUs of this node by ONE solver object
        (idocp_b200_fb_create_sharded: contiguous split, shared contact schedule, no collective)."""
        self.lib = lib or capi.default_library()
        self.problem = problem
        self.B = int(batch)
        self.q_ref = q_ref
        self.contact_sequence = ContactSequence(4, max_num_events or (2 * problem.max_num_impulse + 2), lib=self.lib)
        self._h = C.c_void_p()
        self._sharded = devices is not None
        if self._sharded:
            dev = (C.c_int * len(devices))(*[int(d) for d in devices])
            self.lib.check(self.lib.L.idocp_b200_fb_create_sharded(C.byref(problem), self.contact_sequence._h, self.B, dev, len(devices),
                                                                   C.byref(self._h)))
        else:
            self.lib.check(self.lib.L.idocp_b200_fb_create(C.byref(problem), self.contact_sequence._h, self.B, int(device),
                                                           C.byref(self._h)))
        self._chain = []

    def _f(self, name):
        """The C-ABI entry point `name` of this solver: idocp_b200_fb_<name> or its sharded twin (same arguments)."""
        return self.lib.entry("fb_", name, self._sharded)

    def __del__(self):
        if getattr(self, "_h", None):
            self._f("destroy")(self._h)
            self._h = None

    # ---- contact schedule (ocp_solver.cpp:173-194) ----
    def setContactStatusUniformly(self, is_active, contact_points=None):
        self.contact_sequence.setContactStatusUniformly(is_active, contact_points)

    def pushBackContactStatus(self, is_active, switching_time, contact_points=None):
        self.contact_sequence.push_back(is_active, switching_time, contact_points)

    def popBackContactStatus(self):
        self.contact_sequence.pop_back()

    def popFrontContactStatus(self):
        self.contact_sequence.pop_front()

    def setContactPoints(self, contact_phase, contact_points):
        self.contact_sequence.setContactPoints(contact_phase, contact_points)

    # ---- solution ----
    def setSolution(self, name, value):
        v = np.ascontiguousarray(np.asarray(value, dtype=np.float64))
        per = 1 if v.ndim == 2 else 0
        if per and v.shape[0] != self.B:
            raise ValueError("per-instance value must have %d rows" % self.B)
        self.lib.check(self._f("set_solution")(self._h, name.encode(), capi.dptr(v), per))

    def discretize(self, t):
        cap = capi.MAX_GRID + 1 + 3 * capi.MAX_EVENTS
        kind, index = np.zeros(cap, np.int32), np.zeros(cap, np.int32)
        tt, dt = np.zeros(cap), np.zeros(cap)
        dimf, dimi = np.zeros(cap, np.int32), np.zeros(cap, np.int32)
        ip = C.POINTER(C.c_int)
        n = self.lib.check(self._f("discretize")(self._h, float(t), cap, kind.ctypes.data_as(ip),
                                                               index.ctypes.data_as(ip), capi.dptr(tt), capi.dptr(dt),
                                                               dimf.ctypes.data_as(ip), dimi.ctypes.data_as(ip), None))
        self._chain = [dict(kind=int(kind[e]), index=int(index[e]), t=float(tt[e]), dt=float(dt[e]), dimf=int(dimf[e]),
                            dimi=int(dimi[e])) for e in range(n)]
        return self._chain

    def _sample_reference(self, t):
        chain = self.discretize(t)
        if self.q_ref is None:
            return chain
        for el in chain:
            q_ref, v_ref = self.q_ref(el["t"])
            q_ref = np.ascontiguousarray(q_ref, dtype=np.float64)
            v_ref = np.ascontiguousarray(v_ref, dtype=np.float64)
            kind = KIND_GRID if el["kind"] == KIND_TERMINAL else el["kind"]
            self.lib.check(self._f("set_cost_reference")(self._h, kind, el["index"], capi.dptr(q_ref),
                                                                       capi.dptr(v_ref)))
        return chain

    def initConstraints(self, t):
        self._sample_reference(t)
        self.lib.check(self._f("init_constraints")(self._h, float(t)))
        self.discretize(t)

    def _state(self, q, v):
        q = np.ascontiguousarray(np.broadcast_to(np.asarray(q, dtype=np.float64), (self.B, NQ)))
        v = np.ascontiguousarray(np.broadcast_to(np.asarray(v, dtype=np.float64), (self.B, NV)))
        return q, v

    def updateSolution(self, t, q, v, line_search=False):
        self._sample_reference(t)
        q, v = self._state(q, v)
        self.lib.check(self._f("update_solution")(self._h, float(t), capi.dptr(q), capi.dptr(v), int(line_search)))

    def updateSolutionResident(self, t, line_search=False):
        """updateSolution with the initial states and the cost reference already resident on the device."""
        self.lib.check(self._f("update_solution")(self._h, float(t), None, None, int(line_search)))

    def stream(self):
        p = C.c_void_p()
        self.lib.check(self._f("stream")(self._h, C.byref(p)))
        return p.value or 0

    def computeKKTResidual(self, t, q, v):
        self._sample_reference(t)
        q, v = self._state(q, v)
        self.lib.check(self._f("compute_kkt_residual")(self._h, float(t), capi.dptr(q), capi.dptr(v)))

    def setStrictDiscretization(self, strict):
        """strict (default): a schedule that cannot be discretised at t raises; False: run on like a Release build of
        the reference, whose assert(isWellDefined()) is compiled out (ocp_discretizer.hxx:62-72)."""
        self.lib.check(self._f("set_strict_discretization")(self._h, int(bool(strict))))

    def clearLineSearchFilter(self):
        self.lib.check(self._f("clear_line_search_filter")(self._h))

    def KKTError(self):
        out = np.zeros(self.B)
        self.lib.check(self._f("kkt_error")(self._h, capi.dptr(out)))
        return out

    def stepSizes(self):
        out = np.zeros((self.B, 2))
        self.lib.check(self._f("get_step_sizes")(self._h, capi.dptr(out)))
        return out

    def get(self, stage, name):
        """Field `name` of chain stage `stage` for every instance: (B, dim)."""
        dim = _FIELD_DIMS.get(name, NV)
        out = np.zeros((self.B, dim))
        got = self.lib.check(self._f("get")(self._h, int(stage), name.encode(), capi.dptr(out)))
        assert got == dim, (name, got, dim)
        return out

    def getSolution(self, name):
        """std::vector of the grid-stage values (ocp_solver.cpp:244-280): list over time stages of (B, dim)."""
        out = []
        for e, el in enumerate(self._chain):
            if el["kind"] == KIND_GRID or (el["kind"] == KIND_TERMINAL and name in ("q", "v")):
                out.append(self.get(e, name))
        return out

    def getStateFeedbackGain(self, time_stage):
        """(Kq, Kv), each (B, 12, 18): du = Kq dq + Kv dv at grid stage `time_stage` (ocp_solver.cpp:103-113)."""
        for e, el in enumerate(self._chain):
            if el["kind"] == KIND_GRID and el["index"] == time_stage:
                K = self.get(e, "K").reshape(self.B, 12, 36)
                return K[:, :, :18].copy(), K[:, :, 18:].copy()
        raise ValueError("time_stage outside the horizon")

    def chain(self):
        return self._chain

    def sync(self):
        self.lib.check(self._f("sync")(self._h))

    def launchCount(self):
        n = C.c_longlong()
        self.lib.check(self._f("launch_count")(self._h, C.byref(n)))
        return n.value

    def setProfiling(self, enabled):
        self.lib.check(self._f("set_profiling")(self._h, int(enabled)))

    def getProfile(self):
        cap = 32
        names = (C.c_char_p * cap)()
        ms = np.zeros(cap)
        calls = (C.c_longlong * cap)()
        n = self.lib.check(self._f("get_profile")(self._h, cap, names, capi.dptr(ms), calls))
        return {names[i].decode(): dict(ms=float(ms[i]), calls=int(calls[i])) for i in range(n)}
