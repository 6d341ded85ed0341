"""The fixed-base getters read one slot-major layout: a field's whole horizon (getSolution), one stage of it
(getStageSolution) and the constraint rows (getConstraintData) must agree with each other, for both solver kinds, with and
without the acceleration limits, on one device and sharded.  Each getter accepts only its own kind of name.

CPU: the SIMT-emulator build."""
import numpy as np
import pytest

import idocp_b200 as I
from conftest import make_states
from idocp_b200.capi import SOLVER_UNOCP, SOLVER_UNPARNMPC

SOLUTION_FIELDS = ("lmd", "gmm", "q", "v", "a", "u", "beta")
FULL_HORIZON = ("lmd", "gmm", "q", "v")   # N + 1 stages on UnOCPSolver
BATCH, N = 5, 3


def problem(lib, acc):
    prob = I.benchmark_problem(lib, N=N, T=0.15)
    if acc:
        prob.enable_acceleration_limit[0] = prob.enable_acceleration_limit[1] = 1
        for j in range(7):
            prob.a_min[j], prob.a_max[j] = -25.0, 25.0
    return prob


@pytest.fixture(params=[(kind, acc, devices) for kind in (SOLVER_UNOCP, SOLVER_UNPARNMPC) for acc in (False, True)
                        for devices in (None, [0, 0])],
                ids=lambda p: "%s-%s-%s" % ("unocp" if p[0] == SOLVER_UNOCP else "unparnmpc", "acc" if p[1] else "noacc",
                                            "sharded" if p[2] else "single"))
def solved(request, emu_lib):
    """A solver after two iterations: (solver, kind, acceleration limits on, sharded)."""
    kind, acc, devices = request.param
    prob = problem(emu_lib, acc)
    if devices:
        s = I.ShardedSolver(prob, BATCH, devices, kind=kind, lib=emu_lib)
    else:
        s = (I.UnOCPSolver if kind == SOLVER_UNOCP else I.UnParNMPCSolver)(prob, BATCH, lib=emu_lib)
    q0, v0 = make_states(BATCH, 11)
    s.setSolution("q", q0)
    s.setSolution("v", v0)
    if kind == SOLVER_UNPARNMPC:
        s.initBackwardCorrection(0.0)
    for _ in range(2):
        s.updateSolution(0.0, q0, v0)
    yield s, kind, acc, devices is not None
    s.close()


def test_stage_solution_equals_full_horizon(solved):
    s, kind, _, _ = solved
    for name in SOLUTION_FIELDS:
        full = s.getSolution(name)
        nst = N + 1 if kind == SOLVER_UNOCP and name in FULL_HORIZON else N
        assert full.shape == (BATCH, nst, 7), name
        for i in range(nst):
            assert np.array_equal(s.getStageSolution(name, i), full[:, i]), (name, i)
        for bad in (-1, nst):
            with pytest.raises(I.Idocp_b200Error, match="get_stage_solution: stage out of range"):
                s.getStageSolution(name, bad)


def test_constraint_data_shapes(solved):
    s, _, acc, sharded = solved
    if sharded:
        return   # getConstraintData has no sharded twin
    for name in ("slack", "dual"):
        assert s.getConstraintData(name).shape == (BATCH, N, 6, 7)
    for name in ("acc_slack", "acc_dual"):
        if acc:
            x = s.getConstraintData(name)
            assert x.shape == (BATCH, N, 2, 7)
            assert np.all(x > 0), name
        else:
            with pytest.raises(I.Idocp_b200Error, match="the acceleration limits are not enabled"):
                s.getConstraintData(name)


def test_unknown_names_raise(solved):
    s, _, _, sharded = solved
    for name in ("nope", "dq", "slack", "acc_slack"):
        with pytest.raises(I.Idocp_b200Error, match="get_solution: unknown field"):
            s.getSolution(name)
        with pytest.raises(I.Idocp_b200Error, match="get_stage_solution: unknown field"):
            s.getStageSolution(name, 0)
    for name in ("nope", "beta", "lmd", "gmm", "dq", "slack"):
        with pytest.raises(I.Idocp_b200Error, match="name must be q, v, a, or u"):
            s.setSolution(name, np.zeros(7))
    if sharded:
        return   # the remaining getters have no sharded twin
    for name in ("nope", "q", "slack"):
        with pytest.raises(I.Idocp_b200Error, match="get_direction: unknown field"):
            s.getDirection(name)
    for name in ("nope", "q", "dq", "acc"):
        with pytest.raises(I.Idocp_b200Error, match="name must be slack, dual, acc_slack or acc_dual"):
            s.getConstraintData(name)
