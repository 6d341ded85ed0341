"""Per-instance cost references (idocp_b200_set_instance_reference / _task_reference / clear_instance_references): instance b
of a batch with references r_b gives the bits of the oracle -- and of a shared-mode handle -- whose problem holds r_b, for
both solver kinds, task-space cost off / 6D / 3D, with the line search, the acceleration limits, pipelined and literal
UnOCPSolver, and sharded.

CPU: the SIMT-emulator build (batch 5, not a multiple of 4).  GPU (-m gpu): batch 64, the headline problem at 16384 instances,
and the C++ example examples/iiwa14_reach_targets.cpp."""
import os
import re
import subprocess

import numpy as np
import pytest

import idocp_b200 as I
from conftest import ROOT, make_states
from helpers import DIR_FIELDS, SOL_FIELDS, check_iteration, check_solution, copy_problem
from idocp_b200.capi import SOLVER_UNOCP, SOLVER_UNPARNMPC
from test_emu_parity import with_acceleration_limits

CFG_FIELDS = ("q_ref", "v_ref", "u_ref")


def scenario(lib, task, acc=False, batch=5):
    """problem, initial states and the shared task reference of one case (task None, "6d" or "3d")"""
    rng = np.random.default_rng(31)
    if task is None:
        prob = I.benchmark_problem(lib, N=6, T=0.3)
        q0, v0 = make_states(batch, 17)
        ref = None
    else:
        prob = (I.task_space_problem if task == "6d" else I.task_space_3d_problem)(lib, N=4, T=0.2)
        q0 = np.array([0, np.pi / 2, 0, np.pi / 2, 0, np.pi / 2, 0]) + rng.uniform(-0.3, 0.3, (batch, 7))
        v0 = rng.uniform(-0.2, 0.2, (batch, 7))
        ref = I.task_space_circle_ref
    if acc:
        with_acceleration_limits(prob, 25.0 if task is None else 8.0)
    return prob, q0, v0, ref


def random_references(prob, batch, seed):
    """distinct per-instance q_ref / v_ref / u_ref around the problem's values"""
    rng = np.random.default_rng(seed)
    base = {f: np.array(list(getattr(prob, f))) for f in CFG_FIELDS}
    scale = {"q_ref": 1.0, "v_ref": 0.5, "u_ref": 5.0}
    return {f: base[f] + rng.uniform(-scale[f], scale[f], (batch, 7)) for f in CFG_FIELDS}


def random_task_tables(O, prob, kind, batch, seed, t=0.0):
    """the shared circle table with a per-instance offset of the position target"""
    base = O.task_ref_table(I.task_space_circle_ref, t, prob.T, prob.N, kind)
    rng = np.random.default_rng(seed)
    tables = np.repeat(base[None], batch, axis=0)
    tables[:, :, 9:12] += rng.uniform(-0.08, 0.08, (batch, 1, 3))
    return np.ascontiguousarray(tables)


def make_instance_pair(O, lib, prob, q0, v0, kind, refs, tables, shared_ref=None):
    """the batched solver in per-instance mode and one oracle per instance built from a copy of the problem that holds the
    instance's references (and task table)"""
    batch = q0.shape[0]
    solver = (I.UnOCPSolver if kind == "unocp" else I.UnParNMPCSolver)(prob, batch, lib=lib)
    solver.setSolution("q", q0)
    solver.setSolution("v", v0)
    if shared_ref is not None:
        solver.setTaskReference(shared_ref, 0.0)
    for name, value in refs.items():
        solver.setCostReference(name, value)
    if tables is not None:
        solver.setTaskReference(tables)
    oracles = []
    for b in range(batch):
        oprob = copy_problem(prob, O.default_problem())
        for name, value in refs.items():
            for j in range(7):
                getattr(oprob, name)[j] = value[b][j]
        o = (O.UnOCPSolver if kind == "unocp" else O.UnParNMPCSolver)(oprob)
        o.set_solution("q", q0[b])
        o.set_solution("v", v0[b])
        if tables is not None:
            o.set_task_ref(np.ascontiguousarray(tables[b]))
        elif shared_ref is not None:
            o.set_task_ref(O.task_ref_table(shared_ref, 0.0, prob.T, prob.N, kind))
        oracles.append(o)
    if kind != "unocp":
        solver.initBackwardCorrection(0.0)
        for o in oracles:
            o.init_backward_correction(0.0)
    return solver, oracles


def parity_case(lib, O, kind, task, line_search=False, acc=False, batch=5, iters=4):
    prob, q0, v0, ref = scenario(lib, task, acc, batch)
    refs = random_references(prob, batch, 1000 + batch)
    tables = random_task_tables(O, prob, kind, batch, 2000 + batch) if task else None
    solver, oracles = make_instance_pair(O, lib, prob, q0, v0, kind, refs, tables, shared_ref=ref)
    for it in range(iters):
        check_iteration(solver, oracles, q0, v0, line_search=line_search)
    check_solution(solver, oracles)
    if kind == "unocp":
        names = ("slack", "dual") + (("acc_slack", "acc_dual") if acc else ())
        for name in names:
            ref = np.array([o.get_constraint_data(name) for o in oracles])
            assert np.array_equal(solver.getConstraintData(name), ref, equal_nan=True), name
    return solver


PARITY_CASES = [
    ("unocp", None, False, False), ("unocp", "6d", False, False), ("unocp", "3d", False, False),
    ("unparnmpc", None, False, False), ("unparnmpc", "6d", False, False), ("unparnmpc", "3d", False, False),
    ("unocp", None, True, False), ("unocp", "6d", True, False), ("unocp", None, False, True),
]


@pytest.mark.parametrize("kind,task,line_search,acc", PARITY_CASES)
def test_instance_references_match_per_instance_oracles(emu_lib, oracle, kind, task, line_search, acc):
    parity_case(emu_lib, oracle, kind, task, line_search, acc)


def same_state(a, b, kind):
    for name in SOL_FIELDS:
        assert np.array_equal(a.getSolution(name), b.getSolution(name), equal_nan=True), name
    for name in DIR_FIELDS:
        assert np.array_equal(a.getDirection(name), b.getDirection(name), equal_nan=True), name
    assert np.array_equal(a.getStepSizes(), b.getStepSizes(), equal_nan=True)
    if kind == "unocp":
        for name in ("slack", "dual"):
            assert np.array_equal(a.getConstraintData(name), b.getConstraintData(name), equal_nan=True), name


def equal_references_case(lib, O, kind, task, batch=5, iters=3):
    """per-instance references set to the problem's own values (only q_ref: the other fields start as the problem's) and,
    with a task cost, every instance's table equal to the shared one: the bits of the shared-mode handle"""
    prob, q0, v0, ref = scenario(lib, task, batch=batch)
    cls = I.UnOCPSolver if kind == "unocp" else I.UnParNMPCSolver
    shared, inst = cls(prob, batch, lib=lib), cls(prob, batch, lib=lib)
    for s in (shared, inst):
        s.setSolution("q", q0)
        s.setSolution("v", v0)
        if ref is not None:
            s.setTaskReference(ref, 0.0)
    inst.setCostReference("q_ref", np.tile(np.array(list(prob.q_ref)), (batch, 1)))
    if ref is not None:
        inst.setTaskReference(np.repeat(O.task_ref_table(ref, 0.0, prob.T, prob.N, kind)[None], batch, axis=0))
    for s in (shared, inst):
        if kind != "unocp":
            s.initBackwardCorrection(0.0)
    for it in range(iters):
        for s in (shared, inst):
            s.updateSolution(0.0, q0, v0, it == 1)
            s.computeKKTResidual(0.0, q0, v0)
        assert np.array_equal(shared.KKTError(), inst.KKTError(), equal_nan=True), it
        same_state(shared, inst, kind)


@pytest.mark.parametrize("kind", ["unocp", "unparnmpc"])
@pytest.mark.parametrize("task", [None, "6d"])
def test_equal_references_equal_shared_mode(emu_lib, oracle, kind, task):
    equal_references_case(emu_lib, oracle, kind, task)


def invalidation_case(lib, O, task, batch=5):
    """pipelined UnOCPSolver (kept linearisation + KKT by-product) vs the literal sequence across reference changes and a
    clear between two updateSolution calls: a set or clear that left the kept linearisation in place would step the
    pipelined handle from the old references"""
    prob, q0, v0, ref = scenario(lib, task, batch=batch)
    a, b = I.UnOCPSolver(prob, batch, lib=lib), I.UnOCPSolver(prob, batch, lib=lib)
    b.setPipelining(False)
    for s in (a, b):
        s.setSolution("q", q0)
        s.setSolution("v", v0)
        if ref is not None:
            s.setTaskReference(ref, 0.0)

    def iterate(tag):
        for it in range(3):
            for s in (a, b):
                s.updateSolution(0.0, q0, v0)
                s.computeKKTResidual(0.0, q0, v0)
            assert np.array_equal(a.KKTError(), b.KKTError(), equal_nan=True), (tag, it)
            same_state(a, b, "unocp")
    iterate("shared")
    for k, refs in enumerate((random_references(prob, batch, 7), random_references(prob, batch, 8))):
        for s in (a, b):
            for name, value in refs.items():
                s.setCostReference(name, value)
            if ref is not None:
                s.setTaskReference(random_task_tables(O, prob, "unocp", batch, 50 + k))
        iterate(k)
    for s in (a, b):
        s.clearInstanceReferences()
    iterate("cleared")


@pytest.mark.parametrize("task", [None, "6d"])
def test_reference_changes_invalidate_the_kept_linearisation(emu_lib, oracle, task):
    invalidation_case(emu_lib, oracle, task)


def clear_case(lib, O, kind, batch=5):
    """set then clear before any iteration: the bits of a handle that never left shared mode"""
    prob, q0, v0, ref = scenario(lib, "6d", batch=batch)
    cls = I.UnOCPSolver if kind == "unocp" else I.UnParNMPCSolver
    shared, cleared = cls(prob, batch, lib=lib), cls(prob, batch, lib=lib)
    for s in (shared, cleared):
        s.setSolution("q", q0)
        s.setSolution("v", v0)
        s.setTaskReference(ref, 0.0)
    cleared.setCostReference("v_ref", random_references(prob, batch, 3)["v_ref"])
    cleared.setTaskReference(random_task_tables(O, prob, kind, batch, 4))
    cleared.clearInstanceReferences()
    for s in (shared, cleared):
        if kind != "unocp":
            s.initBackwardCorrection(0.0)
    for it in range(2):
        for s in (shared, cleared):
            s.updateSolution(0.0, q0, v0)
            s.computeKKTResidual(0.0, q0, v0)
        assert np.array_equal(shared.KKTError(), cleared.KKTError()), it
        same_state(shared, cleared, kind)


@pytest.mark.parametrize("kind", ["unocp", "unparnmpc"])
def test_clear_returns_to_shared_references(emu_lib, oracle, kind):
    clear_case(emu_lib, oracle, kind)


def sharded_case(lib, O, kind, devices, batch=7):
    prob, q0, v0, ref = scenario(lib, "6d", batch=batch)
    refs = random_references(prob, batch, 9)
    tables = random_task_tables(O, prob, "unocp" if kind == SOLVER_UNOCP else "unparnmpc", batch, 10)
    one = (I.UnOCPSolver if kind == SOLVER_UNOCP else I.UnParNMPCSolver)(prob, batch, lib=lib)
    many = I.ShardedSolver(prob, batch, devices, kind=kind, lib=lib)
    for s in (one, many):
        s.setSolution("q", q0)
        s.setSolution("v", v0)
        s.setTaskReference(ref, 0.0)
        for name, value in refs.items():
            s.setCostReference(name, value)
        s.setTaskReference(tables)
        if kind == SOLVER_UNPARNMPC:
            s.initBackwardCorrection(0.0)
    for it in range(3):
        for s in (one, many):
            s.updateSolution(0.0, q0, v0, it == 1)
            s.computeKKTResidual(0.0, q0, v0)
        assert np.array_equal(one.KKTError(), many.KKTError(), equal_nan=True), it
    for name in ("q", "v", "a", "u", "lmd", "gmm"):
        assert np.array_equal(one.getSolution(name), many.getSolution(name), equal_nan=True), name
    for s in (one, many):
        s.clearInstanceReferences()
        s.updateSolution(0.0, q0, v0)
    assert np.array_equal(one.getSolution("q"), many.getSolution("q"), equal_nan=True)


@pytest.mark.parametrize("kind", [SOLVER_UNOCP, SOLVER_UNPARNMPC])
def test_sharded_instance_references_equal_single_handle(emu_lib, oracle, kind):
    sharded_case(emu_lib, oracle, kind, [0, 0])


def test_instance_reference_errors(emu_lib):
    prob = I.benchmark_problem(emu_lib, N=3, T=0.15)
    s = I.UnOCPSolver(prob, 2, lib=emu_lib)
    L = emu_lib.L
    with pytest.raises(I.Idocp_b200Error, match="null pointer"):
        emu_lib.check(L.idocp_b200_set_instance_reference(s._h, b"q_ref", None))
    with pytest.raises(I.Idocp_b200Error, match="null pointer"):
        emu_lib.check(L.idocp_b200_set_instance_reference(s._h, None, np.zeros((2, 7)).ctypes.data_as(I.capi._dp)))
    with pytest.raises(I.Idocp_b200Error, match="null pointer"):
        emu_lib.check(L.idocp_b200_set_instance_task_reference(s._h, None))
    with pytest.raises(I.Idocp_b200Error, match="null handle"):
        emu_lib.check(L.idocp_b200_clear_instance_references(None))
    with pytest.raises(I.Idocp_b200Error, match="name must be q_ref, v_ref, or u_ref"):
        s.setCostReference("a_ref", np.zeros((2, 7)))
    with pytest.raises(I.Idocp_b200Error, match="task-space cost"):
        s.setTaskReference(np.zeros((2, prob.N + 1, 12)))
    with pytest.raises(ValueError):
        s.setCostReference("q_ref", np.zeros(7))
    with pytest.raises(ValueError):
        s.setTaskReference(np.zeros((3, prob.N + 1, 12)))
    sh = I.ShardedSolver(prob, 3, [0, 0], lib=emu_lib)
    with pytest.raises(I.Idocp_b200Error, match="name must be q_ref, v_ref, or u_ref"):
        sh.setCostReference("x", np.zeros((3, 7)))
    with pytest.raises(I.Idocp_b200Error, match="task-space cost"):
        sh.setTaskReference(np.zeros((3, prob.N + 1, 12)))


# ---- GPU ---------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("kind,task,line_search,acc", PARITY_CASES)
def test_gpu_instance_references_match_per_instance_oracles(gpu_lib, oracle, kind, task, line_search, acc):
    parity_case(gpu_lib, oracle, kind, task, line_search, acc, batch=64, iters=3)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["unocp", "unparnmpc"])
@pytest.mark.parametrize("task", [None, "6d"])
def test_gpu_equal_references_equal_shared_mode(gpu_lib, oracle, kind, task):
    equal_references_case(gpu_lib, oracle, kind, task, batch=64)


@pytest.mark.gpu
@pytest.mark.parametrize("task", [None, "6d"])
def test_gpu_reference_changes_invalidate_the_kept_linearisation(gpu_lib, oracle, task):
    invalidation_case(gpu_lib, oracle, task, batch=64)


@pytest.mark.gpu
def test_gpu_headline_problem_with_per_instance_q_ref(gpu_lib, oracle):
    """UnOCPSolver, ConfigurationSpaceCost, B = 16384, N = 20: q_ref drawn inside the joint limits from a few distinct targets.
    Every instance equals the shared-mode handle of its target; a fixed sample equals its oracle bit for bit."""
    import bench
    B, iters, ntargets = 16384, 3, 4
    prob = I.benchmark_problem(gpu_lib)
    qmin, qmax = np.array(list(prob.q_min)), np.array(list(prob.q_max))
    q0, v0 = bench.initial_states(0, B, list(qmin), list(qmax))
    rng = np.random.default_rng(12)
    targets = rng.uniform(0.8 * qmin, 0.8 * qmax, (ntargets, 7))
    which = np.arange(B) % ntargets
    q_ref = np.ascontiguousarray(targets[which])
    inst = I.UnOCPSolver(prob, B, lib=gpu_lib)
    inst.setSolution("q", q0)
    inst.setSolution("v", v0)
    inst.setCostReference("q_ref", q_ref)
    for _ in range(iters):
        inst.updateSolution(0.0, q0, v0)
    inst.computeKKTResidual(0.0, q0, v0)
    kkt, q = inst.KKTError(), inst.getSolution("q")
    for k in range(ntargets):
        sel = which == k
        p = I.benchmark_problem(gpu_lib)
        for j in range(7):
            p.q_ref[j] = targets[k][j]
        s = I.UnOCPSolver(p, int(sel.sum()), lib=gpu_lib)
        s.setSolution("q", q0[sel])
        s.setSolution("v", v0[sel])
        for _ in range(iters):
            s.updateSolution(0.0, q0[sel], v0[sel])
        s.computeKKTResidual(0.0, q0[sel], v0[sel])
        assert np.array_equal(s.KKTError(), kkt[sel]), k
        assert np.array_equal(s.getSolution("q"), q[sel]), k
        s.close()
    for b in (0, 1, 2, 3, 4097, 9999, B - 1):
        oprob = copy_problem(prob, oracle.default_problem())
        for j in range(7):
            oprob.q_ref[j] = q_ref[b][j]
        o = oracle.UnOCPSolver(oprob)
        o.set_solution("q", q0[b])
        o.set_solution("v", v0[b])
        for _ in range(iters):
            o.update_solution(0.0, q0[b], v0[b], False)
        o.compute_kkt_residual(0.0, q0[b], v0[b])
        assert o.kkt_error() == kkt[b], b
        assert np.array_equal(o.get_solution("q"), q[b]), b


EXE = os.path.join(ROOT, "build", "iiwa14_reach_targets")


def _build_example():
    import __graft_entry__ as g
    g.build_cuda()
    os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
    lib = os.path.join(ROOT, "idocp_b200")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "iiwa14_reach_targets.cpp"), "-L" + lib, "-lidocp_b200",
                           "-Wl,-rpath," + lib, "-o", EXE])


def test_reach_targets_example_compiles_and_fails_loudly_without_gpu():
    import torch
    _build_example()
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    res = subprocess.run([EXE, "4"], capture_output=True, text=True)
    assert res.returncode != 0
    assert "no CUDA device" in res.stderr


@pytest.mark.gpu
def test_reach_targets_example_equals_the_oracle(oracle):
    """examples/iiwa14_reach_targets.cpp (TaskSpace3DCost, one constant end-effector target per instance through the C++
    host classes): the printed KKT errors equal those of per-instance oracles digit for digit, and every final distance to
    the target is what the oracle's final configuration gives."""
    _build_example()
    batch, iters = 6, 10
    out = subprocess.run([EXE, str(batch), str(iters)], capture_output=True, text=True, check=True).stdout
    rows = re.findall(r"instance (\d+): target \[(\S+) (\S+) (\S+)\] KKT error = (\S+) distance = (\S+)", out)
    assert len(rows) == batch, out
    prob = oracle.task_space_3d_problem()
    q0 = np.array([0, np.pi / 2, 0, np.pi / 2, 0, np.pi / 2, 0])
    for b, tx, ty, tz, kkt, dist in rows:
        target = np.array([1.0, 0, 0, 0, 1.0, 0, 0, 0, 1.0, float(tx), float(ty), float(tz)])
        o = oracle.UnOCPSolver(prob)
        o.set_solution("q", q0)
        o.set_solution("v", np.zeros(7))
        o.set_task_ref(oracle.task_ref_table(lambda t: target, 0.0, prob.T, prob.N, "unocp"))
        for _ in range(iters):
            o.update_solution(0.0, q0, np.zeros(7), False)
        o.compute_kkt_residual(0.0, q0, np.zeros(7))
        assert float(kkt) == o.kkt_error(), b
        _, p, _ = oracle.frame_kinematics(o.get_solution("q")[-1])
        # the example's forward kinematics use the host's libm: agreement to rounding, not bit for bit
        assert abs(float(dist) - float(np.linalg.norm(p - target[9:]))) <= 1e-9, b
