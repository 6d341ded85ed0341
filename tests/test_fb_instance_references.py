"""Per-instance cost references of the floating-base OCPSolver (idocp_b200_fb_set_instance_cost_reference): instance b of one
handle gives the bits of an oracle OCPSolver whose configuration reference q_ref(t) / v_ref is instance b's.  The per-instance
oracles are TrottingProblem copies with their own base height, knee swing amplitude and forward velocity reference; footholds
and contact schedule are shared.  Emulator (CPU) and GPU; the GPU part also covers BatchedMPC and the C++ example
examples/anymal_trotting_instance_refs.cpp."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

import anymal_problems as ap
import idocp_b200 as I
from conftest import ROOT
from fb_scenarios import anymal_states
from test_emu_fb_parity import DIR, EXP, KKT, RIC, SOL, compare


class InstanceTrotting(ap.TrottingProblem):
    """anymal_trotting.cpp with this instance's base height offset, knee swing amplitude and forward velocity reference."""

    def __init__(self, dz=0.0, knee=1.7, vx=None):
        super().__init__()
        self.dz = dz
        self.swing = dict(front_swing_knee=knee, hip_swing_knee=knee)
        if vx is not None:
            self.v_ref = self.v_ref.copy()
            self.v_ref[0] = vx

    def q_ref(self, t):
        q = super().q_ref(t)
        q[2] += self.dz
        return q


FIXED_VARIANTS = [dict(dz=0.0, knee=1.7, vx=0.3), dict(dz=-0.04, knee=1.2, vx=0.2), dict(dz=0.03, knee=2.0, vx=0.4)]


def random_variants(count, seed):
    rng = np.random.default_rng(seed)
    return [dict(dz=rng.uniform(-0.05, 0.05), knee=rng.uniform(1.2, 2.0), vx=rng.uniform(0.1, 0.4)) for _ in range(count)]


def reference_fn(problems):
    """fn(t) -> (q_ref (B, 19), v_ref (B, 18)) of OCPSolver.setInstanceCostReference."""
    return lambda t: (np.stack([p.q_ref(t) for p in problems]), np.stack([p.v_ref for p in problems]))


def setup(lib, fb, variants, q0=None, v0=None, devices=None):
    """The product solver with per-instance references (shared reference: the unmodified trot) and one oracle per instance."""
    problems = [InstanceTrotting(**v) for v in variants]
    B = len(problems)
    base = ap.TrottingProblem()
    q0 = np.tile(base.q0, (B, 1)) if q0 is None else q0
    v0 = np.tile(base.v0, (B, 1)) if v0 is None else v0
    solver = ap.make_product_solver(base, lib, fb, batch=B, q0=q0, v0=v0, devices=devices)
    solver.setInstanceCostReference(reference_fn(problems))
    return problems, solver, q0, v0


def check_instance(o, solver, fb, b, tag):
    for names in (KKT + EXP, RIC, DIR, SOL):
        assert compare(o, solver, fb, names, b=b) == [], (tag, b)
    for e in range(len(solver.chain())):
        for nm in ("slack", "dual"):
            assert np.array_equal(o.get(e, nm), solver.get(e, nm)[b]), (tag, b, e, nm)


def parity_case(lib, fb, variants, line_search, iters=3, sample=None, q0=None, v0=None):
    """Every field of every stage of the sampled instances (default: all) bit-exact against their oracles over `iters`
    iterations of computeKKTResidual / KKTError / updateSolution; step sizes every iteration."""
    problems, solver, q0, v0 = setup(lib, fb, variants, q0, v0)
    sample = range(len(problems)) if sample is None else sample
    oracles = {b: problems[b].make_oracle(fb, q0=q0[b], v0=v0[b]) for b in sample}
    for it in range(iters):
        solver.computeKKTResidual(0.0, q0, v0)
        kkt = solver.KKTError()
        solver.updateSolution(0.0, q0, v0, line_search)
        steps = solver.stepSizes()
        for b, o in oracles.items():
            o.compute_kkt_residual(0.0, q0[b], v0[b])
            assert kkt[b] == o.kkt_error(), (it, b, kkt[b], o.kkt_error())
            assert o.update_solution(0.0, q0[b], v0[b], line_search) == 0, (it, b)
            assert np.array_equal(steps[b], o.step_sizes()), (it, b, steps[b], o.step_sizes())
            check_instance(o, solver, fb, b, it)
    # the references differ between the instances: so do the iterates
    q = np.asarray(solver.get(len(solver.chain()) - 1, "q"))
    assert len(np.unique(q[list(sample)], axis=0)) == len(list(sample))


def same_iterates(a, b, tag):
    assert np.array_equal(a.KKTError(), b.KKTError()), tag
    assert np.array_equal(a.stepSizes(), b.stepSizes()), tag
    for e in range(len(a.chain())):
        for nm in SOL + DIR + RIC + ["slack", "dual", "lq", "lv"]:
            assert np.array_equal(a.get(e, nm), b.get(e, nm), equal_nan=True), (tag, e, nm)


@pytest.fixture(scope="module")
def fb(oracle):
    import fb_py
    fb_py.lib()
    return fb_py


# ---- emulator ----------------------------------------------------------------------------------------------------------

@pytest.mark.parametrize("line_search", [False, True])
def test_instance_references_match_per_instance_oracles(fb, emu_lib, line_search):
    parity_case(emu_lib, fb, FIXED_VARIANTS, line_search)


def test_equal_references_equal_shared_mode(fb, emu_lib):
    pr = ap.TrottingProblem()
    B = 3
    q0, v0 = anymal_states(pr, B, 20240011)
    shared = ap.make_product_solver(pr, emu_lib, fb, batch=B, q0=q0, v0=v0)
    per = ap.make_product_solver(pr, emu_lib, fb, batch=B, q0=q0, v0=v0)
    per.setInstanceCostReference(reference_fn([pr] * B))
    for it in range(3):
        for s in (shared, per):
            s.computeKKTResidual(0.0, q0, v0)
            s.updateSolution(0.0, q0, v0, it == 1)
        same_iterates(shared, per, it)


def test_receding_horizon_resamples_instance_references(fb, emu_lib):
    # updateSolution at advancing t: the chain's slots change between calls, the references are re-sampled every call and
    # only the slots that changed are copied; an event leaves the horizon through popFrontContactStatus
    problems, solver, q, v = setup(emu_lib, fb, FIXED_VARIANTS)
    oracles = [p.make_oracle(fb) for p in problems]

    def step(t, strict=True):
        for p, o in zip(problems, oracles):
            p.set_references(o, t)
        rcs = [o.update_solution(t, q[b], v[b]) for b, o in enumerate(oracles)]
        solver.updateSolution(t, q, v)
        steps = solver.stepSizes()
        for b, o in enumerate(oracles):
            assert np.array_equal(steps[b], o.step_sizes()), (t, b)
            if rcs[b] == 0 or strict:
                assert compare(o, solver, fb, SOL, b=b) == [], (t, b)
                assert compare(o, solver, fb, DIR, b=b) == [], (t, b)

    for t in (0.0, 0.013, 0.04, 0.31, 0.47):
        step(t)
        q = np.stack([o.get(1, "q") for o in oracles])
        v = np.stack([o.get(1, "v") for o in oracles])
    cs0 = oracles[0].cs
    a, pts = cs0.phase(cs0.counts()[0] - 1)
    pts = pts.copy()
    pts[0, 0] += problems[0].step_length
    pts[3, 0] += problems[0].step_length
    t = 0.52
    for o in oracles:
        o.cs.pop_front()
        assert o.cs.push_back([1, 0, 0, 1], t + problems[0].T - 0.02, pts) == 0
    solver.popFrontContactStatus()
    solver.pushBackContactStatus([1, 0, 0, 1], t + problems[0].T - 0.02, pts)
    for t in (0.52, 0.55):
        step(t, strict=False)


def test_clear_returns_to_shared_references(fb, emu_lib):
    problems, solver, q0, v0 = setup(emu_lib, fb, FIXED_VARIANTS)
    oracles = [p.make_oracle(fb) for p in problems]
    base = ap.TrottingProblem()
    for it in range(4):
        if it == 2:
            solver.clearInstanceCostReferences()
            for o in oracles:
                base.set_references(o, 0.0)
        solver.updateSolution(0.0, q0, v0)
        solver.computeKKTResidual(0.0, q0, v0)
        kkt = solver.KKTError()
        for b, o in enumerate(oracles):
            assert o.update_solution(0.0, q0[b], v0[b]) == 0
            o.compute_kkt_residual(0.0, q0[b], v0[b])
            assert kkt[b] == o.kkt_error(), (it, b)
            assert compare(o, solver, fb, SOL, b=b) == [], (it, b)
    # per-instance mode again, with every instance on the shared reference: the oracles' KKT errors
    solver.setInstanceCostReference(reference_fn([base] * 3))
    solver.computeKKTResidual(0.0, q0, v0)
    assert np.array_equal(solver.KKTError(), np.array([o.kkt_error() for o in oracles]))


def test_unset_slots_keep_shared_references_and_shared_sets_leave_the_table(fb, emu_lib):
    """Two C-ABI rules the host layers never show (they write every slot of the chain on every call): (a) the first
    per-instance set fills every slot it does not write from the shared references; (b) in per-instance mode a shared set
    updates the shared references only, which the clear returns to."""
    pr = ap.TrottingProblem()
    B = 2
    q0, v0 = anymal_states(pr, B, 20240018)
    shared = ap.make_product_solver(pr, emu_lib, fb, batch=B, q0=q0, v0=v0)
    per = ap.make_product_solver(pr, emu_lib, fb, batch=B, q0=q0, v0=v0)
    # (a) one slot (grid stage 3) set per instance to the shared reference at its time; every other slot comes from the fill
    el = [c for c in per.chain() if c["kind"] == 0 and c["index"] == 3][0]
    q = np.ascontiguousarray(np.tile(pr.q_ref(el["t"]), (B, 1)))
    v = np.ascontiguousarray(np.tile(pr.v_ref, (B, 1)))
    emu_lib.check(emu_lib.L.idocp_b200_fb_set_instance_cost_reference(per._h, 0, 3, I.capi.dptr(q), I.capi.dptr(v)))
    for it in range(2):
        for s in (shared, per):
            s.updateSolution(0.0, q0, v0)     # samples the shared q_ref(t): shared sets on both handles
            s.computeKKTResidual(0.0, q0, v0)
        same_iterates(shared, per, ("fill", it))
    # (b) another shared reference on `per`: its sets leave the per-instance table as it is
    per.q_ref = lambda t: (pr.q_ref(t) + np.eye(19)[2] * 0.05, pr.v_ref)
    for it in range(2):
        for s in (shared, per):
            s.updateSolution(0.0, q0, v0)
            s.computeKKTResidual(0.0, q0, v0)
        same_iterates(shared, per, ("shared set", it))
    # ... and the clear returns to it: the raised base reference now changes the iterate
    per.clearInstanceCostReferences()
    for s in (shared, per):
        s.updateSolution(0.0, q0, v0)
        s.computeKKTResidual(0.0, q0, v0)
    assert not np.array_equal(shared.KKTError(), per.KKTError())
    assert not np.array_equal(shared.get(len(per.chain()) - 1, "q"), per.get(len(per.chain()) - 1, "q"))


def test_sharded_instance_references_equal_single_handle(fb, emu_lib):
    variants = FIXED_VARIANTS + [dict(dz=0.01, knee=1.5, vx=0.25)]
    pr = ap.TrottingProblem()
    q0, v0 = anymal_states(pr, len(variants), 20240012)
    _, one, _, _ = setup(emu_lib, fb, variants, q0, v0)
    _, many, _, _ = setup(emu_lib, fb, variants, q0, v0, devices=[0, 0])
    for it in range(3):
        for s in (one, many):
            s.updateSolution(0.0, q0, v0, it == 1)
            s.computeKKTResidual(0.0, q0, v0)
        same_iterates(one, many, it)
    for s in (one, many):
        s.clearInstanceCostReferences()
        s.updateSolution(0.0, q0, v0)
    same_iterates(one, many, "clear")


def test_instance_reference_errors(fb, emu_lib):
    pr = ap.TrottingProblem()
    s = ap.make_product_solver(pr, emu_lib, fb, batch=2)
    L = emu_lib.L
    q = np.zeros((2, 19))
    v = np.zeros((2, 18))
    dp = I.capi.dptr
    with pytest.raises(I.Idocp_b200Error, match="null pointer"):
        emu_lib.check(L.idocp_b200_fb_set_instance_cost_reference(s._h, 0, 0, None, dp(v)))
    with pytest.raises(I.Idocp_b200Error, match="null pointer"):
        emu_lib.check(L.idocp_b200_fb_set_instance_cost_reference(s._h, 0, 0, dp(q), None))
    with pytest.raises(I.Idocp_b200Error, match="null pointer"):
        emu_lib.check(L.idocp_b200_fb_set_instance_cost_reference(None, 0, 0, dp(q), dp(v)))
    with pytest.raises(I.Idocp_b200Error, match="null pointer"):
        emu_lib.check(L.idocp_b200_fb_clear_instance_cost_references(None))
    for kind in (-1, 5):
        with pytest.raises(I.Idocp_b200Error, match="fb_set_instance_cost_reference: kind"):
            emu_lib.check(L.idocp_b200_fb_set_instance_cost_reference(s._h, kind, 0, dp(q), dp(v)))
    for kind, index in ((0, -1), (0, pr.N + 1), (4, pr.N + 1), (1, pr.max_num_impulse), (2, pr.max_num_impulse), (3, -1)):
        with pytest.raises(I.Idocp_b200Error, match="fb_set_instance_cost_reference: index"):
            emu_lib.check(L.idocp_b200_fb_set_instance_cost_reference(s._h, kind, index, dp(q), dp(v)))
    # the terminal stage is FB_GRID / FB_TERMINAL with index N, as for the shared reference
    emu_lib.check(L.idocp_b200_fb_set_instance_cost_reference(s._h, 0, pr.N, dp(q), dp(v)))
    emu_lib.check(L.idocp_b200_fb_set_instance_cost_reference(s._h, 4, pr.N, dp(q), dp(v)))
    emu_lib.check(L.idocp_b200_fb_clear_instance_cost_references(s._h))
    for bad in (lambda t: (np.zeros(19), np.zeros((2, 18))), lambda t: (np.zeros((2, 19)), np.zeros((3, 18))),
                lambda t: (np.zeros((2, 18)), np.zeros((2, 18)))):
        s.setInstanceCostReference(bad)
        with pytest.raises(ValueError):
            s.updateSolution(0.0, pr.q0, pr.v0)
    sh = ap.make_product_solver(pr, emu_lib, fb, batch=3, devices=[0, 0])
    with pytest.raises(I.Idocp_b200Error, match="null pointer"):
        emu_lib.check(L.idocp_b200_fb_sharded_set_instance_cost_reference(sh._h, 0, 0, None, dp(np.zeros((3, 18)))))
    with pytest.raises(I.Idocp_b200Error, match="fb_set_instance_cost_reference: kind"):
        emu_lib.check(L.idocp_b200_fb_sharded_set_instance_cost_reference(sh._h, 7, 0, dp(np.zeros((3, 19))), dp(np.zeros((3, 18)))))


# ---- GPU ---------------------------------------------------------------------------------------------------------------

@pytest.mark.gpu
@pytest.mark.parametrize("line_search", [False, True])
def test_gpu_instance_references_match_per_instance_oracles(fb, gpu_lib, line_search):
    pr = ap.TrottingProblem()
    q0, v0 = anymal_states(pr, 64, 20240013)
    parity_case(gpu_lib, fb, random_variants(64, 20240014), line_search, sample=[0, 1, 17, 38, 50, 63], q0=q0, v0=v0)


@pytest.mark.gpu
def test_gpu_four_references_over_1024_instances_equal_shared_handles(fb, gpu_lib):
    # instance b gets reference b % 4; every instance equals the same instance of the shared-mode handle of its reference
    B = 1024
    variants = [dict(dz=0.0, knee=1.7, vx=0.3), dict(dz=-0.04, knee=1.2, vx=0.2), dict(dz=0.03, knee=2.0, vx=0.4),
                dict(dz=0.015, knee=1.5, vx=0.25)]
    problems = [InstanceTrotting(**v) for v in variants]
    q0, v0 = anymal_states(problems[0], B, 20240015)
    per = ap.make_product_solver(problems[0], gpu_lib, fb, batch=B, q0=q0, v0=v0)
    per.setInstanceCostReference(reference_fn([problems[b % 4] for b in range(B)]))
    shared = [ap.make_product_solver(p, gpu_lib, fb, batch=B, q0=q0, v0=v0) for p in problems]
    rows = [np.arange(k, B, 4) for k in range(4)]
    for it in range(3):
        kkt = []
        for s in [per] + shared:
            s.computeKKTResidual(0.0, q0, v0)
            kkt.append(s.KKTError())
            s.updateSolution(0.0, q0, v0, it == 1)
        for k, s in enumerate(shared):
            assert np.array_equal(kkt[0][rows[k]], kkt[1 + k][rows[k]]), (it, k)
            assert np.array_equal(per.stepSizes()[rows[k]], s.stepSizes()[rows[k]]), (it, k)
        for e in range(len(per.chain())):
            for nm in SOL + ["slack", "dual", "dq", "dv"]:
                got = per.get(e, nm)
                for k, s in enumerate(shared):
                    assert np.array_equal(got[rows[k]], s.get(e, nm)[rows[k]], equal_nan=True), (it, e, nm, k)


@pytest.mark.gpu
def test_gpu_batched_mpc_ticks_with_instance_references(fb, gpu_lib):
    B, iterations = 6, 2
    q, v = anymal_states(ap.TrottingProblem(), B, 20240017)
    problems, solver, q, v = setup(gpu_lib, fb, random_variants(B, 20240016), q, v)
    oracles = [p.make_oracle(fb, q0=q[b], v0=v[b]) for b, p in enumerate(problems)]
    mpc = I.BatchedMPC(solver, iterations=iterations)
    for t in (0.0, 0.3, 0.52):
        u0 = mpc.tick(t, q, v)
        cs = oracles[0].cs
        while cs.counts()[1] + cs.counts()[2] > 0:
            first = min(([cs.impulse(0)[2]] if cs.counts()[1] else []) + ([cs.lift_time(0)] if cs.counts()[2] else []))
            if first > t:
                break
            for o in oracles:
                o.cs.pop_front()
        for _ in range(iterations):
            for p, o in zip(problems, oracles):
                p.set_references(o, t)
            assert all(o.update_solution(t, q[b], v[b]) == 0 for b, o in enumerate(oracles)), t
        assert np.array_equal(u0, fb.batch_get(oracles, 0, "u")), t
        for b, o in enumerate(oracles):
            assert compare(o, solver, fb, SOL, b=b) == [], (t, b)
        q, v = fb.batch_get(oracles, 1, "q"), fb.batch_get(oracles, 1, "v")
    assert mpc.popped >= 1


EXE = os.path.join(ROOT, "build", "anymal_trotting_instance_refs")


def _build_example():
    import __graft_entry__ as g
    g.build_cuda()
    os.makedirs(os.path.join(ROOT, "build"), exist_ok=True)
    lib = os.path.join(ROOT, "idocp_b200")
    subprocess.check_call(["g++", "-std=c++17", "-Wall", "-Wextra", "-I" + os.path.join(ROOT, "include"),
                           os.path.join(ROOT, "examples", "anymal_trotting_instance_refs.cpp"), "-L" + lib, "-lidocp_b200",
                           "-Wl,-rpath," + lib, "-o", EXE])


def test_trotting_instance_refs_example_compiles_and_fails_loudly_without_gpu():
    import torch
    _build_example()
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    res = subprocess.run([EXE, "4"], capture_output=True, text=True)
    assert res.returncode != 0
    assert "no CUDA device" in res.stderr


@pytest.mark.gpu
def test_trotting_instance_refs_example_equals_the_oracles(fb):
    """examples/anymal_trotting_instance_refs.cpp (a base height offset and a knee swing amplitude per instance through the
    C++ host classes): the printed KKT errors equal those of per-instance oracles digit for digit."""
    _build_example()
    batch, iters = 5, 6
    out = subprocess.run([EXE, str(batch), str(iters)], capture_output=True, text=True, check=True).stdout
    rows = re.findall(r"instance (\d+): base height offset = (\S+) knee swing = (\S+) KKT error = (\S+)", out)
    assert len(rows) == batch, out
    # the host classes compute the contact points with the host's forward kinematics (anymal_trotting_golden.json holds them)
    with open(os.path.join(ROOT, "tests", "golden", "anymal_trotting_golden.json")) as f:
        pts = np.array(json.load(f)["contact_points"])
    for b, dz, knee, kkt in rows:
        b = int(b)
        assert float(dz) == 0.01 * (b % 5) - 0.02 and float(knee) == 1.3 + 0.1 * (b % 9), b
        p = InstanceTrotting(dz=float(dz), knee=float(knee))
        p.standing_points = pts
        o = p.make_oracle(fb)
        for _ in range(iters):
            assert o.update_solution(0.0, p.q0, p.v0) == 0
        o.compute_kkt_residual(0.0, p.q0, p.v0)
        assert float(kkt) == o.kkt_error(), (b, kkt, o.kkt_error())
