"""bench.py output contract on the CPU box: the reference arm (`--impl reference`, the CPU oracle timed on the host
cores) prints exactly ONE line on stdout, that line is the JSON object the driver parses, and chatter written to
file descriptor 1 by libraries (NCCL's version banner) cannot get in front of it."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(args, env=None):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, capture_output=True, text=True,
                         timeout=600, env={**os.environ, **(env or {})})
    assert res.returncode == 0, res.stderr[-2000:]
    return res.stdout


def test_reference_arm_prints_one_json_line():
    out = _run(["--impl", "reference", "--steps", "3", "--warmup", "3"])
    lines = out.splitlines()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["n_gpus"] == 1 and d["higher_is_better"] is True
    assert d["unit"] == "instance-iterations/s" and d["value"] > 0 and d["dtype"] == "f64"
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"]


def test_reference_arm_other_ranks_print_nothing():
    out = _run(["--impl", "reference", "--gpus", "2", "--steps", "3", "--warmup", "3"], env={"RANK": "1", "WORLD_SIZE": "2"})
    assert out == ""


def test_stdout_is_claimed_before_any_library_can_write_to_it():
    code = ("import os, sys; sys.path.insert(0, %r); import bench; bench.claim_stdout(); "
            "os.write(1, b'NCCL version 2.28.9+cuda12.9\\n'); print('chatter'); bench.emit_line({'ok': 1})" % ROOT)
    res = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
    assert res.returncode == 0, res.stderr
    assert res.stdout == '{"ok": 1}\n'
    assert "NCCL version" in res.stderr and "chatter" in res.stderr


def test_dump_outputs_needs_the_gpu_solver(tmp_path):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", str(tmp_path)],
                         cwd=ROOT, capture_output=True, text=True, timeout=120)
    assert res.returncode != 0 and "--dump-outputs" in res.stderr
    assert os.listdir(tmp_path) == []


def _solution_after(workload, B, warmup, steps):
    """The solution of a solver set up and iterated as bench.py's timed path does, read back through the public API."""
    import bench
    import idocp_b200 as I
    from idocp_b200 import problems as P
    lib = I.default_library()
    if workload in bench.IIWA_WORKLOADS:
        prob = bench.workload_problem(workload, I, lib)
        q0, v0 = bench.workload_states(workload, 0, B, list(prob.q_min), list(prob.q_max))
        solver = I.UnOCPSolver(prob, B)
        solver.setSolution("q", q0)
        solver.setSolution("v", v0)
        for _ in range(warmup + steps):
            solver.updateSolution(0.0, q0, v0)
        return {n: solver.getSolution(n) for n in ("q", "v", "a", "u", "lmd", "gmm", "beta")}
    pr = bench.anymal_problem(workload, lib)
    ls = bench.ANYMAL_LINE_SEARCH[workload]
    q0, v0 = P.anymal_initial_states(0, B, q_nominal=pr.q_nominal, seed=bench.ANYMAL_SEED[workload])
    solver = P.make_solver(pr, B, q0, v0, lib=lib)
    solver.updateSolution(0.0, q0, v0, ls)
    for _ in range(warmup + steps):
        solver.updateSolutionResident(0.0, ls)
    return {n: np.stack(solver.getSolution(n), axis=1) for n in ("q", "v", "a", "u", "f")}


@pytest.mark.gpu
@pytest.mark.parametrize("workload, B", [("iiwa14_unocp", 256), ("anymal_trotting", 16)])
def test_dump_outputs_hold_the_solution_after_the_last_timed_step(tmp_path, workload, B):
    """--dump-outputs writes the solution after the warmup + steps iterations of the timed path, the same numbers on every run."""
    steps, warmup = 4, 3
    args = ["--workload", workload, "--batch", str(B), "--steps", str(steps), "--warmup", str(warmup), "--no-cpu-baseline"]
    _run(args + ["--dump-outputs", str(tmp_path / "a")])
    _run(args + ["--dump-outputs", str(tmp_path / "b")])
    ref = _solution_after(workload, B, warmup, steps)
    assert sorted(os.listdir(tmp_path / "a")) == sorted(n + ".npy" for n in ref)
    for n, want in ref.items():
        a, b = np.load(tmp_path / "a" / (n + ".npy")), np.load(tmp_path / "b" / (n + ".npy"))
        assert a.dtype == np.float64 and np.array_equal(a, b, equal_nan=True), n
        assert np.array_equal(a, want, equal_nan=True), n
