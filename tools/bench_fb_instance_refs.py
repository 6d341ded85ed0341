#!/usr/bin/env python3
"""What per-instance cost references cost the floating-base OCPSolver on the GPU (idocp_b200_fb_set_instance_cost_reference):
the set-up of tools/bench_fb.py (anymal_trotting, B = 4096 by default), one solver per arm, arms alternated round by round
inside one process.

  python tools/bench_fb_instance_refs.py [--batch 4096] [--rounds 5] [--warmup 2] [--iters 10] [--out profiles/fb_instance_refs_b200.json]

Every arm first runs `--converge` updateSolution(0, q0, v0) calls without the line search: they upload the initial states and
the references (the resident arms below copy nothing afterwards) and bring every arm to its converged iterate, so all arms
are timed on the same kind of iterate.  (From bench_fb.py's states the filter line search on this problem diverges to NaN
after three iterations, shared and per-instance alike; from a converged iterate it stays finite, with the filter rejecting
the full step down to the 0.05 floor, so the line-search arms time every backtracking round.)
Arms (ms per updateSolution: host clock around `iters` calls, the device synchronised before the clock stops):
  shared             shared reference, updateSolutionResident (nothing sampled, states resident)
  instance_constant  per-instance references; updateSolutionResident, so the table is not copied again
  shared_sampled     shared reference, updateSolution(t, q, v): the reference sampled per stage and call, q / v copied
  instance_varying   per-instance references re-sampled every call (a per-call base height change): every slot of the chain
                     is rewritten and copied with q / v before the first kernel
  shared_sampled_ls    shared_sampled with the filter line search
  instance_varying_ls  instance_varying with the filter line search (k_fb_ls_eval<., IREF>)
The initial states are bench_fb.py's (random joint offsets and velocities); the KKT errors and primal step sizes after the
last call (NaN count included) are recorded with the times.
Per-kernel-class times (set_profiling, CUDA events around every launch) come from a separate profiled pass per arm:
fb_robot = k_fb_robot, line_search = the whole line-search class (k_fb_ls_eval + k_fb_ls_filter; k_fb_ls_eval is not timed
alone).  One full-table copy is timed through the library: every slot set through the C-ABI (host clock), then
computeKKTResidual with resident states (CUDA events on the solver's stream) with the whole table dirty minus the same call
with nothing dirty.
The device name and power limit are read in the same run.  There is no CPU path: without a GPU the script fails."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
sys.path.insert(0, os.path.join(ROOT, "tests"))

KNEES = [9, 12, 15, 18]
ARMS = ["shared", "instance_constant", "shared_sampled", "instance_varying", "shared_sampled_ls", "instance_varying_ls"]


def device_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                         check=True).stdout.strip()
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap_ = argparse.ArgumentParser()
    ap_.add_argument("--batch", type=int, default=4096)
    ap_.add_argument("--rounds", type=int, default=5)
    ap_.add_argument("--warmup", type=int, default=2)
    ap_.add_argument("--iters", type=int, default=10)
    ap_.add_argument("--converge", type=int, default=30)
    ap_.add_argument("--out", default=None)
    args = ap_.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_fb_instance_refs: no CUDA device (there is no CPU path)")
    import anymal_problems as ap
    import fb_py
    import idocp_b200 as I
    import oracle_py
    oracle_py.build()
    fb_py.lib()
    B = args.batch
    pr = ap.TrottingProblem()
    lib = I.default_library()
    rng = np.random.default_rng(0)
    q0 = np.tile(pr.q0, (B, 1))
    q0[:, 7:] += rng.uniform(-0.02, 0.02, (B, 12))
    v0 = rng.uniform(-0.1, 0.1, (B, 18))
    # per-instance references: the trot with a base height offset and a knee swing amplitude per instance
    dz = rng.uniform(-0.05, 0.05, B)
    knee = rng.uniform(1.2, 2.0, B)

    def q_ref_batch(t, shift=0.0):
        q = np.tile(pr.q_ref(t), (B, 1))
        q[:, 2] += dz + shift
        if t > pr.t_start:   # the knee swing of trotting_q_ref scales with the amplitude
            q[:, KNEES] = pr.q0[KNEES] + (q[:, KNEES] - pr.q0[KNEES]) * (knee / 1.7)[:, None]
        return q
    v_ref_batch = np.tile(pr.v_ref, (B, 1))
    calls = {"n": 0}

    def varying(t):
        return q_ref_batch(t, 1e-4 * (calls["n"] % 2)), v_ref_batch

    solvers = {}
    for arm in ARMS:
        s = ap.make_product_solver(pr, lib, fb_py, batch=B, q0=q0, v0=v0)
        if arm == "instance_constant":
            s.setInstanceCostReference(lambda t: (q_ref_batch(t), v_ref_batch))
        elif arm.startswith("instance_varying"):
            s.setInstanceCostReference(varying)
        for _ in range(args.converge):
            s.updateSolution(0.0, q0, v0)          # uploads x0 and the references; the resident arms copy nothing later
        solvers[arm] = s

    def run(arm, n):
        s = solvers[arm]
        ls = arm.endswith("_ls")
        for _ in range(n):
            if arm in ("shared", "instance_constant"):
                s.updateSolutionResident(0.0, ls)
            else:
                calls["n"] += 1
                s.updateSolution(0.0, q0, v0, ls)

    ms = {arm: [] for arm in ARMS}
    for r in range(args.rounds):
        order = ARMS if r % 2 == 0 else ARMS[::-1]
        for arm in order:
            run(arm, args.warmup)
            solvers[arm].sync()
            t0 = time.perf_counter()
            run(arm, args.iters)
            solvers[arm].sync()
            ms[arm].append((time.perf_counter() - t0) / args.iters * 1e3)
    kernels = {}
    for arm in ARMS:
        s = solvers[arm]
        s.sync()
        s.setProfiling(True)
        run(arm, args.iters)
        prof = s.getProfile()
        s.setProfiling(False)
        kernels[arm] = {k: prof[k]["ms"] / args.iters for k in ("fb_robot", "line_search") if k in prof and prof[k]["calls"]}
    kkt = {}
    for arm in ARMS:
        alpha = solvers[arm].stepSizes()[:, 0]
        solvers[arm].computeKKTResidual(0.0, q0, v0)
        e = solvers[arm].KKTError()
        kkt[arm] = {"median": float(np.median(e)), "nan": int(np.isnan(e).sum()), "primal_step_median": float(np.median(alpha))}

    # one full-table copy through the library: every slot set through the C-ABI, then a resident computeKKTResidual that
    # copies the dirty slots before its kernels, against the same call with nothing dirty
    s = solvers["instance_constant"]
    stream = torch.cuda.ExternalStream(s.stream())
    n_slots = pr.N + 1 + 3 * pr.max_num_impulse
    qb, vb = np.ascontiguousarray(q_ref_batch(0.0)), np.ascontiguousarray(v_ref_batch)
    slots = [(0, i) for i in range(pr.N + 1)] + [(k, i) for k in (1, 2, 3) for i in range(pr.max_num_impulse)]

    def kkt_call():
        s.sync()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        lib.check(s._f("compute_kkt_residual")(s._h, 0.0, None, None))
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1)
    set_ms, dirty_ms, clean_ms = [], [], []
    for _ in range(6):
        s.sync()
        t0 = time.perf_counter()
        for kind, index in slots:
            lib.check(s._f("set_instance_cost_reference")(s._h, kind, index, I.capi.dptr(qb), I.capi.dptr(vb)))
        set_ms.append((time.perf_counter() - t0) * 1e3)
        dirty_ms.append(kkt_call())
        clean_ms.append(kkt_call())
    set_ms, dirty_ms, clean_ms = set_ms[1:], dirty_ms[1:], clean_ms[1:]
    table_bytes = n_slots * B * 37 * 8

    out = {
        "what": "floating-base OCPSolver, anymal_trotting, per-instance cost references against the shared reference",
        "device": device_info(), "batch": B, "stages": len(solvers["shared"].chain()), "slots": n_slots,
        "rounds": args.rounds, "iters_per_round": args.iters, "warmup_per_round": args.warmup,
        "ms_per_update_solution": {arm: {"median": float(np.median(v)), "rounds": v} for arm, v in ms.items()},
        "kernel_class_ms_per_call": kernels,
        "kkt_after": kkt,
        "table": {"bytes": table_bytes, "chain_bytes_per_call": len(solvers["shared"].chain()) * B * 37 * 8,
                  "host_set_all_slots_ms": {"median": float(np.median(set_ms)), "samples": set_ms},
                  "kkt_residual_whole_table_dirty_ms": {"median": float(np.median(dirty_ms)), "samples": dirty_ms},
                  "kkt_residual_nothing_dirty_ms": {"median": float(np.median(clean_ms)), "samples": clean_ms},
                  "copy_ms": float(np.median(dirty_ms) - np.median(clean_ms))},
    }
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
