"""What per-instance cost references cost on the GPU: time per batched updateSolution with the shared references against the
same solver with per-instance references (idocp_b200_set_instance_reference / _task_reference), arms alternated round by
round inside one process, CUDA events on the solver's stream.

  python tools/bench_instance_refs.py [--rounds 5] [--warmup 10] [--iters 100] [--out profiles/instance_refs_b200.json]

Workloads (bench.py's problems and initial states):
  iiwa14_unocp           UnOCPSolver, configuration-space cost, B = 16384, N = 20, no line search; arms: shared, per-instance
                         q_ref / v_ref / u_ref equal to the shared values, per-instance random q_ref inside the joint limits
  iiwa14_unparnmpc_task  UnParNMPCSolver, 6D task-space cost, B = 2048, N = 120; arms: shared table, per-instance tables
                         (the shared circle with a per-instance position offset)
plus the host-to-device time of one per-instance task table (set_instance_task_reference: transpose + copy, blocking).
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


def device_info():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=" + q, "--format=csv,noheader"], capture_output=True, text=True,
                         check=True).stdout.strip()
    name, power, clock = [x.strip() for x in out.split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def time_arm(torch, solver, q0, v0, warmup, iters):
    """ms per updateSolution: CUDA events on the solver's stream around `iters` calls after `warmup` untimed ones"""
    stream = torch.cuda.ExternalStream(solver.stream())
    dq = torch.from_numpy(q0).cuda()
    dv = torch.from_numpy(v0).cuda()
    torch.cuda.synchronize()
    for _ in range(warmup):
        solver.updateSolutionDevice(0.0, dq.data_ptr(), dv.data_ptr())
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(iters):
        solver.updateSolutionDevice(0.0, dq.data_ptr(), dv.data_ptr())
    e1.record(stream)
    e1.synchronize()
    return e0.elapsed_time(e1) / iters


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--iters", type=int, default=100)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_instance_refs: no CUDA device (there is no CPU measurement)")
    import bench
    import idocp_b200 as I
    lib = I.default_library()
    info = device_info()
    result = {"device": info, "rounds": args.rounds, "warmup": args.warmup, "iters": args.iters, "workloads": {}}

    # ---- headline: iiwa14_unocp --------------------------------------------------------------------------------------
    prob = bench.workload_problem("iiwa14_unocp", I, lib)
    B = bench.IIWA_WORKLOADS["iiwa14_unocp"]["batch"]
    qmin, qmax = np.array(list(prob.q_min)), np.array(list(prob.q_max))
    q0, v0 = bench.workload_states("iiwa14_unocp", 0, B, list(qmin), list(qmax))
    rng = np.random.default_rng(1)
    arms = {}
    for arm in ("shared", "instance_shared_values", "instance_random"):
        s = I.UnOCPSolver(prob, B, lib=lib)
        s.setSolution("q", q0)
        s.setSolution("v", v0)
        if arm == "instance_shared_values":
            for name in ("q_ref", "v_ref", "u_ref"):
                s.setCostReference(name, np.tile(np.array(list(getattr(prob, name))), (B, 1)))
        elif arm == "instance_random":
            s.setCostReference("q_ref", rng.uniform(0.8 * qmin, 0.8 * qmax, (B, 7)))
        arms[arm] = s
    result["workloads"]["iiwa14_unocp"] = run_rounds(torch, arms, q0, v0, args)

    # ---- iiwa14_unparnmpc_task ---------------------------------------------------------------------------------------
    name = "iiwa14_unparnmpc_task"
    prob = bench.workload_problem(name, I, lib)
    B = bench.IIWA_WORKLOADS[name]["batch"]
    q0, v0 = bench.workload_states(name, 0, B, list(prob.q_min), list(prob.q_max))
    arms = {}
    for arm in ("shared", "instance_tables"):
        s = I.UnParNMPCSolver(prob, B, lib=lib)
        s.setSolution("q", q0)
        s.setSolution("v", v0)
        s.setTaskReference(I.task_space_circle_ref, 0.0)
        if arm == "instance_tables":
            base = np.array([I.task_space_circle_ref(t) for t in s.stageTimes(0.0)])
            tables = np.repeat(base[None], B, axis=0)
            tables[:, :, 9:12] += rng.uniform(-0.05, 0.05, (B, 1, 3))
            tables = np.ascontiguousarray(tables)
            s.setTaskReference(tables)
            t0 = time.perf_counter()
            for _ in range(5):
                s.setTaskReference(tables)
            upload_ms = (time.perf_counter() - t0) / 5 * 1e3
        s.initBackwardCorrection(0.0)
        arms[arm] = s
    result["workloads"][name] = run_rounds(torch, arms, q0, v0, args)
    result["task_table_upload"] = {"batch": B, "N": int(prob.N), "bytes": int(tables.nbytes), "ms_per_upload": upload_ms,
                                   "what": "setTaskReference(batch, N+1, 12): host transpose + blocking H2D copy, mean of 5"}
    line = json.dumps(result, indent=1)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


def run_rounds(torch, arms, q0, v0, args):
    """every round times every arm once, in turn; per arm: the per-round ms and their median"""
    ms = {a: [] for a in arms}
    for r in range(args.rounds):
        for a, s in arms.items():
            ms[a].append(time_arm(torch, s, q0, v0, args.warmup, args.iters))
    out = {a: {"ms_per_update": v, "median_ms": float(np.median(v))} for a, v in ms.items()}
    base = out[next(iter(arms))]["median_ms"]
    for a in out:
        out[a]["vs_shared"] = out[a]["median_ms"] / base
    return out


if __name__ == "__main__":
    main()
