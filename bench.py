#!/usr/bin/env python3
"""bench.py -- batched SQP iterations/sec of the iiwa14 UnOCPSolver hot path (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (N>1: launched through torch.distributed.run)
  python bench.py --impl reference --gpus N --steps K --warmup W

One "step" = one updateSolution (one SQP / Newton iteration) of EVERY instance of the batch.
Workload = BASELINE.json configs[2]: examples/iiwa14/unocp_benchmark.cpp problem (N=20, T=1),
16384 random initial states per GPU (counter-based splitmix64, seed 20240001; SURVEY.md 8d).
Weak scaling: every rank owns its own 16384 instances, no data-path collective.

  value  : instance-iterations/s over all ranks with q0/v0 already resident in HBM
  e2e    : same through the public host API (updateSolution(host q, host v) + getStageSolution("u", 0)):
           H2D of x0 and D2H of the first control input inside the timed region
  roofline / cpu_baseline : see DESIGN.md "Measurement"
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SEED = 20240001
BATCH_PER_GPU = 16384
HORIZON_N = 20
NV = 7
# algorithmic FP64 work / mandatory HBM bytes per instance-iteration (SURVEY.md section 8d)
FLOP_PER_UNIT = 0.46e6
BYTES_PER_UNIT = 44e3
# algorithmic bytes per (instance, stage) of each kernel = its mandatory inputs + outputs, unpadded
# doubles (DESIGN.md "Kernels"):  linearize: s_i 49 + s_{i+1} 28 + slack/dual 84 in; Q 231 + res 35 + exp 147 out
KERNEL_ALGO_DOUBLES_PER_STAGE = {
    # s_i 49 + (q,v,lmd,gmm)_{i+1} 28 + slack/dual 84 in; Q (3 sym 28 + 3 full 49) 231 + res 35 + expansion 147 out
    "linearize": 49 + 28 + 84 + 231 + 35 + 147,
    # Q 231 + res 35 in; K 98 + k 7 + P (28+49+28) + s 14 out; forward: K,k 105 + Fx 14 in, (dq,dv,da) 21 out
    "riccati": 231 + 35 + 105 + 105 + 14 + 105 + 14 + 21,
    # P,s 119 + expansion 147 + (dq,dv,da) 21 + (q,v,u) 21 + slack/dual 84 in; (dlmd,dgmm,du,dbeta) 28 out
    "expand": 119 + 147 + 21 + 21 + 84 + 28,
    # s 49 + slack/dual 84 + d 49 in; s 49 + slack/dual 84 out
    "update": 2 * (49 + 84) + 49,
    # the persistent fused kernel (update of iteration k + linearisation for iteration k + 1; its step sizes come from
    # k_step_min, class "step_min"): linearize + the direction in (d_i 49, d_{i+1} 28) + the new iterate out (s 49 + slack/dual 84)
    "update_linearize": (49 + 28 + 84 + 231 + 35 + 147) + (49 + 28) + (49 + 84),
    # UnParNMPC coarse update (k_parnmpc_invert): Q 231 + res 35 + aux_next 105 + s 35 in; the four blocks of the inverse the
    # sweeps multiply with (14x14 + 21x14 + 14x14 + 21x14 = 980) + s_new 35 out
    "parnmpc_coarse": 231 + 35 + 105 + 35 + 980 + 35,
}
# UnParNMPC: k_expand<PARNMPC> reads no Riccati data (the costate direction comes from the correction sweeps):
# expansion 147 + (dq,dv,da) 21 + (q,v,u) 21 + slack/dual 84 in; (du,dbeta) 14 out
KERNEL_ALGO_DOUBLES_PER_STAGE_PARNMPC = dict(KERNEL_ALGO_DOUBLES_PER_STAGE, expand=147 + 21 + 21 + 84 + 14)


# ncu evidence is PARSED, not typed in: tools/ncu_capture.sh (run under gpurun) writes profiles/kernel_counters_<workload>.json
# (per kernel: DRAM bytes read + written, executed FP64 thread instructions, pipe / issue utilisation of one launch at the
# bench batch); tools/fp64_peak (DFMA microbenchmark on the B200) writes profiles/fp64_peak.json.
# (instantiation names as ncu prints them; the older spellings are kept for captures made before the ACC / KKT template flags)
KERNEL_OF_CLASS = {"linearize": ("k_linearize<0,0,0,0>", "k_linearize<0,0,0>"), "riccati": ("k_riccati<0>",),
                   "expand": ("k_expand<0,0,0>", "k_expand<0,0>"), "update": ("k_update",),
                   "update_linearize": ("k_update_linearize<0,0>", "k_update_linearize<0>"),
                   "fb_robot": ("k_fb_robot<0>",), "fb_condense": ("k_fb_condense",), "fb_riccati_backward": ("k_fb_riccati_backward",),
                   "parnmpc_coarse": ("k_parnmpc_invert",)}
# The iiwa14 workloads of bench.py (all through the same code path, run_iiwa):
#   iiwa14_unocp           BASELINE configs[2] -- the headline: UnOCPSolver, unocp_benchmark problem, N = 20, 16384 states / GPU
#   iiwa14_unparnmpc_task  BASELINE configs[1]: task_space_ocp problem (T = 6, N = 120, TimeVaryingTaskSpace6DCost, circular
#                          reference) through UnParNMPCSolver with initBackwardCorrection, as unparnmpc_benchmark.cpp:46-56 drives
#                          it; 2048 states / GPU = the example's q0 (task_space_ocp.cpp:86-88) + 0.3 U(-1,1), v0 = 0.2 U(-1,1)
#   iiwa14_unocp_config    BASELINE configs[0]: config_space_ocp problem (T = 3, N = 60) through UnOCPSolver, 8192 states / GPU
#                          = the example's q0 + 0.3 U(-1,1), v0 = 0.2 U(-1,1)
IIWA_WORKLOADS = {
    "iiwa14_unocp": {"solver": "unocp", "problem": "benchmark", "batch": 16384, "seed": 20240001,
                     "what": "iiwa14 config-space UnOCPSolver (examples/iiwa14/unocp_benchmark.cpp problem), N=20, T=1"},
    "iiwa14_unparnmpc_task": {"solver": "unparnmpc", "problem": "task", "batch": 2048, "seed": 20240002,
                              "what": "iiwa14 task_space_ocp problem (examples/iiwa14/task_space_ocp.cpp:55-93, 6D circular "
                                      "reference) through UnParNMPCSolver + initBackwardCorrection, N=120, T=6"},
    "iiwa14_unocp_config": {"solver": "unocp", "problem": "config", "batch": 8192, "seed": 20240000,
                            "what": "iiwa14 config_space_ocp problem (examples/iiwa14/config_space_ocp.cpp:26-61) through "
                                    "UnOCPSolver, N=60, T=3"},
}
# 64 DFMA / clk / SM (ncu: sm__sass_thread_inst_executed_op_dfma_pred_on.avg.peak_sustained) x 148 SMs x 1.965 GHz x 2
FP64_PEAK_NOMINAL_TFLOPS = 64 * 148 * 1.965e9 * 2 / 1e12


def load_kernel_counters(workload):
    """profiles/kernel_counters_<workload>.json -> ({class name: counters}, source) or ({}, None)."""
    path = os.path.join(ROOT, "profiles", "kernel_counters_%s.json" % workload)
    if not os.path.exists(path):
        return {}, None
    with open(path) as f:
        rec = json.load(f)
    out = {}
    for cls, names in KERNEL_OF_CLASS.items():
        for kname in names:
            if kname in rec["kernels"]:
                out[cls] = rec["kernels"][kname]
                break
    return out, "profiles/kernel_counters_%s.json (%s)" % (workload, rec.get("source"))


def fp64_peak():
    """(burst TFLOP/s, sustained TFLOP/s, source): measured DFMA peak of this pool's B200 (tools/fp64_peak.cu)."""
    path = os.path.join(ROOT, "profiles", "fp64_peak.json")
    if os.path.exists(path):
        with open(path) as f:
            rec = json.load(f)
        return rec["fp64_dfma_tflops"], rec["fp64_dfma_tflops_sustained"], "measured (profiles/fp64_peak.json, tools/fp64_peak.cu)"
    return FP64_PEAK_NOMINAL_TFLOPS, FP64_PEAK_NOMINAL_TFLOPS, "fallback: 64 DFMA/clk/SM x 148 SMs x 1965 MHz (no profiles/fp64_peak.json)"


def kernel_roofline(name, per_launch_ms, algo_bytes, counters, batch_matches, hbm_peak, fp64_sustained):
    """Both roofline fractions of one kernel: HBM from the ALGORITHMIC bytes, FP64 from the FP64 thread instructions
    ncu counted for one launch at the same batch (executed work: the padding lane and redundant lanes included)."""
    k = {"ms_per_launch": per_launch_ms, "algo_gbs": algo_bytes / (per_launch_ms * 1e-3) / 1e9}
    k["frac_hbm"] = k["algo_gbs"] / hbm_peak
    c = counters.get(name) if batch_matches else None
    if c and "fp64_flop_executed" in c:
        k["fp64_tflops"] = c["fp64_flop_executed"] / (per_launch_ms * 1e-3) / 1e12
        k["frac_fp64"] = k["fp64_tflops"] / fp64_sustained
        k["ncu_dram_bytes"] = c.get("dram_bytes")
        k["ncu_dram_gbs_at_measured_time"] = c.get("dram_bytes", 0.0) / (per_launch_ms * 1e-3) / 1e9
        k["ncu_fp64_pipe_pct"] = c.get("fp64_pipe_pct")
        k["ncu_issue_active_pct"] = c.get("issue_active_pct")
        k["ncu_registers"] = c.get("registers")
    else:
        k["frac_fp64"] = None
    k["bound"] = "fp64" if (k["frac_fp64"] or 0.0) > k["frac_hbm"] else "hbm"
    return k


def roofline_object(dom, kern, algo_bytes, hbm_peak, peak_src, fp64_sustained, fp64_src, counters_src, note):
    """The contract's roofline object for the dominant kernel: bound = the larger of its two fractions."""
    k = kern[dom]
    if k["bound"] == "fp64":
        head = {"bound": "fp64", "achieved": k["fp64_tflops"], "peak": fp64_sustained, "unit": "TFLOP/s", "frac": k["frac_fp64"],
                "peak_source": fp64_src + " (sustained figure: the kernel is timed inside a long step)"}
    else:
        head = {"bound": "hbm", "achieved": k["algo_gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": k["frac_hbm"], "peak_source": peak_src}
    head.update({"kernel": dom, "frac_hbm": k["frac_hbm"], "frac_fp64": k["frac_fp64"], "traffic": k.get("ncu_dram_bytes"),
                 "traffic_source": counters_src if k.get("ncu_dram_bytes") else None,
                 "algorithmic_bytes_per_launch": algo_bytes, "hbm_peak_gbs": hbm_peak, "fp64_peak_tflops": fp64_sustained,
                 "fp64_peak_source": fp64_src, "note": note, "kernels": kern})
    return head


_JSON_OUT = None


def claim_stdout():
    """stdout carries exactly ONE JSON line: file descriptor 1 is pointed at stderr for the rest of the process
    (NCCL prints its version banner to fd 1 at NCCL_DEBUG=VERSION and WARN; libraries may chat), and the line is
    written through a private duplicate of the original stdout."""
    global _JSON_OUT
    if _JSON_OUT is None:
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit_line(line):
    out = _JSON_OUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


# --dump-outputs: every array of one run together stays under 64 MB (np.save adds a header of about 128 bytes per file)
DUMP_LIMIT_BYTES = 60 << 20


def dump_outputs(out_dir, arrays, seed):
    """Write out_dir/<name>.npy (float64) for each (batch, ...) array of `arrays`.  When all instances do not fit in
    DUMP_LIMIT_BYTES, every file holds the same instances: a sample drawn with `seed`, in ascending instance order."""
    os.makedirs(out_dir, exist_ok=True)
    batch = len(next(iter(arrays.values())))
    per_instance = sum(a[0].nbytes for a in arrays.values())
    n = min(batch, DUMP_LIMIT_BYTES // per_instance)
    idx = np.sort(np.random.default_rng(seed).choice(batch, n, replace=False)) if n < batch else np.arange(batch)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a[idx], dtype=np.float64))


def splitmix_uniform(seed, index):
    """Counter-based splitmix64 -> double in [0,1); vectorised twin of oracle_splitmix_uniform."""
    idx = np.asarray(index, dtype=np.uint64)
    with np.errstate(over="ignore"):
        z = np.uint64(seed) + (idx + np.uint64(1)) * np.uint64(0x9E3779B97F4A7C15)
        z = (z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        z = (z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        z = z ^ (z >> np.uint64(31))
    return (z >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)


def initial_states(first_instance, count, q_min, q_max):
    """q0_j = c_j + 0.8 h_j U(-1,1), v0_j = 0.5 U(-1,1); element index = instance*14 + j."""
    inst = np.arange(first_instance, first_instance + count, dtype=np.uint64)[:, None]
    j = np.arange(NV, dtype=np.uint64)[None, :]
    uq = 2.0 * splitmix_uniform(SEED, inst * np.uint64(14) + j) - 1.0
    uv = 2.0 * splitmix_uniform(SEED, inst * np.uint64(14) + np.uint64(7) + j) - 1.0
    c = 0.5 * (np.asarray(q_max) + np.asarray(q_min))
    h = 0.5 * (np.asarray(q_max) - np.asarray(q_min))
    return np.ascontiguousarray(c + 0.8 * h * uq), np.ascontiguousarray(0.5 * uv)


def workload_states(name, first_instance, count, q_min, q_max):
    """Initial states of instances first_instance .. first_instance + count - 1 of an iiwa14 workload (counter-based: a
    shard of the batch is the same numbers on any rank / world size)."""
    w = IIWA_WORKLOADS[name]
    if w["problem"] == "benchmark":
        return initial_states(first_instance, count, q_min, q_max)
    base = np.array([0, np.pi / 2, 0, np.pi / 2, 0, np.pi / 2, 0]) if w["problem"] == "task" else \
        np.array([np.pi / 2, 0, np.pi / 2, 0, np.pi / 2, 0, np.pi / 2])
    inst = np.arange(first_instance, first_instance + count, dtype=np.uint64)[:, None]
    j = np.arange(NV, dtype=np.uint64)[None, :]
    uq = 2.0 * splitmix_uniform(w["seed"], inst * np.uint64(14) + j) - 1.0
    uv = 2.0 * splitmix_uniform(w["seed"], inst * np.uint64(14) + np.uint64(7) + j) - 1.0
    return np.ascontiguousarray(base + 0.3 * uq), np.ascontiguousarray(0.2 * uv)


def workload_problem(name, mod, lib=None):
    """The problem of an iiwa14 workload from idocp_b200 (mod = idocp_b200, lib = its library) or from the oracle
    (mod = oracle_py, lib = None): both expose benchmark_problem / task_space_problem / config_space_problem."""
    kind = IIWA_WORKLOADS[name]["problem"]
    args = (lib,) if lib is not None else ()
    if kind == "benchmark":
        return mod.benchmark_problem(*args, N=HORIZON_N, T=1.0)
    return mod.task_space_problem(*args) if kind == "task" else mod.config_space_problem(*args)


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.samples = []
        self.stop_flag = False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                parts = [p.strip() for p in out.strip().split(",")]
                if len(parts) >= 7:
                    self.samples.append(parts)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = [float(s[0]) for s in self.samples if s[0].replace(".", "").isdigit()]
        mx = [float(s[1]) for s in self.samples if s[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for k, n in enumerate(names) if any(s[3 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return json.load(f).get("hbm_gbs"), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


CPU_WARM_SECONDS = 3.0     # both CPU legs warm up for this long first: OpenMP team start-up, page faults and the cores'
                           # frequency ramp cost ~30 % on a cold 20-sweep run (VERDICT r1: 260 k/s vs 382 k/s on one box)


def _oracle_batch(workload, cores):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle_py as O
    w = IIWA_WORKLOADS[workload]
    prob = workload_problem(workload, O)
    nb = max(cores * 16, 256) if prob.N <= 20 else max(cores * 4, 64)
    q0, v0 = workload_states(workload, 0, nb, list(prob.q_min), list(prob.q_max))
    batch = O.Batch(prob, nb, kind=w["solver"])
    for b, s in enumerate(batch.solvers):
        s.set_solution("q", q0[b])
        s.set_solution("v", v0[b])
        if w["problem"] == "task":
            s.set_task_ref(O.task_ref_table(O.task_space_ref, 0.0, prob.T, prob.N, kind=w["solver"]))
        if w["solver"] == "unparnmpc":
            s.init_backward_correction(0.0)
    t_end = time.perf_counter() + CPU_WARM_SECONDS
    sweeps = 0
    while time.perf_counter() < t_end or sweeps < 3:
        batch.update_solution(0.0, q0, v0, False, cores)
        sweeps += 1
    t0 = time.perf_counter()
    batch.update_solution(0.0, q0, v0, False, cores)
    return batch, nb, q0, v0, time.perf_counter() - t0


def oracle_throughput(seconds_target, workload="iiwa14_unocp", threads=None):
    """cpu_baseline leg: the CPU oracle (restatement of idocp's UnOCPSolver / UnParNMPCSolver) on the host cores, OpenMP over
    instances, every instance single-threaded (BASELINE.md mode B), ~seconds_target of sweeps after the warm-up.
    Returns (units/s, cores, sample, ms per sweep)."""
    cores = threads or os.cpu_count() or 1
    batch, nb, q0, v0, one = _oracle_batch(workload, cores)
    sweeps = int(max(3, min(4000, seconds_target / max(one, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(sweeps):
        batch.update_solution(0.0, q0, v0, False, cores)
    total = time.perf_counter() - t0
    sample = "%d instances x %d updateSolution sweeps after %.0f s of warm-up sweeps, OpenMP over instances, %d threads" % (
        nb, sweeps, CPU_WARM_SECONDS, cores)
    return nb * sweeps / total, cores, sample, total / sweeps * 1e3


def iiwa_metric(workload):
    return {"iiwa14_unocp": "batched SQP iterations/sec (iiwa14 N=20, FP64)",
            "iiwa14_unparnmpc_task": "batched ParNMPC iterations/sec (iiwa14 task-space N=120, UnParNMPCSolver, FP64)",
            "iiwa14_unocp_config": "batched SQP iterations/sec (iiwa14 config-space N=60, FP64)"}[workload]


def run_reference(args, rank, world):
    """--impl reference: idocp's own CPU algorithm.  The upstream library cannot be built in this image (Eigen / Boost /
    pinocchio / urdfdom absent), so this times the oracle restatement -- with the SAME protocol as the cpu_baseline leg of the
    GPU arm (same instance sample, same warm-up): one step = R sweeps over the sample, R sized for ~0.5 s per step."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    w = IIWA_WORKLOADS[args.workload]
    batch, nb, q0, v0, one = _oracle_batch(args.workload, cores)
    per_step = int(max(1, min(1000, round(0.5 / max(one, 1e-6)))))

    def step():
        for _ in range(per_step):
            batch.update_solution(0.0, q0, v0, False, cores)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    total = time.perf_counter() - t0
    value = float(nb) * per_step * args.steps / total
    sample = "%d instances x %d sweeps per step x %d steps after %.0f s + %d steps of warm-up, OpenMP over instances, %d threads" % (
        nb, per_step, args.steps, CPU_WARM_SECONDS, args.warmup, cores)
    line = {
        "impl": "reference", "metric": iiwa_metric(args.workload), "value": value,
        "unit": "instance-iterations/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": total / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic",
        "config": {"workload": "%s, random initial states (splitmix64 seed %d); bounded sample: %d instances x %d sweeps per step"
                               % (w["what"], w["seed"], nb, per_step)},
        "cpu_baseline": {"value": value, "unit": "instance-iterations/s", "cores": cores, "kind": "port",
                         "sample": sample},
        "e2e": {"value": value, "unit": "instance-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle restatement of idocp (oracle/idocp_oracle.c), not the upstream binary: pinocchio/Eigen absent",
    }
    emit_line(line)


# ---------------------------------------------------------------------------------------------------
# ANYmal workloads (BASELINE.json configs[3], configs[4]): batched OCPSolver with contacts and impulses
# ---------------------------------------------------------------------------------------------------
ANYMAL_BATCH = {"anymal_trotting": 4096, "anymal_running": 1024}
ANYMAL_SEED = {"anymal_trotting": 20240004, "anymal_running": 20240005}   # SURVEY 8(d) configs 4 and 5
ANYMAL_LINE_SEARCH = {"anymal_trotting": False, "anymal_running": True}
# algorithmic doubles per (instance, stage) of the heavy kernels at dimf = 12 (DESIGN.md section 8): mandatory inputs + outputs
FB_ALGO_DOUBLES_PER_STAGE = {
    "fb_robot": (181 + 224 + 73 + 19) + (30 + 1080 + 324 + 216 + 132 + 240 + 108),
    "fb_condense": (30 + 1080 + 324 + 216 + 132 + 240 + 108) + (972 + 648 + 324 + 972 + 90) + 3660,
    "fb_riccati_backward": (972 + 648 + 324 + 972 + 90) + (432 + 12 + 972 + 36),
}
# SURVEY section 8d: about 0.45 MFLOP per stage of the ANYmal path
FB_FLOP_PER_STAGE = 0.45e6


def anymal_problem(name, lib=None):
    from idocp_b200 import problems as P
    return P.AnymalTrotting(lib=lib) if name == "anymal_trotting" else P.AnymalRunning(lib=lib)


def anymal_oracle_throughput(name, seconds_target, steps=None, warmup=1):
    """CPU oracle of the ANYmal OCPSolver (oracle/fb_ocp.c) on the host cores: one oracle object per instance, a
    thread pool over instances (ctypes releases the GIL), every instance single-threaded = BASELINE.md mode B."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import anymal_problems as tp
    import fb_py
    import oracle_py
    from idocp_b200 import problems as P
    oracle_py.build()
    fb_py.lib()
    cores = os.cpu_count() or 1
    pr = tp.TrottingProblem() if name == "anymal_trotting" else tp.RunningProblem(10)
    ls = ANYMAL_LINE_SEARCH[name]
    nb = 2 * cores
    q0, v0 = P.anymal_initial_states(0, nb, q_nominal=pr.q0, seed=ANYMAL_SEED[name])
    solvers = [pr.make_oracle(fb_py, q0=q0[b], v0=v0[b]) for b in range(nb)]
    t_end = time.perf_counter() + CPU_WARM_SECONDS      # same warm-up protocol in the cpu_baseline leg and the reference arm
    n_warm = 0
    while time.perf_counter() < t_end or n_warm < max(warmup, 1):
        fb_py.batch_update_solution(solvers, 0.0, q0, v0, ls, cores)
        n_warm += 1
    t0 = time.perf_counter()
    fb_py.batch_update_solution(solvers, 0.0, q0, v0, ls, cores)
    first = time.perf_counter() - t0
    if steps is None:
        steps = int(max(2, min(200, seconds_target / max(first, 1e-6))))
    t0 = time.perf_counter()
    for _ in range(steps):
        fb_py.batch_update_solution(solvers, 0.0, q0, v0, ls, cores)
    total = time.perf_counter() - t0
    cores_used = cores
    sample = "%d instances x %d updateSolution sweeps, OpenMP over instances, %d threads" % (nb, steps, cores_used)
    return nb * steps / total, cores_used, sample, total / steps * 1e3


def anymal_metric(name):
    return ("batched SQP iterations/sec (ANYmal trotting OCPSolver N=30, FP64)" if name == "anymal_trotting"
            else "batched SQP iterations/sec (ANYmal running OCPSolver N=240, filter line search, FP64)")


def run_reference_anymal(args, rank):
    if rank != 0:
        return
    value, cores, sample, ms = anymal_oracle_throughput(args.workload, None, args.steps, args.warmup)
    line = {
        "impl": "reference", "metric": anymal_metric(args.workload), "value": value, "unit": "instance-iterations/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s (examples/anymal/%s.cpp problem), perturbed initial states (splitmix64 seed %d); "
                               "bounded sample of %d instances per step" % (args.workload, args.workload, ANYMAL_SEED[args.workload], 2 * cores)},
        "cpu_baseline": {"value": value, "unit": "instance-iterations/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "instance-iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "oracle restatement of idocp's OCPSolver (oracle/fb_ocp.c), not the upstream binary: pinocchio/Eigen absent",
    }
    emit_line(line)


def run_anymal(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import idocp_b200 as I
    from idocp_b200 import problems as P
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    lib = I.default_library()
    pr = anymal_problem(args.workload, lib)
    ls = ANYMAL_LINE_SEARCH[args.workload]
    B = args.batch if args.batch else ANYMAL_BATCH[args.workload]
    if args.scaling == "strong":
        B //= world
    q0, v0 = P.anymal_initial_states(rank * B, B, q_nominal=pr.q_nominal, seed=ANYMAL_SEED[args.workload])
    solver = P.make_solver(pr, B, q0, v0, device=local_rank, lib=lib)
    n_stages = len(solver.chain())
    stream = torch.cuda.ExternalStream(solver.stream(), device=local_rank)
    u_host = np.zeros((B, 12))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def count_over_ranks(n):
        if world == 1:
            return n
        t = torch.tensor([n], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return int(t.item())

    solver.updateSolution(0.0, q0, v0, ls)          # uploads x0 and the cost reference once
    for _ in range(args.warmup):
        solver.updateSolutionResident(0.0, ls)
    solver.sync()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    solver.setProfiling(True)
    launches0 = solver.launchCount()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        solver.updateSolutionResident(0.0, ls)
    e1.record(stream)
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = solver.launchCount() - launches0
    profile = solver.getProfile()
    solver.setProfiling(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {n: np.stack(solver.getSolution(n), axis=1) for n in ("q", "v", "a", "u", "f")},
                     ANYMAL_SEED[args.workload])
    # end-to-end: host states in, first control input out, through the public API
    for _ in range(3):
        solver.updateSolution(0.0, q0, v0, ls)
        u_host[:] = solver.get(0, "u")
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        solver.updateSolution(0.0, q0, v0, ls)
        u_host[:] = solver.get(0, "u")
    barrier()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3)
    if rank == 0:
        sampler.stop_flag = True
        sampler.join(timeout=2)
    solver.computeKKTResidual(0.0, q0, v0)
    kkt = solver.KKTError()
    # health: an instance whose KKT error is NaN has left the interior (the 0.05 floor of the filter line search can
    # exceed the fraction-to-boundary step, line_search.hpp:84-91 -- upstream behaviour, reproduced by the oracle at the
    # same iteration: tests/test_gpu_baseline_configs.py::test_config4_running_full_horizon); `value` counts LIVE ones
    live = np.isfinite(kkt)
    n_live = count_over_ranks(int(live.sum()))
    units = float(B) * world * args.steps
    value_all = units / (ms_total * 1e-3)
    value = float(n_live) * args.steps / (ms_total * 1e-3)
    hbm_peak, peak_src = measured_peaks()
    _, fp64_sus, fp64_src = fp64_peak()
    counters, counters_src = load_kernel_counters(args.workload)
    stages = B * n_stages
    kern = {}
    for name, rec in profile.items():
        if rec["calls"] and name in FB_ALGO_DOUBLES_PER_STAGE:
            per_launch = rec["ms"] / rec["calls"]
            kern[name] = kernel_roofline(name, per_launch, FB_ALGO_DOUBLES_PER_STAGE[name] * 8.0 * stages, counters,
                                         B == ANYMAL_BATCH[args.workload], hbm_peak, fp64_sus)
            kern[name]["ms_per_step"] = rec["ms"] / args.steps
            kern[name]["launches_per_step"] = rec["calls"] / args.steps
        elif rec["calls"]:
            kern[name] = {"ms_per_step": rec["ms"] / args.steps, "launches_per_step": rec["calls"] / args.steps}
    dom = max((n for n in kern if "algo_gbs" in kern[n]), key=lambda n: kern[n]["ms_per_step"], default=None)
    roofline = None
    if dom:
        roofline = roofline_object(dom, kern, FB_ALGO_DOUBLES_PER_STAGE[dom] * 8.0 * stages, hbm_peak, peak_src, fp64_sus, fp64_src,
                                   counters_src,
                                   "the ANYmal kernels are latency-bound (dependent FP64 chains of the factorisations, block "
                                   "barriers, 10-20 resident warps / SM); both fractions are reported, `bound` names the larger")
        roofline["step_fp64_tflops_algorithmic"] = FB_FLOP_PER_STAGE * n_stages * value_all / world / 1e12
    line = {
        "metric": anymal_metric(args.workload), "value": value, "unit": "instance-iterations/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s: OCPSolver on examples/anymal/%s.cpp (T=%g, N=%d, %d stages incl. impulse / aux / lift), %d "
                               "perturbed initial states per GPU (splitmix64 seed %d), line_search=%s"
                               % (args.workload, args.workload, pr.T, pr.N, n_stages, B, ANYMAL_SEED[args.workload], str(ls).lower()),
                   "batch_per_gpu": B, "stages": n_stages, "parallelism": "batch-sharded x%d, no collective" % world,
                   "l2_policy": "working set %.1f GB per GPU >> 126 MB L2" % (B * n_stages * 127e3 / 1e9)},
        "e2e": {"value": float(n_live) * args.steps / (e2e_ms * 1e-3), "unit": "instance-iterations/s", "h2d_bytes_per_step": B * 37 * 8,
                "d2h_bytes_per_step": B * 12 * 8, "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches), "roofline": roofline, "clocks": sampler.summary() if rank == 0 else None,
        "value_all_instances": value_all,
        "health": {"instances": int(B) * world, "live": int(n_live), "nan": int(B) * world - int(n_live),
                   "rank0_converged_kkt_below_1e-6": int((kkt[live] < 1e-6).sum()),
                   "rank0_kkt_median_live": float(np.median(kkt[live])) if live.any() else None,
                   "iterations_run": int(args.warmup + 2 * args.steps + 4),
                   "note": "value counts live instances only (finite KKT error after the run)"},
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cval, cores, sample, _ = anymal_oracle_throughput(args.workload, args.cpu_seconds)
        line["cpu_baseline"] = {"value": cval, "unit": "instance-iterations/s", "cores": cores, "kind": "port", "sample": sample}
    if rank == 0:
        emit_line(line)
    if world > 1:
        dist.destroy_process_group()


def run_iiwa(args, rank, local_rank, world):
    """The iiwa14 workloads (IIWA_WORKLOADS): device-resident arm, end-to-end arm, convergence pattern, roofline, cpu_baseline."""
    import torch
    import torch.distributed as dist
    import idocp_b200 as I

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # NCCL prints its version banner to STDOUT at VERSION level; keep stdout to the one JSON line
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    w = IIWA_WORKLOADS[args.workload]
    unocp = w["solver"] == "unocp"
    lib = I.default_library()
    prob = workload_problem(args.workload, I, lib)
    N = int(prob.N)
    # weak scaling: every rank owns a full per-GPU batch; strong scaling: the workload's batch is split over the ranks
    B_total = args.batch if args.batch else w["batch"]
    strong = args.scaling == "strong"
    if strong and B_total % world:
        raise SystemExit("--scaling strong needs a batch divisible by the number of GPUs")
    B = B_total // world if strong else B_total
    q0, v0 = workload_states(args.workload, rank * B, B, list(prob.q_min), list(prob.q_max))
    solver = (I.UnOCPSolver if unocp else I.UnParNMPCSolver)(prob, B, device=local_rank)
    if args.no_pipelining and unocp:
        solver.setPipelining(False)
    solver.setSolution("q", q0)
    solver.setSolution("v", v0)
    if w["problem"] == "task":
        solver.setTaskReference(I.task_space_circle_ref, 0.0)
    if not unocp:
        solver.initBackwardCorrection(0.0)
    stream = torch.cuda.ExternalStream(solver.stream(), device=local_rank)
    q_dev = torch.from_numpy(q0).cuda(local_rank)
    v_dev = torch.from_numpy(v0).cuda(local_rank)
    q_pin = torch.from_numpy(q0).pin_memory()
    v_pin = torch.from_numpy(v0).pin_memory()
    u_pin = torch.empty((B, NV), dtype=torch.float64).pin_memory()
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- device-resident arm -----------------------------------------------------------------
    for _ in range(args.warmup):
        solver.updateSolutionDevice(0.0, q_dev.data_ptr(), v_dev.data_ptr())
    solver.sync()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    solver.setProfiling(True)
    launches0 = solver.launchCount()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        solver.updateSolutionDevice(0.0, q_dev.data_ptr(), v_dev.data_ptr())
    e1.record(stream)
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = solver.launchCount() - launches0
    profile = solver.getProfile()
    solver.setProfiling(False)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {n: solver.getSolution(n) for n in ("q", "v", "a", "u", "lmd", "gmm", "beta")}, w["seed"])

    # ---- end-to-end arm: host buffers through the public API ----------------------------------
    q_host = q_pin.numpy()
    v_host = v_pin.numpy()
    u_host = u_pin.numpy()
    for _ in range(3):
        solver.updateSolution(0.0, q_host, v_host)
        solver.getStageSolution("u", 0, out=u_host)
    barrier()
    t0 = time.perf_counter()
    e0.record(stream)
    for _ in range(args.steps):
        solver.updateSolution(0.0, q_host, v_host)
        solver.getStageSolution("u", 0, out=u_host)
    e1.record(stream)
    barrier()
    e2e_wall_ms = (time.perf_counter() - t0) * 1e3
    e2e_ms = max_over_ranks(max(e0.elapsed_time(e1), e2e_wall_ms))
    if rank == 0:
        sampler.stop_flag = True
        sampler.join(timeout=2)

    # ---- secondary metric (SURVEY section 8d): the ocpbenchmarker::Convergence pattern --------------------------
    # (utils/ocp_benchmarker.hxx:37-51) = updateSolution + computeKKTResidual + KKTError every iteration, the KKT
    # errors of the batch read back to the host each time; device-resident x0, reported beside `value`, not in it
    conv_steps = max(1, min(args.steps, 50))
    barrier()
    e0.record(stream)
    for _ in range(conv_steps):
        solver.updateSolutionDevice(0.0, q_dev.data_ptr(), v_dev.data_ptr())
        solver.computeKKTResidualDevice(0.0, q_dev.data_ptr(), v_dev.data_ptr())
        solver.KKTError()
    e1.record(stream)
    barrier()
    conv_ms = max_over_ranks(e0.elapsed_time(e1))

    # sanity: the batch must have stayed numerically healthy
    solver.computeKKTResidualDevice(0.0, q_dev.data_ptr(), v_dev.data_ptr())
    kkt = solver.KKTError()
    status = solver.getStatus()

    units = float(B) * world * args.steps
    value = units / (ms_total * 1e-3)
    e2e_value = units / (e2e_ms * 1e-3)
    hbm_peak, peak_src = measured_peaks()
    _, fp64_sus, fp64_src = fp64_peak()
    counters, counters_src = load_kernel_counters(args.workload)
    # dominant kernel by measured device time
    stages = B * N
    algo = KERNEL_ALGO_DOUBLES_PER_STAGE if unocp else KERNEL_ALGO_DOUBLES_PER_STAGE_PARNMPC
    kern = {}
    for name, (ms, calls) in profile.items():
        if calls and name in algo:
            kern[name] = kernel_roofline(name, ms / calls, algo[name] * 8.0 * stages, counters,
                                         B == w["batch"], hbm_peak, fp64_sus)
            kern[name]["share"] = ms
        elif calls:
            kern[name] = {"ms_per_launch": ms / calls, "launches_per_step": calls / args.steps, "share": ms}
    tot = sum(k["share"] for k in kern.values()) or 1.0
    for k in kern.values():
        k["share"] = k["share"] / tot
    ranked = [n for n in kern if "algo_gbs" in kern[n]]
    dom = max(ranked, key=lambda n: kern[n]["ms_per_launch"]) if ranked else None
    roofline = None
    if dom:
        roofline = roofline_object(dom, kern, algo[dom] * 8.0 * stages, hbm_peak, peak_src, fp64_sus, fp64_src,
                                   counters_src,
                                   "per kernel: frac_hbm = algorithmic bytes / time / measured copy bandwidth, frac_fp64 = FP64 thread "
                                   "instructions counted by ncu for one launch at this batch (DFMA = 2 flop) / time / measured DFMA "
                                   "peak; `bound` = the larger.  FP64 has no tensor-core path at 7x7 (DESIGN.md section 4)")
        fl = sum(counters[n]["fp64_flop_executed"] for n in kern if n in counters and "fp64_flop_executed" in counters[n])
        if args.workload == "iiwa14_unocp":
            roofline["step_hbm_frac_algorithmic"] = BYTES_PER_UNIT * value / world / 1e9 / hbm_peak
            roofline["step_fp64_tflops_algorithmic"] = FLOP_PER_UNIT * value / world / 1e12
        if fl and B == w["batch"]:
            roofline["step_fp64_tflops_executed"] = fl / (ms_total / args.steps * 1e-3) / 1e12
            roofline["step_frac_fp64_executed"] = roofline["step_fp64_tflops_executed"] / fp64_sus
            roofline["step_dram_bytes_ncu"] = sum(counters[n].get("dram_bytes", 0.0) for n in kern if n in counters)

    line = {
        "metric": iiwa_metric(args.workload), "value": value, "unit": "instance-iterations/s",
        "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
        "us_per_iteration": ms_total / args.steps * 1e3,
        "higher_is_better": True, "scaling": args.scaling, "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "%s, %d random initial states per GPU (splitmix64 seed %d), line_search=false"
                               % (w["what"], B, w["seed"]),
                   "batch_per_gpu": B, "batch_total": B * world, "horizon": N,
                   "parallelism": "batch-sharded x%d, no collective" % world,
                   "l2_policy": "working set %.1f GB per GPU >> 126 MB L2 (inputs larger than L2)"
                                % (B * N * (22.5e3 if unocp else 81e3 / 4) / 1e9)},
        "e2e": {"value": e2e_value, "unit": "instance-iterations/s", "h2d_bytes_per_step": 2 * B * NV * 8,
                "d2h_bytes_per_step": B * NV * 8, "ms_per_step": e2e_ms / args.steps},
        "gpu_launches": int(launches),
        "convergence_pattern": {"value": float(B) * world * conv_steps / (conv_ms * 1e-3), "unit": "instance-iterations/s",
                                "ms_per_step": conv_ms / conv_steps, "steps": conv_steps,
                                "what": "updateSolution + computeKKTResidual + KKTError (errors read back) per iteration"},
        "roofline": roofline,
        "clocks": sampler.summary() if rank == 0 else None,
        "health": {"kkt_max": float(np.nanmax(kkt)), "kkt_median": float(np.nanmedian(kkt)), "kkt_nan": int(np.isnan(kkt).sum()),
                   "status_nonzero": int((status != 0).sum()), "converged_kkt_below_1e-6": int((kkt < 1e-6).sum()),
                   "iterations_run": int(args.warmup + 2 * args.steps + 3 + conv_steps)},
    }
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cval, cores, sample, _ = oracle_throughput(args.cpu_seconds, args.workload)
        line["cpu_baseline"] = {"value": cval, "unit": "instance-iterations/s", "cores": cores, "kind": "port",
                                "sample": sample}
    if rank == 0:
        emit_line(line)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="instances per GPU (total with --scaling strong); 0 = the workload's own")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="weak: every GPU owns a full batch (default, the driver's 1-8 GPU run); strong: BASELINE configs[2] "
                         "taken literally, 16384 instances in total split over the GPUs")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-pipelining", action="store_true",
                    help="UnOCPSolver: the literal linearise / Riccati / expand / update sequence (A/B of k_update_linearize)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--workload", default="iiwa14_unocp", choices=list(IIWA_WORKLOADS) + ["anymal_trotting", "anymal_running"],
                    help="iiwa14_unocp = BASELINE configs[2] (the headline); iiwa14_unocp_config / iiwa14_unparnmpc_task = "
                         "configs[0] / configs[1]; anymal_* = configs[3] / configs[4]")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the solution of the last one (rank 0's instances) as DIR/<field>.npy, "
                         "float64; beyond 64 MB in all, a fixed seeded sample of the instances")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes what the GPU solver computed; it needs --impl b200")
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.warmup < 3:
        args.warmup = 3

    if args.workload not in IIWA_WORKLOADS:
        if args.impl == "reference":
            run_reference_anymal(args, rank)
        else:
            run_anymal(args, rank, local_rank, world)
    elif args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_iiwa(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
