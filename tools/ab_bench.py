#!/usr/bin/env python
"""Alternating A/B timing of two builds of the library with bench.py, on one GPU in one session.

  tools/ab_bench.py --lib parent=build/ab/libidocp_b200_parent.so --lib new=idocp_b200/libidocp_b200.so \\
      --rounds 5 --out results.json -- --steps 200 --warmup 20 --no-cpu-baseline

Runs bench.py once per library per round, in the order A B A B ... so that clock and neighbour drift hit both sides
alike, and reports the median and the min..max spread of ms_per_step and of every kernel's ms_per_launch for each
library, and of e2e.ms_per_step (the same steps through the host API, with its host <-> device copies) where
bench.py reports it.  The GPU's name, power limit and maximum SM clock are read with nvidia-smi in the same session and
stored with the numbers.  Arguments after `--` go to bench.py unchanged.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(lib, bench_args):
    env = dict(os.environ, IDOCP_B200_LIBRARY=os.path.abspath(lib))
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + bench_args, env=env, cwd=ROOT,
                         capture_output=True, text=True)
    if res.returncode != 0:
        raise SystemExit("bench.py failed for %s:\n%s" % (lib, res.stderr[-3000:]))
    return json.loads(res.stdout.strip().splitlines()[-1])


def spread(xs):
    return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "runs": xs}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", required=True, help="tag=path of a library build (two or more)")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", default=None, help="write the summary JSON here as well")
    ap.add_argument("bench_args", nargs=argparse.REMAINDER)
    a = ap.parse_args()
    libs = [tuple(s.split("=", 1)) for s in a.lib]
    bench_args = [x for x in a.bench_args if x != "--"]
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    step = {t: [] for t, _ in libs}
    e2e = {t: [] for t, _ in libs}
    kern = {t: {} for t, _ in libs}
    for r in range(a.rounds):
        for t, path in libs:
            d = run_bench(path, bench_args)
            step[t].append(d["ms_per_step"])
            if "ms_per_step" in (d.get("e2e") or {}):
                e2e[t].append(d["e2e"]["ms_per_step"])
            for name, k in ((d.get("roofline") or {}).get("kernels") or {}).items():
                # the ANYmal lines give some kernels only per-step figures
                ms = k["ms_per_launch"] if "ms_per_launch" in k else k["ms_per_step"] / k["launches_per_step"]
                kern[t].setdefault(name, []).append(ms)
            print("round %d %-8s ms_per_step %.4f  e2e %s  %s" % (r, t, d["ms_per_step"], e2e[t][-1] if e2e[t] else None,
                  {n: round(v[-1], 4) for n, v in kern[t].items()}), flush=True)
    summary = {"gpu": smi, "bench_args": bench_args, "rounds": a.rounds,
               "libraries": {t: {"ms_per_step": spread(step[t]),
                                 "e2e_ms_per_step": spread(e2e[t]) if e2e[t] else None, "kernels": {n: spread(v) for n, v in kern[t].items()}}
                             for t, _ in libs}}
    text = json.dumps(summary)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
