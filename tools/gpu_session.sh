#!/bin/bash
# One gpurun call of the round: tests, peaks, bench lines, launch list, ncu captures.  Everything lands in gpurun_out/.
#   gpurun --timeout 1500 -- 'bash tools/gpu_session.sh <label> [steps...]'     steps: test peak bench ref anymal running launches ncu ncufb
L=$1; shift
STEPS=${*:-test peak bench ref anymal launches ncu}
mkdir -p gpurun_out/profiles
has() { [[ " $STEPS " == *" $1 "* ]]; }
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,power.draw --format=csv > gpurun_out/${L}_smi.txt 2>&1
if has peak; then
  tools/fp64_peak > gpurun_out/${L}_fp64_peak.json 2> gpurun_out/${L}_fp64_peak.err && cp gpurun_out/${L}_fp64_peak.json profiles/fp64_peak.json
  cat gpurun_out/${L}_fp64_peak.json
fi
if has test; then
  timeout 1500 python -m pytest tests -m gpu -x -q --durations=12 > gpurun_out/${L}_pytest.log 2>&1; echo "pytest rc=$?"; tail -n 25 gpurun_out/${L}_pytest.log
fi
if has bench; then
  python bench.py --steps 100 --warmup 10 > gpurun_out/${L}_bench.json 2> gpurun_out/${L}_bench.err; echo "bench rc=$?"; cut -c 1-600 gpurun_out/${L}_bench.json
fi
if has benchab; then
  python bench.py --steps 100 --warmup 10 --no-pipelining --no-cpu-baseline > gpurun_out/${L}_bench_nopipe.json 2> gpurun_out/${L}_bench_nopipe.err; cut -c 1-300 gpurun_out/${L}_bench_nopipe.json
fi
if has testfast; then
  timeout 900 python -m pytest tests/test_gpu_parity.py tests/test_gpu_baseline_configs.py::test_config2_full_batch_bit_exact_and_iteration_gate -m gpu -x -q > gpurun_out/${L}_pytest_fast.log 2>&1; echo "pytest rc=$?"; tail -n 5 gpurun_out/${L}_pytest_fast.log
fi
if has ref; then
  python bench.py --impl reference --steps 20 --warmup 3 > gpurun_out/${L}_bench_reference.json 2> gpurun_out/${L}_bench_reference.err; cut -c 1-300 gpurun_out/${L}_bench_reference.json
fi
if has anymal; then
  python bench.py --workload anymal_trotting --steps 20 --warmup 5 > gpurun_out/${L}_bench_anymal_trotting.json 2> gpurun_out/${L}_bench_anymal_trotting.err; cut -c 1-400 gpurun_out/${L}_bench_anymal_trotting.json
fi
if has running; then
  python bench.py --workload anymal_running --steps 10 --warmup 3 > gpurun_out/${L}_bench_anymal_running.json 2> gpurun_out/${L}_bench_anymal_running.err; cut -c 1-400 gpurun_out/${L}_bench_anymal_running.json
fi
if has dmma; then
  tools/dmma_probe > gpurun_out/${L}_dmma_probe.json 2> gpurun_out/${L}_dmma_probe.err; cat gpurun_out/${L}_dmma_probe.json
fi
if has configs01; then
  python bench.py --workload iiwa14_unparnmpc_task --steps 20 --warmup 5 > gpurun_out/${L}_bench_iiwa14_unparnmpc_task.json 2> gpurun_out/${L}_bench_iiwa14_unparnmpc_task.err; echo "unparnmpc_task rc=$?"; cut -c 1-500 gpurun_out/${L}_bench_iiwa14_unparnmpc_task.json
  python bench.py --workload iiwa14_unocp_config --steps 50 --warmup 5 > gpurun_out/${L}_bench_iiwa14_unocp_config.json 2> gpurun_out/${L}_bench_iiwa14_unocp_config.err; echo "unocp_config rc=$?"; cut -c 1-500 gpurun_out/${L}_bench_iiwa14_unocp_config.json
fi
if has testnew; then
  timeout 900 python -m pytest tests/test_sharded_solver.py tests/test_cpp_host.py tests/test_gpu_parity.py -m gpu -x -q > gpurun_out/${L}_pytest_new.log 2>&1; echo "pytest rc=$?"; tail -n 5 gpurun_out/${L}_pytest_new.log
fi
if has ncuparnmpc; then
  NCU_SKIP=5 NCU_COUNT=2 tools/ncu_capture.sh $L iiwa14_unparnmpc_task 'k_parnmpc_invert'
fi
if has parnmpc; then
  python tools/bench_solver.py --solver unparnmpc --batch 16384 --steps 20 > gpurun_out/${L}_bench_solver_unparnmpc.json 2> gpurun_out/${L}_bench_solver_unparnmpc.err; cut -c 1-700 gpurun_out/${L}_bench_solver_unparnmpc.json
fi
if has variants; then   # A/B builds from tools/build_variant.py: VARIANT_WORKLOAD (default iiwa14_unocp), VARIANT_STEPS
  for so in build/variants/*.so; do
    tag=$(basename $so .so); tag=${tag#libidocp_b200_}
    IDOCP_B200_LIBRARY=$PWD/$so python bench.py --workload ${VARIANT_WORKLOAD:-iiwa14_unocp} --steps ${VARIANT_STEPS:-100} --warmup 10 --no-cpu-baseline ${VARIANT_ARGS:-} \
        > gpurun_out/${L}_variant_${tag}.json 2> gpurun_out/${L}_variant_${tag}.err
    python - "$tag" gpurun_out/${L}_variant_${tag}.json <<'PY'
import json, sys
try:
    d = json.loads(open(sys.argv[2]).read().strip().splitlines()[-1])
    print("variant", sys.argv[1], "ms_per_step", round(d["ms_per_step"], 4), {k: round(v["ms_per_launch"], 4) for k, v in d["roofline"]["kernels"].items()}, "kkt_max", d["health"]["kkt_max"])
except Exception as e:
    print("variant", sys.argv[1], "FAILED", e)
PY
  done
fi
if has scale; then   # multi-GPU call (gpurun --gpus 8): strong scaling of configs[2] / [3], configs[4] at its definition (8 x 1024)
  tr() { n=$1; shift; python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port $((29500 + n)) bench.py --gpus $n "$@"; }
  for n in ${SCALE_NS:-2 4 8}; do
    tr $n --scaling strong --steps 100 --warmup 10 > gpurun_out/${L}_scale_strong_iiwa14_unocp_n$n.json 2> gpurun_out/${L}_scale_strong_iiwa14_unocp_n$n.err
    cut -c 1-330 gpurun_out/${L}_scale_strong_iiwa14_unocp_n$n.json
  done
  n=${SCALE_NMAX:-8}
  tr $n --workload anymal_trotting --scaling strong --steps 20 --warmup 5 > gpurun_out/${L}_scale_strong_anymal_trotting_n$n.json 2> gpurun_out/${L}_scale_strong_anymal_trotting_n$n.err
  cut -c 1-330 gpurun_out/${L}_scale_strong_anymal_trotting_n$n.json
  tr $n --workload anymal_running --steps 10 --warmup 3 > gpurun_out/${L}_scale_anymal_running_n$n.json 2> gpurun_out/${L}_scale_anymal_running_n$n.err
  cut -c 1-330 gpurun_out/${L}_scale_anymal_running_n$n.json
fi
if has sanitize; then   # compute-sanitizer over small runs of every solver path (tools/sanitize_run.py), all four tools
  out=gpurun_out/${L}_compute_sanitizer.txt
  echo "# compute-sanitizer over tools/sanitize_run.py all (label $L)" > $out
  for tool in memcheck racecheck synccheck initcheck; do
    echo "== $tool" >> $out
    timeout 1500 compute-sanitizer --tool $tool python tools/sanitize_run.py all > gpurun_out/${L}_sanitize_$tool.log 2>&1
    grep -E "ERROR SUMMARY|RACECHECK SUMMARY" gpurun_out/${L}_sanitize_$tool.log >> $out || echo "(no summary line: see ${L}_sanitize_$tool.log)" >> $out
  done
  cat $out
fi
if has launches; then
  ncu --metrics gpu__time_duration.sum --clock-control none -s 40 -c 200 --csv --log-file gpurun_out/${L}_launches.csv \
      python bench.py --steps 20 --warmup 3 --no-cpu-baseline > gpurun_out/${L}_launches_run.log 2>&1; echo "launches rc=$?"
fi
if has ncu; then
  NCU_SKIP=40 NCU_COUNT=6 KEEP_REP=1 tools/ncu_capture.sh $L iiwa14_unocp 'k_linearize|k_riccati|k_expand|k_update'
fi
if has ncufb; then
  NCU_SKIP=30 NCU_COUNT=6 tools/ncu_capture.sh $L anymal_trotting 'k_fb_robot|k_fb_condense|k_fb_riccati_backward'
fi
echo "session $L done"
