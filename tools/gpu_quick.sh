#!/bin/bash
# quick check: GPU tests, temporal-conv phase timers, both benches
cd "${GRAFT_REPO_ROOT:-/root/repo}"
mkdir -p gpurun_out
rm -f gpurun_out/summary.txt
run() { name=$1; shift; timeout $1 "${@:2}" > gpurun_out/$name.log 2>&1; echo "$name rc=$?" >> gpurun_out/summary.txt; }
run pytest_gpu 1500 python -m pytest tests -m gpu -x -q
run trace_tcn 300 bash tools/gpu_trace_tcn.sh
run bench_auto 900 python bench.py --steps 200 --warmup 8 --no-cpu-baseline
run bench_auto_mod 900 python bench.py --workload cost_gcn_mod --steps 100 --warmup 8 --no-cpu-baseline
cat gpurun_out/summary.txt; tail -3 gpurun_out/pytest_gpu.log | cut -c1-200; cat gpurun_out/trace_tcn.log
