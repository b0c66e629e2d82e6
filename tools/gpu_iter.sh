#!/bin/bash
# Quick iteration check: kernel 3 + f16x3 ops + f16x3 slice loop + bench, each in its own process.
#   gpurun --timeout 1200 -- bash tools/gpu_iter.sh
mkdir -p gpurun_out
cd "$(dirname "$0")/.."
run() { local name=$1 t=$2; shift 2
  echo "=== $name" | tee -a gpurun_out/iter_summary.txt
  timeout $t "$@" > gpurun_out/$name.log 2>&1
  echo "exit $?" | tee -a gpurun_out/iter_summary.txt
  tail -n 5 gpurun_out/$name.log | cut -c1-1800 | tee -a gpurun_out/iter_summary.txt
}
: > gpurun_out/iter_summary.txt
run it_gc    300 python -m pytest tests/test_gpu_gc.py -q -x -m gpu
run it_ops   600 python -m pytest tests/test_gpu_ops.py -q -m gpu
run it_loop  900 python -m pytest tests/test_gpu_slice_loop.py -q -m gpu
run it_bench 600 python bench.py --no-cpu-baseline
run it_bench1 600 python bench.py --no-cpu-baseline --lanes 1
run it_layers 300 python tools/layer_times.py
exit 0
