#!/bin/bash
mkdir -p gpurun_out; cd "$(dirname "$0")/.."
timeout 300 python -m pytest tests/test_gpu_ops.py -q -m gpu -k "f16x3" > gpurun_out/ops_f16.log 2>&1; echo "ops_f16 exit $?"; grep -E "^E +assert|passed|failed|Error" gpurun_out/ops_f16.log | head -20 | cut -c1-300
timeout 400 python -m pytest tests/test_gpu_slice_loop.py -q -m gpu -s -k "f16x3" > gpurun_out/loop_f16.log 2>&1; echo "loop_f16 exit $?"; grep -E "^\[|passed|failed|^E +assert" gpurun_out/loop_f16.log | cut -c1-300
timeout 300 python bench.py --math f16x3 --no-cpu-baseline > gpurun_out/bench_f16.log 2>&1; echo "bench exit $?"; python - <<'PY'
import json
try:
    l=[x for x in open('gpurun_out/bench_f16.log') if x.startswith('{')][-1]; d=json.loads(l)
    print('f16 bench', round(d['value']), round(d['ms_per_step'],2), 'e2e', round(d['e2e']['value']), {k:(round(v['ms_per_step'],2), v['launches_per_step']) for k,v in d['kernel_families'].items()}, d['clocks'])
except Exception as e: print('no bench line', e); print(open('gpurun_out/bench_f16.log').read()[-1500:])
PY
