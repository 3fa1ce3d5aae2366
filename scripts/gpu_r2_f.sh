#!/bin/bash
mkdir -p gpurun_out
timeout 600 python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-bf16 --no-sample > gpurun_out/bench_persist.log 2>&1
python -c "import json;d=json.loads(open('gpurun_out/bench_persist.log').read().strip().splitlines()[-1]);print('persist   ', d['ms_per_step'], d['e2e']['ms_per_step'], d['gpu_launches'])"
timeout 1500 python -m pytest tests -m gpu -q --timeout 600 -x > gpurun_out/pytest_gpu.log 2>&1
echo "pytest exit $?" >> gpurun_out/pytest_gpu.log
grep -E 'passed|failed|FAILED|ERROR|assert|Error' gpurun_out/pytest_gpu.log | tail -20
