#!/bin/bash
mkdir -p gpurun_out
nvidia-smi --query-gpu=index,name --format=csv
timeout 900 python -m pytest tests/test_gpu_dp2.py -m gpu -q --timeout 600 > gpurun_out/pytest_dp2.log 2>&1
grep -E 'passed|failed|skipped|FAILED|ERROR|assert|Error' gpurun_out/pytest_dp2.log | tail -8
timeout 600 python bench.py --steps 20 --warmup 5 --no-cpu-baseline --no-bf16 --no-sample > gpurun_out/bench_1gpu.log 2>&1
python -c "import json;d=json.loads(open('gpurun_out/bench_1gpu.log').read().strip().splitlines()[-1]);print('1 GPU ms/step', d['ms_per_step'])"
