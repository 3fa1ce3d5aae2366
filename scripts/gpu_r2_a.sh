#!/bin/bash
# round 2, visit A: the new persistent encoder first (fast feedback), then the existing suites, smoke, a short bench
mkdir -p gpurun_out
nvidia-smi --query-gpu=name,clocks.sm,clocks.max.sm,memory.total --format=csv > gpurun_out/gpu.txt 2>&1
timeout 600 python -m pytest tests/test_gpu_paths.py -m gpu -q --timeout 300 -k "persistent_encoder" -x > gpurun_out/pytest_enc.log 2>&1
echo "pytest enc exit $?" >> gpurun_out/pytest_enc.log
grep -E 'passed|failed|FAILED|ERROR|assert|Error|timed out' gpurun_out/pytest_enc.log | tail -20
timeout 1500 python -m pytest tests -m gpu -q --timeout 600 --deselect tests/test_gpu_pinned.py -k "not persistent_encoder" > gpurun_out/pytest_gpu.log 2>&1
echo "pytest exit $?" >> gpurun_out/pytest_gpu.log
grep -E 'passed|failed|FAILED|ERROR|assert|Error' gpurun_out/pytest_gpu.log | tail -30
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1
echo "smoke exit $?" >> gpurun_out/smoke.log
tail -5 gpurun_out/smoke.log
timeout 600 python bench.py --steps 10 --warmup 3 --no-cpu-baseline --no-bf16 > gpurun_out/bench.log 2>&1
echo "bench exit $?" >> gpurun_out/bench.log
tail -3 gpurun_out/bench.log
