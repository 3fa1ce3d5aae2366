#!/bin/bash
mkdir -p gpurun_out
timeout 600 python -m pytest tests/test_gpu_paths.py -m gpu -q --timeout 300 -k "persistent_encoder" > gpurun_out/pytest_enc.log 2>&1
echo "pytest enc exit $?" >> gpurun_out/pytest_enc.log
grep -E 'passed|failed|FAILED|ERROR|assert|Error|timed out' gpurun_out/pytest_enc.log | tail -20
timeout 300 python scripts/step_phases.py > gpurun_out/phases.log 2>&1
sort gpurun_out/phases.log | uniq -c | sort -rn | awk '{$1="";print}' | sort -u | head -20
timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none --profile-from-start off --csv --log-file gpurun_out/launches.csv \
  python bench.py --ncu-step > gpurun_out/ncu_bench.log 2>&1
echo "ncu exit $?"
python scripts/ncu_summary.py gpurun_out/launches.csv > gpurun_out/launch_summary.txt 2>&1
head -16 gpurun_out/launch_summary.txt
timeout 1500 python -m pytest tests -m gpu -q --timeout 600 -k "not persistent_encoder" > gpurun_out/pytest_gpu.log 2>&1
echo "pytest exit $?" >> gpurun_out/pytest_gpu.log
grep -E 'passed|failed|FAILED|ERROR|assert|Error' gpurun_out/pytest_gpu.log | tail -40
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1
echo "smoke exit $?" >> gpurun_out/smoke.log
tail -3 gpurun_out/smoke.log
