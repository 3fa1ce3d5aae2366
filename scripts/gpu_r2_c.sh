#!/bin/bash
mkdir -p gpurun_out
timeout 900 python -m pytest tests/test_gpu_autograd_api.py -m gpu -q --timeout 300 > gpurun_out/pytest_autograd.log 2>&1
grep -E 'passed|failed|FAILED|ERROR|assert|Error' gpurun_out/pytest_autograd.log | tail -20
