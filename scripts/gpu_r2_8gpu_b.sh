#!/bin/bash
# 8-GPU experiments: NCCL CTA budget for the overlapped gradient bucket, and the wide variant (configs[4]) on 8 GPUs
mkdir -p gpurun_out
run() {  # name, env..., -- bench args
  local name=$1; shift
  local envs=()
  while [ "$1" != "--" ]; do envs+=("$1"); shift; done
  shift
  env "${envs[@]}" timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 --master-addr 127.0.0.1 --master-port 29531 bench.py --gpus 8 "$@" > gpurun_out/b8_$name.log 2>&1
  python - <<PY
import json
try:
    d=json.loads([l for l in open('gpurun_out/b8_$name.log') if l.startswith('{')][-1])
    print('$name: ms/step', round(d['ms_per_step'],3), 'value', round(d['value']), 'e2e', round(d['e2e']['value']))
except Exception as e:
    print('$name: FAILED', e)
PY
}
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline --no-bf16 --no-sample > gpurun_out/b8_n1.log 2>&1
python -c "import json;d=json.loads([l for l in open('gpurun_out/b8_n1.log') if l.startswith('{')][-1]);print('N=1 ms/step', d['ms_per_step'])"
run default NCCL_DEBUG=INFO -- --steps 20 --warmup 5 --no-cpu-baseline --no-bf16 --no-sample
grep -o "NVLS[^ ]*\|Using network[^,]*\|[0-9]* coll channels[^,]*\|Connected all [a-z]*" gpurun_out/b8_default.log | sort | uniq -c | head -8
run cta4 NCCL_MAX_CTAS=4 -- --steps 20 --warmup 5 --no-cpu-baseline --no-bf16 --no-sample
run cta16 NCCL_MAX_CTAS=16 -- --steps 20 --warmup 5 --no-cpu-baseline --no-bf16 --no-sample
run ring NCCL_ALGO=Ring -- --steps 20 --warmup 5 --no-cpu-baseline --no-bf16 --no-sample
run widelstm -- --variant wide-lstm --gemm bf16 --steps 10 --warmup 3 --no-cpu-baseline --no-bf16 --no-sample
run widegru -- --variant wide-gru --gemm bf16 --steps 10 --warmup 3 --no-cpu-baseline --no-bf16 --no-sample
cp gpurun_out/b8_widelstm.log gpurun_out/b8_widelstm_line.json 2>/dev/null
