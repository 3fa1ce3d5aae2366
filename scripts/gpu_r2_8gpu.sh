#!/bin/bash
mkdir -p gpurun_out
nvidia-smi --query-gpu=index,name --format=csv | head -3
timeout 600 python bench.py --gpus 1 --steps 20 --warmup 5 --no-cpu-baseline --no-bf16 > gpurun_out/bench8_n1.log 2>&1
python -c "import json;d=json.loads([l for l in open('gpurun_out/bench8_n1.log') if l.startswith('{')][-1]);print('N=1 ms/step', d['ms_per_step'], 'value', d['value'], 'sample', d['sample']['value'])"
for n in 2 4 8; do
timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port 2951$n bench.py --gpus $n --steps 20 --warmup 5 > gpurun_out/bench8_n$n.log 2>&1
python - <<PY
import json
d=json.loads([l for l in open('gpurun_out/bench8_n$n.log') if l.startswith('{')][-1])
print('N=$n ms/step', d['ms_per_step'], 'value', d['value'], 'e2e', d['e2e']['value'], 'sample', d.get('sample',{}).get('value'))
PY
done
