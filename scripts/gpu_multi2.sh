#!/bin/bash
# Multi-GPU call, short form: bench under torchrun (cfg3 only + the sharded cfg4 leg), config 5 with native clients.
tag=${1:-multi}; n=${2:-2}; scale=${3:-1.0}
mkdir -p gpurun_out
timeout 900 python -m torch.distributed.run --nnodes=1 --nproc-per-node $n --master-addr 127.0.0.1 --master-port 29571 \
  bench.py --gpus $n --steps 20 --warmup 5 --configs '' --no-cpu-baseline --sustain-s 0 > gpurun_out/${tag}_bench_n${n}.json 2> gpurun_out/${tag}_bench_n${n}.err
echo "bench rc=$?"; tail -3 gpurun_out/${tag}_bench_n${n}.err | cut -c1-300
python -c "
import json; b=json.load(open('gpurun_out/${tag}_bench_n${n}.json')); print('value', b['value'], 'e2e', b['e2e']['value']); print(json.dumps(b.get('configs',{}).get('cfg4_sharded'))[:1200])"
for sc in $scale; do
  timeout 900 python scripts/cfg5_replay.py --devices $n --clients 1000 --scale $sc --rounds 2 > gpurun_out/${tag}_cfg5_n${n}_s${sc}.json 2> gpurun_out/${tag}_cfg5_n${n}_s${sc}.err
  echo "cfg5 scale $sc rc=$?"; tail -3 gpurun_out/${tag}_cfg5_n${n}_s${sc}.err | cut -c1-300; cut -c1-1400 gpurun_out/${tag}_cfg5_n${n}_s${sc}.json
done
