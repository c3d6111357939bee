#!/bin/bash
# Short multi-GPU session (gpurun --gpus N): parity with the default exchange, graph-replay timings, full bench line.
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
N="${1:-4}"
port=29800
timeout 400 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 \
  --master-port $port tests/multigpu/check_sharded_update.py > gpurun_out/multigpu_parity_g${N}.log 2>&1
echo "exit $?" >> gpurun_out/multigpu_parity_g${N}.log
grep -E "^\[(small|wide)|MULTIGPU|^exit|MinppoError" gpurun_out/multigpu_parity_g${N}.log | cut -c1-400 | tail -n 4
OUT=gpurun_out/multi_timing_g$N.log
: > $OUT
for cfg in $TIMING_CFGS; do   # e.g. TIMING_CFGS="MINPPO_PX_TWO_PHASE=0 MINPPO_NCCL_ALLREDUCE=1"
  port=$((port + 1))
  echo "## $cfg" >> $OUT
  env $cfg timeout 300 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 \
    --master-port $port bench.py --gpus $N --quick --steps 10 --warmup 3 2>&1 | grep -E "quick|rror" | cut -c1-120 >> $OUT
done
cat $OUT
port=$((port + 1))
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 \
  --master-port $port bench.py --gpus $N --steps 10 --warmup 3 > gpurun_out/bench_g$N.log 2>&1
echo "exit $?" >> gpurun_out/bench_g$N.log
python - <<PY
import json
for l in open('gpurun_out/bench_g$N.log'):
    if l.startswith('{'):
        d = json.loads(l)
        print('bench $N GPUs: ms_per_step', round(d['ms_per_step'], 3), 'value', round(d['value']), 'e2e', round(d['e2e']['value']))
        print({k: round(v['ms_per_update'], 3) for k, v in d['kernel_classes'].items() if v['ms_per_update'] > 0})
    elif 'rror' in l:
        print(l.rstrip()[:300])
PY
