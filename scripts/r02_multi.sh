#!/bin/bash
# round 2 multi-GPU session (one box with N GPUs): sharded parity, weak-scaling and
# configs[3] strong-scaling timings, full bench lines.  Usage: bash scripts/r02_multi.sh N [full]
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
N="${1:-2}"
port=29800
echo "## single GPU reference on this box: configs[1], configs[3]"
timeout 200 python bench.py --quick --steps 10 --warmup 3 2>&1 | grep -E "quick|rror" | cut -c1-100
timeout 200 python bench.py --quick --steps 10 --warmup 3 --workload c4 2>&1 | grep -E "quick|rror" | cut -c1-100
run() { port=$((port + 1)); env "${@:2}" timeout "$1" python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port $port "${CMD[@]}"; }
CMD=(tests/multigpu/check_sharded_update.py)
for cfg in "X=default" $PARITY_EXTRA; do
  run 400 $cfg > gpurun_out/multigpu_parity_g${N}_${cfg#*=}.log 2>&1
  echo "exit $?" >> gpurun_out/multigpu_parity_g${N}_${cfg#*=}.log
  echo "## parity at $N GPUs, $cfg"
  grep -E "^\[(small|wide)|MULTIGPU|^exit|MinppoError" gpurun_out/multigpu_parity_g${N}_${cfg#*=}.log | cut -c1-700 | tail -n 4
done
OUT=gpurun_out/multi_timing_g$N.log
: > $OUT
CMD=(bench.py --gpus $N --quick --steps 10 --warmup 3)
for cfg in "X=default" $EXTRA_ABLATE; do
  echo "## weak (configs[1] per GPU) $cfg" >> $OUT
  run 300 $cfg 2>&1 | grep -E "quick|rror" | cut -c1-140 >> $OUT
done
CMD=(bench.py --gpus $N --quick --steps 10 --warmup 3 --workload c4)
for cfg in "X=default" $EXTRA_ABLATE; do
  echo "## strong (configs[3]: 16384 x 64 global) $cfg" >> $OUT
  run 300 $cfg 2>&1 | grep -E "quick|rror" | cut -c1-140 >> $OUT
done
cat $OUT
if [ "$2" == "full" ]; then
  for wl in auto c4; do
    CMD=(bench.py --gpus $N --steps 10 --warmup 3 --workload $wl)
    run 600 X=1 > gpurun_out/bench_${wl}_g$N.log 2>&1
    echo "exit $?" >> gpurun_out/bench_${wl}_g$N.log
    grep -E "^\{" gpurun_out/bench_${wl}_g$N.log | python -c "
import json,sys
for l in sys.stdin:
    d=json.loads(l); print('bench $wl $N GPUs: ms_per_step', round(d['ms_per_step'],3), 'value', round(d['value']), 'e2e', round(d['e2e']['value']), d['scaling'])"
  done
fi
