#!/bin/bash
# short 8-GPU session (one box with 8 GPUs): 1-GPU reference, sharded parity, weak scaling, configs[3] strong scaling
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
N="${1:-8}"
port=29900
OUT=gpurun_out/multi8_timing_g$N.log
: > $OUT
echo "## single GPU reference on this box: configs[1]" >> $OUT
timeout 200 python bench.py --quick --steps 10 --warmup 3 2>&1 | grep -E "quick|rror" | cut -c1-100 >> $OUT
run() { port=$((port + 1)); env "${@:2}" timeout "$1" python -m torch.distributed.run --nnodes=1 --nproc-per-node $N --master-addr 127.0.0.1 --master-port $port "${CMD[@]}"; }
CMD=(tests/multigpu/check_sharded_update.py)
run 400 X=1 > gpurun_out/multigpu_parity_g${N}.log 2>&1
echo "exit $?" >> gpurun_out/multigpu_parity_g${N}.log
echo "## parity at $N GPUs" >> $OUT
grep -E "^\[(small|wide)|MULTIGPU|^exit|MinppoError" gpurun_out/multigpu_parity_g${N}.log | cut -c1-400 | tail -n 4 >> $OUT
CMD=(bench.py --gpus $N --quick --steps 10 --warmup 3)
echo "## weak (configs[1] per GPU)" >> $OUT
run 300 X=1 2>&1 | grep -E "quick|rror" | cut -c1-140 >> $OUT
CMD=(bench.py --gpus $N --quick --steps 10 --warmup 3 --workload c4)
echo "## strong (configs[3]: 16384 x 64 global)" >> $OUT
run 300 X=1 2>&1 | grep -E "quick|rror" | cut -c1-140 >> $OUT
cat $OUT
