#!/bin/bash
# One GPU session (single GPU): parity tests, smoke, fused-kernel cycle trace,
# full bench, ncu launch list and ncu --set full captures.  Everything lands in gpurun_out/.
# Usage: bash scripts/gpu_call.sh [tests] [trace] [bench] [ncu] [ncufull]   (default: all)
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
WHAT="${*:-tests trace bench ncu ncufull}"
has() { [[ " $WHAT " == *" $1 "* ]]; }
nvidia-smi > gpurun_out/nvidia_smi.txt 2>&1
nproc > gpurun_out/nproc.txt
if has tests; then
  for f in gae perm gemm update policy; do
    timeout 900 python -m pytest tests/test_gpu_$f.py -m gpu -q --timeout=600 -p no:cacheprovider > gpurun_out/pytest_$f.log 2>&1
    echo "exit $?" >> gpurun_out/pytest_$f.log
  done
  timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > gpurun_out/smoke.log 2>&1
  echo "exit $?" >> gpurun_out/smoke.log
  tail -n 3 gpurun_out/pytest_*.log gpurun_out/smoke.log
fi
if has trace; then
  timeout 600 python scripts/trace_fused.py > gpurun_out/trace_fused.log 2>&1
  echo "exit $?" >> gpurun_out/trace_fused.log
  tail -n 60 gpurun_out/trace_fused.log
fi
if has bench; then
  timeout 900 python bench.py --steps 10 --warmup 3 > gpurun_out/bench.log 2>&1
  echo "exit $?" >> gpurun_out/bench.log
  tail -c 3500 gpurun_out/bench.log
fi
if has ncu; then
  timeout 900 ncu --metrics gpu__time_duration.sum --clock-control none -s 200 -c 400 --csv \
    --log-file gpurun_out/launches.csv python bench.py --quick --steps 2 --warmup 3 > gpurun_out/ncu_bench.log 2>&1
  echo "exit $?" >> gpurun_out/ncu_bench.log
  python scripts/summarize_launches.py gpurun_out/launches.csv > gpurun_out/launches_summary.txt 2>&1
  cat gpurun_out/launches_summary.txt
fi
if has ncudw; then
  timeout 900 ncu --set full --clock-control none --import-source on -k regex:"dwopt_kernel" -s 20 -c 2 -f -o gpurun_out/prof_dwopt \
    python bench.py --quick --steps 1 --warmup 3 > gpurun_out/ncu_dwopt.log 2>&1
  echo "exit $?" >> gpurun_out/ncu_dwopt.log
  tail -n 2 gpurun_out/ncu_dwopt.log
fi
if has ncufull; then
  timeout 1500 ncu --set full --clock-control none --import-source on \
    -k regex:"umma_gemm_kernel|opt_kernel|fused_step_kernel" -s 40 -c 4 -f -o gpurun_out/prof_full \
    python bench.py --quick --steps 1 --warmup 3 > gpurun_out/ncu_full.log 2>&1
  echo "exit $?" >> gpurun_out/ncu_full.log
  tail -n 3 gpurun_out/ncu_full.log
  ls -la gpurun_out/*.ncu-rep
fi
