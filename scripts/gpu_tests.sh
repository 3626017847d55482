#!/bin/bash
# Runs the GPU parity suite in separate processes (a hung kernel in one group must not take the others down).
# usage: scripts/gpu_tests.sh [outdir]
OUT=${1:-gpurun_out}
mkdir -p $OUT
nvidia-smi --query-gpu=name,driver_version,memory.total --format=csv > $OUT/gpu.txt 2>&1
run() { # name, timeout, args...
  local name=$1; local to=$2; shift 2
  echo "=== $name" | tee -a $OUT/summary.txt
  timeout -k 10 $to python -m pytest "$@" -q -rP -m gpu -x --no-header -p no:cacheprovider > $OUT/$name.log 2>&1
  echo "exit $?: $(tail -1 $OUT/$name.log)" | tee -a $OUT/summary.txt
}
runall() { # same but without -x
  local name=$1; local to=$2; shift 2
  echo "=== $name" | tee -a $OUT/summary.txt
  timeout -k 10 $to python -m pytest "$@" -q -rP -m gpu --no-header -p no:cacheprovider > $OUT/$name.log 2>&1
  echo "exit $?: $(tail -1 $OUT/$name.log)" | tee -a $OUT/summary.txt
}
: > $OUT/summary.txt
runall kernels 900 tests/test_gpu_kernels.py
runall models 900 tests/test_gpu_models.py
runall aten_rng 600 tests/test_gpu_aten_rng.py
runall full_config 900 tests/test_gpu_full_config.py
runall fused_tail 600 tests/test_gpu_fused_tail.py
runall attention_edges 600 tests/test_gpu_attention_edges.py
cat $OUT/summary.txt
