#!/bin/bash
# Static FP64 issue-cost estimate of the rollout fast path (sincos resync removed, rotation tier TIER=0|1 only where n has two tiers) for n in "$@".
# usage: tools/fastpath_mix.sh 3 5 10
set -e
ROOT=$(cd "$(dirname "$0")/.." && pwd)
SRC=$ROOT/safe-exploration-with-simulator-in-rl-algorithms_b200/csrc
mkdir -p /tmp/fastpath
for n in "$@"; do
  nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -DSWM_ANALYZE_TIER=${TIER:-0} ${EXTRA_DEFS} -c $SRC/rollout_n$n.cu -o /tmp/fastpath/n$n.o &
done
wait
for n in "$@"; do
  for pat in "Li${n}ELi0ELi0ELb0ELb0ELi0E" "Li${n}ELi0ELi[123]ELb1ELb1ELi0E"; do
    python $ROOT/tools/sass_mix.py /tmp/fastpath/n$n.o "$pat" | grep -E "^==|loop|reuse|DFMA|DMUL|DADD|UMOV|IMAD|LDS|STS" 
  done
done
