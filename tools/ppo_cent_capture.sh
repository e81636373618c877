#!/bin/sh
# The CENT family's PPO update on the hand-written kernels (--fused 1) against torch autograd (--fused 0) on one GPU: ppo_bench
# rounds alternated, two runs each, at C1 (1024 envs), the C3 shape (128 envs) and C5 (32 envs), then the kernel times of the wide
# layers.  Writes $OUT/ppo_cent.jsonl and $OUT/ppo_cent_kernels.jsonl.
set -e
OUT=${1:-ppo_cent_out}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader > "$OUT/gpu.txt"
: > "$OUT/ppo_cent.jsonl"
for cfg in "c1 1024" "c3 128" "c5 32"; do
  set -- $cfg
  for rep in 1 2; do
    for fused in 0 1; do
      python tools/ppo_bench.py --kind cent --config "$1" --envs "$2" --epochs 3 --mini-epochs 2 --minibatches 3 --fused $fused >> "$OUT/ppo_cent.jsonl"
    done
  done
done
: > "$OUT/ppo_cent_kernels.jsonl"
for cfg in "c1 1024" "c3 128" "c5 32"; do
  set -- $cfg
  python tools/ppo_cent_kernels.py --config "$1" --envs "$2" --minibatches 3 >> "$OUT/ppo_cent_kernels.jsonl"
done
