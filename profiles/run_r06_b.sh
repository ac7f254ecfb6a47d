#!/bin/bash
# k_playout, one lane per game, with the tile draw and the stacking-mask pick on fewer ALU-pipe instructions: correctness
# first, then A/B of this tree's library against libharmonies_b200_parent.so (the previous commit's sources, built
# beforehand with build.py: nvcc needs no GPU) in one run.  Usage: bash profiles/run_r06_b.sh [output directory]
# Prints card/power limit, the playout tests, playout_ab.py alternated 6x at 65,536 games and 2x at 262,144 games per
# build, the byte comparison of bench.py --dump-outputs between the builds and bench.py's result line of each build.
set -u
OUT=${1:-${TMPDIR:-/tmp}/hz_profile}   # output directory (first argument)
mkdir -p "$OUT"
L=$PWD/harmonies_alphazero_b200
LIBS="default parent"
libpath() { if [ "$1" = default ]; then echo "$L/libharmonies_b200.so"; else echo "$L/libharmonies_b200_$1.so"; fi; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
timeout 900 python -m pytest -q -m gpu -p no:cacheprovider tests/test_gpu_playout_pick.py tests/test_gpu_playout_rounds.py \
  tests/test_gpu_engine.py tests/test_gpu_rollout_eval.py 2>&1 | tail -n 8
for i in 1 2 3 4 5 6; do
  for b in $LIBS; do HZ_LIB_PATH=$(libpath $b) timeout 300 python profiles/playout_ab.py 2>&1 | tail -n 2 | sed "s|^|$b 65536 run $i: |"; done
done
for i in 1 2; do
  for b in $LIBS; do HZ_LIB_PATH=$(libpath $b) timeout 300 python profiles/playout_ab.py 262144 2>&1 | tail -n 1 | sed "s|^|$b 262144 run $i: |"; done
done
for b in $LIBS; do
  HZ_LIB_PATH=$(libpath $b) timeout 600 python bench.py --no-mcts --no-cpu-baseline --no-python-reference \
    --dump-outputs "$OUT"/dump_$b > "$OUT"/dump_$b.json 2> "$OUT"/dump_$b.err; echo "dump $b rc=$?"
  for f in states steps total_steps; do cmp "$OUT"/dump_default/$f.npy "$OUT"/dump_$b/$f.npy && echo "$b: $f.npy identical to default"; done
done
rm -rf "$OUT"/dump_*/   # 64 MB each: the comparison above is the result
for b in $LIBS; do
  echo "bench $b:"; HZ_LIB_PATH=$(libpath $b) timeout 900 python bench.py --gpus 1 2> "$OUT"/bench_$b.err | tail -n 1
done
