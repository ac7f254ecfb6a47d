#!/bin/bash
# Round 6 of k_playout, two lanes per game (lane parity p plays board p; profiles/r06_pair_lanes.patch), measured against
# this tree's one-lane kernel and not merged.  Usage: bash profiles/run_r06_a.sh [output directory]
# PAIRS (default $TMPDIR/hz_pairs) is a copy of this tree with the patch applied and its library built; it is made here
# when missing (nvcc needs no GPU, so it can be made beforehand).  Prints card/power limit, the premise check (this tree's
# hz_playout_keys at 65,536 and 85,248 games, alternated 3x; 85,248 = one full wave at 9 blocks of 64 per SM), the
# playout tests on the two-lane build (with its own test file), playout_ab.py alternated 6x at 65,536 games and 2x at
# 262,144 games per build, the byte comparison of bench.py --dump-outputs between the builds and bench.py's result
# line of each build.
set -u
OUT=${1:-${TMPDIR:-/tmp}/hz_profile}   # output directory (first argument)
PAIRS=${PAIRS:-${TMPDIR:-/tmp}/hz_pairs}
mkdir -p "$OUT"
ROOT=$PWD
if [ ! -f "$PAIRS/harmonies_alphazero_b200/libharmonies_b200.so" ]; then
  rm -rf "$PAIRS" && mkdir -p "$PAIRS"
  tar -C "$ROOT" --exclude=./.git --exclude=./build --exclude='*.so' -cf - . | tar -C "$PAIRS" -xf -
  (cd "$PAIRS" && patch -p1 -s < profiles/r06_pair_lanes.patch && python -m harmonies_alphazero_b200.build --force > /dev/null) || exit 1
fi
LIBS="default pairs"
libpath() { if [ "$1" = default ]; then echo "$ROOT/harmonies_alphazero_b200/libharmonies_b200.so"; else echo "$PAIRS/harmonies_alphazero_b200/libharmonies_b200.so"; fi; }
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
for i in 1 2 3; do
  for n in 65536 85248; do timeout 300 python profiles/playout_ab.py $n 2>&1 | tail -n 1 | sed "s|^|premise $n run $i: |"; done
done
(cd "$PAIRS" && timeout 900 python -m pytest -q -m gpu -p no:cacheprovider tests/test_gpu_playout_pairs.py \
  tests/test_gpu_playout_rounds.py tests/test_gpu_playout_pick.py tests/test_gpu_engine.py tests/test_gpu_rollout_eval.py 2>&1 | tail -n 3)
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
