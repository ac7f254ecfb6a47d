#!/bin/bash
# Rollout evaluator (hz_tree_rollout_eval): correctness first, then the measurements, in one run.
#   Build beforehand (nvcc needs no GPU): the in-tree library, libharmonies_b200_dbg.so (nvcc -DHZ_DEBUG_BOUNDS, as in
#   run_bounds.sh) and, for the bench.py A/B, a checkout of the parent commit with its own library built, named by
#   HZ_PARENT_TREE (a directory).  Usage: bash profiles/run_r04_a.sh <output directory>
# Writes: card.txt, smoke.txt, gpu_suite.txt (whole GPU suite), bounds_rollout.txt (the rollout tests on the bounds-checked
# build), bench_<build>_<i>.json (bench.py alternated between the parent and this build), dump comparison lines in
# bench_dump.txt, and rollout_bench.txt (profiles/rollout_bench.py).
set -u
OUT=${1:?usage: run_r04_a.sh <output directory>}
mkdir -p "$OUT"
L=$PWD/harmonies_alphazero_b200
PARENT=${HZ_PARENT_TREE:-}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT"/card.txt
timeout 600 python -c "import __graft_entry__ as g; g.build(); g.smoke(); print('smoke ok')" > "$OUT"/smoke.txt 2>&1
tail -n 3 "$OUT"/smoke.txt
timeout 2400 python -m pytest -q -m gpu -p no:cacheprovider tests 2>&1 | tail -n 15 > "$OUT"/gpu_suite.txt
tail -n 3 "$OUT"/gpu_suite.txt
HZ_LIB_PATH=$L/libharmonies_b200_dbg.so timeout 1200 python -m pytest -q -m gpu -p no:cacheprovider tests/test_gpu_rollout_eval.py \
  2>&1 | tail -n 8 > "$OUT"/bounds_rollout.txt
tail -n 2 "$OUT"/bounds_rollout.txt
BUILDS="this"
[ -n "$PARENT" ] && BUILDS="parent this"
tree_of() { if [ "$1" = parent ]; then echo "$PARENT"; else echo "$PWD"; fi; }
for i in 1 2 3; do
  for b in $BUILDS; do
    (cd "$(tree_of $b)" && timeout 900 python bench.py --gpus 1 --steps 20 --warmup 3 --no-cpu-baseline --no-python-reference \
      --mcts-play-games 0) > "$OUT"/bench_${b}_$i.json 2> "$OUT"/bench_${b}_$i.err
    echo "bench $b run $i rc=$?: $(tail -n 1 "$OUT"/bench_${b}_$i.json | cut -c1-400)"
  done
done
D=${TMPDIR:-/tmp}/hz_r04_dump
for b in $BUILDS; do
  (cd "$(tree_of $b)" && timeout 600 python bench.py --no-mcts --no-cpu-baseline --no-python-reference --dump-outputs "$D"/$b) \
    > /dev/null 2>&1
  echo "dump $b rc=$?"
done | tee "$OUT"/bench_dump.txt
if [ -n "$PARENT" ]; then
  for f in $(cd "$D"/parent && ls); do cmp "$D"/parent/$f "$D"/this/$f && echo "$f identical"; done | tee -a "$OUT"/bench_dump.txt
fi
rm -rf "$D"
timeout 2400 python profiles/rollout_bench.py > "$OUT"/rollout_bench.txt 2>&1
tail -n 20 "$OUT"/rollout_bench.txt | cut -c1-300
