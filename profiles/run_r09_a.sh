#!/bin/bash
# k_playout's tables copied in one round trip (fetch_tables / store_tables) against libharmonies_b200_parent.so (the
# previous commit's sources, built beforehand with build.py: nvcc needs no GPU), in one run.
# Usage: bash profiles/run_r09_a.sh [output directory]; everything printed also goes to <output directory>/log.txt.
# Correctness first: the whole GPU suite, smoke() and the bounds-checked build (run_bounds.sh); the timing runs only if
# they passed.  Then playout_ab.py alternated 6x at 65,536 games and 2x at 262,144 games per build, the device-side phase
# timeline of both table copies (playout_timeline.py), the byte comparison of bench.py --dump-outputs between the
# builds and bench.py's engine leg twice per build, alternated.
set -u
OUT=${1:-${TMPDIR:-/tmp}/hz_profile}   # output directory (first argument)
mkdir -p "$OUT"
L=$PWD/harmonies_alphazero_b200
LIBS="default parent"
libpath() { if [ "$1" = default ]; then echo "$L/libharmonies_b200.so"; else echo "$L/libharmonies_b200_$1.so"; fi; }
exec > >(tee "$OUT"/log.txt) 2>&1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
timeout 1500 python -m pytest -q -m gpu -p no:cacheprovider tests 2>&1 | tail -n 8
ok=${PIPESTATUS[0]}
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -n 2
ok=$((ok + PIPESTATUS[0]))
timeout 1200 bash profiles/run_bounds.sh 2>&1 | grep -E "passed|failed|error|games_per_s" | head -n 6
if [ "$ok" != 0 ]; then echo "correctness failed: no timing"; exit 1; fi
for i in 1 2 3 4 5 6; do
  for b in $LIBS; do HZ_LIB_PATH=$(libpath $b) timeout 300 python profiles/playout_ab.py 2>&1 | tail -n 2 | sed "s|^|$b 65536 run $i: |"; done
done
for i in 1 2; do
  for b in $LIBS; do HZ_LIB_PATH=$(libpath $b) timeout 300 python profiles/playout_ab.py 262144 2>&1 | tail -n 2 | sed "s|^|$b 262144 run $i: |"; done
done
timeout 600 python profiles/playout_timeline.py --libdir "$PWD/build/timeline" --json "$OUT"/timeline.json 2>&1
for b in $LIBS; do
  HZ_LIB_PATH=$(libpath $b) timeout 600 python bench.py --no-mcts --no-cpu-baseline --no-python-reference \
    --dump-outputs "$OUT"/dump_$b > "$OUT"/dump_$b.json 2> "$OUT"/dump_$b.err; echo "dump $b rc=$?"
  for f in states steps total_steps; do cmp "$OUT"/dump_default/$f.npy "$OUT"/dump_$b/$f.npy && echo "$b: $f.npy identical to default"; done
done
rm -rf "$OUT"/dump_*/   # 64 MB each: the comparison above is the result
for i in 1 2; do
  for b in $LIBS; do
    echo "bench $b run $i:"; HZ_LIB_PATH=$(libpath $b) timeout 600 python bench.py --gpus 1 --no-mcts --no-cpu-baseline \
      --no-python-reference 2> "$OUT"/bench_$b.err | tail -n 1
  done
done
