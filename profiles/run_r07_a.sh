#!/bin/bash
# Symmetry feature on the GPU, in stages of a few minutes each.  Usage: bash profiles/run_r07_a.sh [stage] [output directory]
#   sym   (default) card and power limit, the new GPU tests, smoke(), profiles/symmetry_step.py (step cost of the
#         leaf-frame modes, bulk transforms at 1 M rows)
#   suite the rest of the GPU suite
#   bench bench.py of this tree, then of a parent-commit tree staged in _parent_tree/ (when present)
set -u
STAGE=${1:-sym}
OUT=${2:-${TMPDIR:-/tmp}/hz_profile}   # output directory (second argument)
mkdir -p "$OUT" && OUT=$(cd "$OUT" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT"/gpu_$STAGE.txt
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -3
if [ "$STAGE" = sym ]; then
  timeout 300 python -m pytest -q -m gpu -p no:cacheprovider tests/test_gpu_symmetry.py 2>&1 | tail -n 60 > "$OUT"/sym_tests.txt; echo "sym tests rc=${PIPESTATUS[0]}"
  tail -n 40 "$OUT"/sym_tests.txt
  timeout 120 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3
  timeout 150 python profiles/symmetry_step.py --out "$OUT"/symmetry_step.json 2>&1 | tail -n 3
elif [ "$STAGE" = suite ]; then
  timeout 560 python -m pytest -q -m gpu -p no:cacheprovider tests/ --ignore=tests/test_gpu_symmetry.py 2>&1 | tail -n 30 > "$OUT"/gpu_suite.txt; echo "gpu suite rc=${PIPESTATUS[0]}"
  tail -n 12 "$OUT"/gpu_suite.txt
elif [ "$STAGE" = bench ]; then
  echo "bench this tree:"; timeout 270 python bench.py --gpus 1 2> "$OUT"/bench_new.err | tail -n 1 | tee "$OUT"/bench_new.json
  if [ -d _parent_tree ]; then
    echo "bench parent:"; (cd _parent_tree && timeout 270 python bench.py --gpus 1 2> "$OUT"/bench_parent.err | tail -n 1 | tee "$OUT"/bench_parent.json)
  fi
fi
