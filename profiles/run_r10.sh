#!/bin/bash
# Gumbel search (DESIGN.md §13) on one B200, in one run: the card, the whole GPU suite, smoke(), the Gumbel tests on the
# bounds-checked build (libharmonies_b200_dbg.so, built beforehand with HZ_NVCC_EXTRA=-DHZ_DEBUG_BOUNDS as in
# run_bounds.sh), then gumbel_bench.py (step split, whole searches, whole games, arena) and bench.py.
# Usage: bash profiles/run_r10.sh [output directory]; everything printed also goes to <output directory>/log.txt.
set -u
OUT=${1:-${TMPDIR:-/tmp}/hz_profile}
mkdir -p "$OUT"
L=$PWD/harmonies_alphazero_b200
exec > >(tee "$OUT"/log.txt) 2>&1
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
timeout 1500 python -m pytest -q -m gpu -p no:cacheprovider tests 2>&1 | tail -n 12
ok=${PIPESTATUS[0]}
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -n 2
ok=$((ok + PIPESTATUS[0]))
echo "== Gumbel tests on the bounds-checked build"
HZ_LIB_PATH=$L/libharmonies_b200_dbg.so timeout 900 python -m pytest -q -m gpu -p no:cacheprovider tests/test_gpu_gumbel.py 2>&1 | tail -n 4
ok=$((ok + PIPESTATUS[0]))
if [ "$ok" != 0 ]; then echo "correctness failed: no timing"; exit 1; fi
timeout 1500 python profiles/gumbel_bench.py --json "$OUT"/r10_gumbel.json 2>&1 | grep -v '^ ' | tail -n 20
timeout 900 python bench.py --gpus 1 --steps 20 --warmup 3 2> "$OUT"/bench.err | tail -n 1 | cut -c1-400
