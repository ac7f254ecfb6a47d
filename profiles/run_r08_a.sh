#!/bin/bash
# Leaf evaluation cache on the GPU in one call: card and power limit, the new tests (release and -DHZ_DEBUG_BOUNDS
# builds), the self-play and symmetry suites, smoke(), bench.py, then profiles/eval_cache_bench.py at 100 sims (with the
# step split), 32 sims, 400 sims and 100 sims with eval_symmetry="board".
# Usage: bash profiles/run_r08_a.sh [output directory]
set -u
OUT=${1:-${TMPDIR:-/tmp}/hz_profile}
mkdir -p "$OUT" && OUT=$(cd "$OUT" && pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT"/gpu.txt
python -c "import __graft_entry__ as g; g.build()" 2>&1 | tail -3
timeout 600 python -m pytest -q -m gpu -p no:cacheprovider tests/test_gpu_eval_cache.py 2>&1 | tail -n 40 > "$OUT"/eval_cache_tests.txt; echo "eval cache tests rc=${PIPESTATUS[0]}"
tail -n 25 "$OUT"/eval_cache_tests.txt
timeout 150 python -c "import __graft_entry__ as g; g.smoke(); print('smoke ok')" 2>&1 | tail -3
timeout 300 python bench.py --gpus 1 2> "$OUT"/bench.err | tail -n 1 | tee "$OUT"/bench.json
timeout 420 python profiles/eval_cache_bench.py --sims 100 --games 8192 --reps 3 --split --out "$OUT"/r08_eval_cache_100.json 2>&1 | tail -n 8
timeout 240 python profiles/eval_cache_bench.py --sims 32 --games 8192 --reps 2 --out "$OUT"/r08_eval_cache_32.json 2>&1 | tail -n 1
timeout 420 python profiles/eval_cache_bench.py --sims 400 --games 4096 --reps 1 --out "$OUT"/r08_eval_cache_400.json 2>&1 | tail -n 1
timeout 240 python profiles/eval_cache_bench.py --sims 100 --games 8192 --reps 1 --symmetry board --out "$OUT"/r08_eval_cache_100_board.json 2>&1 | tail -n 1
if [ -f harmonies_alphazero_b200/libharmonies_b200_dbg.so ]; then
  HZ_LIB_PATH=$PWD/harmonies_alphazero_b200/libharmonies_b200_dbg.so timeout 900 python -m pytest -q -m gpu -p no:cacheprovider tests/test_gpu_eval_cache.py 2>&1 | tail -n 8 > "$OUT"/eval_cache_bounds.txt; echo "bounds build rc=${PIPESTATUS[0]}"
  tail -n 4 "$OUT"/eval_cache_bounds.txt
fi
timeout 900 python -m pytest -q -m gpu -p no:cacheprovider tests/test_gpu_selfplay.py tests/test_gpu_symmetry.py tests/test_gpu_mcts.py 2>&1 | tail -n 12 > "$OUT"/gpu_suite_part.txt; echo "selfplay/symmetry/mcts suites rc=${PIPESTATUS[0]}"
tail -n 5 "$OUT"/gpu_suite_part.txt
