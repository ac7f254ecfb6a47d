#!/bin/bash
# bench.py (default arguments) three times on each of two builds, alternated, with the card's name and power limit read in
# the same run; then the whole GPU suite and smoke() on the in-tree build.  HZ_AB_OLD names the other build
# (libharmonies_b200_<name>.so, default: stepwise = nvcc -DHZ_PLAYOUT_STEPWISE).  One JSON line per run under the
# output directory.  Usage: bash profiles/run_r03_b.sh [output directory]
set -u
OUT=${1:-${TMPDIR:-/tmp}/hz_profile}   # output directory (first argument)
mkdir -p "$OUT"
L=$PWD/harmonies_alphazero_b200
OLD=${HZ_AB_OLD:-stepwise}
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader
for i in 1 2 3; do
  for b in $OLD default; do
    lib=$L/libharmonies_b200.so; [ $b = default ] || lib=$L/libharmonies_b200_$b.so
    HZ_LIB_PATH=$lib timeout 900 python bench.py > "$OUT"/r03_bench_${b}_$i.json 2> "$OUT"/r03_bench_${b}_$i.err
    echo "bench $b run $i rc=$?"
    python - "$OUT"/r03_bench_${b}_$i.json <<'PY'
import json, sys
d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
print(f"  value {d['value']:.4g} steps/s  ms_per_step {d['ms_per_step'] * 1e3:.2f} us  e2e {d['e2e']['value']:.4g}  wall_s {d.get('wall_s')}  "
      f"clocks {d.get('clocks', {}).get('sm_mhz')}  roofline {d['roofline'].get('note', '')[:60]}")
PY
  done
done
nvidia-smi --query-gpu=name,power.limit --format=csv,noheader
timeout 1500 python -m pytest -q -m gpu -p no:cacheprovider tests 2>&1 | tail -n 4
timeout 300 python __graft_entry__.py --smoke 2>&1 | tail -n 2
