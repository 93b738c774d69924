#!/bin/bash
# A/B of the fp32-filtered pair kernel against the all-fp64 one: pair parity tests (all, not -x), then the pair-only bench
# for both.  Usage: gpurun --timeout 1200 -- 'bash tools/gpu_fast_ab.sh [ncu] [frames]'
set -u
cd "$(dirname "$0")/.."
OUT=gpurun_out
mkdir -p $OUT
FR=${2:-256}
timeout 900 python -m pytest tests -m gpu -q -p no:cacheprovider --timeout 600 -k "pair or rdf or cn or bin or large or smoke or cluster or hydration or residence" > $OUT/pytest_fast.log 2>&1; echo "pytest rc=$?"
tail -5 $OUT/pytest_fast.log
for mode in fast f64; do
  unset MDP_PAIR_F64
  if [ $mode = f64 ]; then export MDP_PAIR_F64=1; fi
  timeout 600 python bench.py --steps 6 --warmup 3 --frames $FR --skip-msd --skip-cpu --skip-gk --skip-residence --skip-clusters > $OUT/bench_ab_$mode.json 2> $OUT/bench_ab_$mode.err; echo "bench $mode rc=$?"
  tail -3 $OUT/bench_ab_$mode.err
  python - <<PY
import json
try:
    d=json.load(open('gpurun_out/bench_ab_$mode.json'))
    print('$mode', {k:d.get(k) for k in ('value','ms_per_step','evaluated_pair_evals_per_step','exact_path_pairs_per_step','kernel_share','pairs_in_cutoff_frame0','hist_sha256')})
    print('$mode roofline', d['roofline']['achieved'], d['roofline']['frac'], 'e2e', d['e2e']['value'])
    t=d.get('rdf_triclinic',{}); print('$mode tricl', t.get('pair_kernel_ms_per_step'), t.get('pairs_in_cutoff_frame0'))
except Exception as e:
    print('no bench json', e)
PY
done
unset MDP_PAIR_F64
if [ "${1:-}" = "ncu" ]; then
  timeout 900 ncu --set full --clock-control none --import-source on -k regex:k_pair -s 3 -c 1 -f -o $OUT/prof_pair_fast \
      python bench.py --steps 1 --warmup 1 --frames 16 --skip-msd --skip-cpu --skip-gk --skip-residence --skip-clusters --skip-triclinic > $OUT/ncu_pair_fast.log 2>&1
  echo "ncu pair rc=$?"
fi
