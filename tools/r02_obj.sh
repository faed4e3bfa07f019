#!/usr/bin/env bash
# Round 2: objective kernel chunking sweep; then parity tests and the cfg3 A/B against the round-1 tree on the same box.
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
run() { echo -n "$1: "; shift; env "$@" timeout 300 python tools/bench_objective.py --clips ${CLIPS:-16} --reps 3 --check 2>&1 | tail -1; }
run "planned chunks"
for t in 36 22 10; do run "tpc=$t" VND_OBJ_TPC=$t; done
echo "== gpu tests (objective, optimisers, cfg5, tmem FIR)"; timeout 900 python -m pytest tests -q -m gpu -k "objective or sweeps or optimis or cfg5 or batch or tmem or size_independent or cfg4 or planar" 2>&1 | tail -8
for rep in 1; do
  (cd .r1copy && timeout 200 python bench.py --steps 10 --warmup 3 --no-cpu-baseline --e2e-channels 2 2>&1 | tail -1 | python -c "
import sys, json
d = json.loads(sys.stdin.read()); print('cfg3 r1   %.1f Gs/s  frac %.3f' % (d['value'], d['roofline']['frac']))")
  timeout 300 python bench.py --steps 10 --warmup 3 --no-cpu-baseline --e2e-channels 2 --configs "" 2>&1 | tail -1 | python -c "
import sys, json
d = json.loads(sys.stdin.read()); print('cfg3 new  %.1f Gs/s  frac %.3f' % (d['value'], d['roofline']['frac']))"
done
