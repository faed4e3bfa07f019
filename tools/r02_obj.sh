#!/usr/bin/env bash
# Round 2: objective kernels - shared-memory kernel vs tensor-memory kernel, chunking sweep; then parity tests and the
# cfg3 / cfg4 A/B against the round-1 tree on the same box.
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
run() { echo -n "$1: "; shift; env "$@" timeout 300 python tools/bench_objective.py --clips ${CLIPS:-16} --reps 3 --check 2>&1 | tail -1; }
run "smem kernel, planned chunks" VND_OBJ_TMEM=0
for t in 36 22 10; do run "smem kernel, tpc=$t" VND_OBJ_TMEM=0 VND_OBJ_TPC=$t; done
run "tmem kernel, planned chunks" VND_OBJ_TMEM=1
for t in 48 16 8; do run "tmem kernel, tpc=$t" VND_OBJ_TMEM=1 VND_OBJ_TPC=$t; done
echo "== gpu tests (objective, optimisers, cfg5, tmem FIR)"; timeout 900 python -m pytest tests -q -m gpu -k "objective or sweeps or optimis or cfg5 or batch or tmem or size_independent or cfg4 or planar" 2>&1 | tail -8
echo "== same, every tap through shared memory"; VND_OBJ_TMEM=0 timeout 900 python -m pytest tests -q -m gpu -k "objective or sweeps or optimis or cfg5 or batch" 2>&1 | tail -4
for rep in 1; do
  (cd .r1copy && timeout 200 python bench.py --steps 10 --warmup 3 --no-cpu-baseline --e2e-channels 2 2>&1 | tail -1 | python -c "
import sys, json
d = json.loads(sys.stdin.read()); print('cfg3 r1   %.1f Gs/s  frac %.3f' % (d['value'], d['roofline']['frac']))")
  timeout 300 python bench.py --steps 10 --warmup 3 --no-cpu-baseline --e2e-channels 2 --configs "" 2>&1 | tail -1 | python -c "
import sys, json
d = json.loads(sys.stdin.read()); print('cfg3 new  %.1f Gs/s  frac %.3f' % (d['value'], d['roofline']['frac']))"
done
for r in 8 12 16; do
  VND_LONG_R=$r timeout 300 python bench.py --steps 3 --warmup 3 --no-cpu-baseline --channels-per-gpu 16 --frames 2000000 --e2e-channels 2 --configs 4 --cfg4-channels-per-gpu 64 2>&1 | tail -1 | python -c "
import sys, json
d = json.loads(sys.stdin.read()); c = d['configs']['cfg4']; print('cfg4 R=$r  %.2f Gs/s  lsu %.3f  %s' % (c['value'], c['lsu_pipe']['frac'], c['parity'][:20]))"
done
