#!/usr/bin/env bash
# Round 2: same-box A/B of the cfg3 kernel: round-1 tree (.r1copy) vs this tree, then the new parity tests.
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
for rep in 1 2; do
  echo "== round-1 kernel (rep $rep)"
  (cd .r1copy && timeout 200 python bench.py --steps 10 --warmup 3 --no-cpu-baseline --e2e-channels 2 2>&1 | tail -1 | python -c "
import sys, json
d = json.loads(sys.stdin.read()); print('r1   %.1f Gs/s  frac %.3f' % (d['value'], d['roofline']['frac']))")
  echo "== this tree (rep $rep)"
  timeout 300 python bench.py --steps 10 --warmup 3 --no-cpu-baseline --e2e-channels 2 --configs "" 2>&1 | tail -1 | python -c "
import sys, json
d = json.loads(sys.stdin.read()); print('new  %.1f Gs/s  frac %.3f' % (d['value'], d['roofline']['frac']))"
done
echo "== new gpu tests"; timeout 900 python -m pytest tests -x -q -m gpu -k "cfg5 or batch_optimiser or small_sweeps or optimisers or tmem or size_independent" 2>&1 | tail -8
echo "== cfg5 bench"; timeout 600 python bench.py --steps 3 --warmup 3 --no-cpu-baseline --channels-per-gpu 16 --frames 2000000 --e2e-channels 2 --configs 5 2>&1 | tail -1 | python -c "
import sys, json
d = json.loads(sys.stdin.read()); c = d['configs']['cfg5']; print(json.dumps({k: c[k] for k in ('value', 'ms', 'evaluations', 'kernel_launches', 'grid_kernel', 'lsu_pipe')}))"
