#!/usr/bin/env bash
# Round 2, call 5: full gpu suite; cfg3 A/B (this tree's tensor-memory FIR file vs round 1's inside this tree).
cd "$(dirname "$0")/.."
mkdir -p gpurun_out
echo "== gpu tests"; timeout 900 python -m pytest tests -x -q -m gpu 2>&1 | tail -6
b() { timeout 300 env "$@" python bench.py --steps 10 --warmup 3 --no-cpu-baseline --e2e-channels 2 --configs "" 2>&1 | tail -1 | python -c "
import sys, json
d = json.loads(sys.stdin.read()); print('%.1f Gs/s  frac %.3f' % (d['value'], d['roofline']['frac']))"; }
echo -n "cfg3 this tree:            "; b A=1
echo -n "cfg3 round-1 kernel file:  "; b VND_B200_LIB=$PWD/vndecorrelate_b200/_lib/libvnd_b200_r1tm.so
echo -n "cfg3 this tree:            "; b A=1
echo -n "cfg3 round-1 kernel file:  "; b VND_B200_LIB=$PWD/vndecorrelate_b200/_lib/libvnd_b200_r1tm.so
