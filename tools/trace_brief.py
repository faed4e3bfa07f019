"""Per-phase durations from gpurun_out/tm_trace.npy (tools/trace_tmem.py): medians over tiles 8..40 per quarter."""
import os, sys
import numpy as np
t = np.load(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "gpurun_out", "tm_trace.npy")).astype(np.int64)
tiles = slice(8, 40)
for q in range(4):
    w = q  # group 0 warp of the quarter
    st, wt, nd, fd, sf, sg = (t[w, tiles, e] for e in (0, 1, 2, 3, 5, 4))
    h = 12 + q
    hin, hf0, hf1, hst = (t[h, tiles, e] for e in (4, 0, 1, 2))
    med = lambda a: int(np.median(a))
    period = med(np.diff(t[w, 8:41, 0]))
    print(f"q{q}: period {period}  wait {med(wt - st)}  tmem {med(nd - wt)}  far {med(fd - nd)}  stfree {med(sf - fd)}  stage {med(sg - sf)} | "
          f"helper: fill {med(hf1 - hf0)}  fill start after near-done {med(hf0 - np.roll(nd, 1)[1:].tolist()[0:1][0]) if False else med(hf0[1:] - nd[:-1])}  fill end before next wait-done {med(wt[1:] - hf1[1:])}  store-done after fill-end {med(hst - hf1)}")
print("phase offsets of quarter starts vs q0 (median):", [int(np.median(t[q, tiles, 0] - t[0, tiles, 0])) for q in range(4)])
