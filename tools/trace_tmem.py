#!/usr/bin/env python
"""Timeline of CTA 0 of the tensor-memory kernel (debug build with -DVND_TM_TRACE; GPU box only).

    VND_EXTRA_DEFS=-DVND_TM_TRACE bash vndecorrelate_b200/csrc/build.sh && python tools/trace_tmem.py

Prints, per lane quarter, the clock of every traced event of tiles 8..15 of the first run relative to the
start of tile 8 on warp 0, and saves the raw table to gpurun_out/tm_trace.npy."""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from vndecorrelate_b200 import _native as N  # noqa: E402
from vndecorrelate_b200.decorrelation import VelvetNoise  # noqa: E402

Cn, L = 148, 2_000_000
vn = VelvetNoise(sample_rate_hz=48000, duration_seconds=0.03, num_impulses=30, num_outs=Cn, filtered_channels=tuple(range(Cn)), mode="LR",
                 normalizer=None, seed=1)
x = torch.randn((Cn, L), device="cuda") * 0.1
for _ in range(3):
    y = vn.convolve(x.t())
torch.cuda.synchronize()
buf = np.zeros((16, 64, 8), dtype=np.uint64)
rc = N.lib().vnd_debug_tm_trace(buf.ctypes.data_as(C.c_void_p))
assert rc == 0, rc
os.makedirs(os.path.join(ROOT, "gpurun_out"), exist_ok=True)
np.save(os.path.join(ROOT, "gpurun_out", "tm_trace.npy"), buf)
t = buf.astype(np.int64)
t0 = t[0, 8, 0]
names_c = ["start", "waits done", "near done", "far done", "staged", "stage free"]
names_h = ["fill start", "fill end", "store done", "-", "in_full ok"]
for q in range(4):
    print(f"== quarter {q}")
    for ti in range(8, 14):
        line = f"tile {ti}: "
        for g in range(3):
            w = q + 4 * g
            line += f"| g{g} " + " ".join(f"{names_c[e][:5]}={t[w, ti, e] - t0:6d}" for e in (0, 1, 2, 3, 5, 4))
        h = 12 + q
        line += " | helper " + " ".join(f"{names_h[e][:7]}={t[h, ti, e] - t0:6d}" for e in (4, 0, 1, 2))
        print(line)
per_tile = (t[0, 40, 0] - t[0, 8, 0]) / 32
print("clk per tile (warp 0, tiles 8..40):", per_tile)
