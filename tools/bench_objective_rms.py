#!/usr/bin/env python
"""grid_scan over rms-normalised velvet-noise families against the candidate-by-candidate loop (GPU box).

    python tools/bench_objective_rms.py [--reps 5] [--warmup 2] [--loop-cands 32] [--out FILE]

Sweeps of VelvetNoise with the default normaliser (rms_normalize), mode MS, both channels filtered:
  strength  30 s at 48 kHz (seeded noise), log_distribution_strength over [0, 1], 1024 candidates
  seed      viola excerpt of tests/golden (44.1 kHz), seeds 0..399
  width     30 s at 48 kHz, width over [0, 1], 400 candidates
The input is a CUDA tensor.  For each: the family call (`grid_scan`, CUDA events around it, host work included), its
launches, and the time of each of its three kernels (torch.profiler, a separate run); the candidate-by-candidate loop
(decorrelate, download, score: the path these candidates took before) timed on the first `loop_cands` candidates and
scaled to the grid.  Every score of those candidates is checked equal to the loop's first.

Both sides of the routing threshold `_RMS_FAMILY_MIN` on a 10-minute 48 kHz clip, as numpy array and as CUDA tensor:
the loop over K candidates and the family call over K candidates for K from 1 to 8, so that the table shows where the
family starts to win (and the same on the 30 s clip, where the loop is cheapest per frame); `threshold` holds the loop
at `_RMS_FAMILY_MIN - 1` candidates and the family at `_RMS_FAMILY_MIN`.  Each timing: `warmup` untimed calls, then median and best of `reps` (the 10-minute ones: one warm-up,
three reps).  Prints one JSON line (and writes it to --out), with the card's name and power limit read in the same run."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
from bench_decorrelate_batch import card, launches, time_events  # noqa: E402
from bench_objective_families import quiet  # noqa: E402

from tests import _golden as G  # noqa: E402
from vndecorrelate_b200 import decorrelation as D  # noqa: E402
from vndecorrelate_b200 import optimization as opt  # noqa: E402

KW = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)
KERNELS = ("vn_rms_sums_kernel", "vn_stereo_objective_kernel", "obj_combine_kernel")


def candidates(kind, fs, grid):
    g = np.linspace(0.0, 1.0, grid)
    if kind == "strength":
        return [D.VelvetNoise(sample_rate_hz=fs, log_distribution_strength=k, seed=1) for k in g]
    if kind == "width":
        return [D.VelvetNoise(sample_rate_hz=fs, width=w, seed=1) for w in g]
    return [D.VelvetNoise(sample_rate_hz=fs, seed=s) for s in range(grid)]


def kernel_ms(fn, reps=3):
    """Mean device time per call of each of the family's kernels, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    fn()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    out = {k: 0.0 for k in KERNELS}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        for k in KERNELS:
            if k in e.key:
                out[k] += t / 1e3 / reps
    return out


def check_parity(x, cands, family_scores, what):
    want = [opt._score_signal(d.decorrelate(x), KW) for d in cands]
    assert all(g == w and type(g) is type(w) for g, w in zip(family_scores, want)), f"{what}: a score differs from the loop"


def run(kind, clip_name, x, fs, grid, args) -> dict:
    cands = candidates(kind, fs, grid)
    family = quiet(lambda: opt.grid_scan(x, cands, **KW))
    sub = cands[: args.loop_cands]
    loop = lambda: [opt._score_signal(d.decorrelate(x), KW) for d in sub]  # noqa: E731
    check_parity(x, sub, family()[: len(sub)], f"{kind} on {clip_name}")
    f_med, f_best = time_events(family, args.warmup, args.reps)
    l_med, _ = time_events(loop, 1, max(1, args.reps // 2))
    return {"workload": kind, "clip": clip_name, "frames": int(x.shape[0]), "grid": grid, "parity_checked_candidates": len(sub),
            "family_ms_median": f_med, "family_ms_best": f_best, "family_launches": launches(family),
            "kernel_ms": kernel_ms(family), "loop_ms_per_candidate_median": l_med / len(sub), "loop_ms_scaled_to_grid": l_med / len(sub) * grid,
            "loop_launches_per_candidate": launches(loop) / len(sub), "loop_over_family": l_med / len(sub) * grid / f_med}


def threshold_sides(x, what) -> dict:
    cands = candidates("strength", 48000, 8)
    loop_ms, family_ms = {}, {}
    for k in range(1, 9):
        sub = cands[:k]
        loop = lambda: [opt._score_signal(d.decorrelate(x), KW) for d in sub]  # noqa: E731
        fam = quiet(lambda: opt._vn_stereo_rms_partials(opt._cast_input(x), opt._planar_input(opt._cast_input(x)), sub))
        loop_ms[k] = time_events(loop, 1, 3)[0]
        family_ms[k] = time_events(fam, 1, 3)[0] if k >= 2 else None
    scan = quiet(lambda: opt.grid_scan(x, cands[:2], **KW))
    check_parity(x, cands[:2], scan(), f"threshold on {what}")
    m = opt._RMS_FAMILY_MIN
    fam_k = quiet(lambda: opt.grid_scan(x, cands[:m], **KW))
    return {"input": what, "frames": int(x.shape[0]), "loop_ms_by_candidates": loop_ms, "family_partials_ms_by_candidates": family_ms,
            "kernel_ms_at_2": kernel_ms(lambda: opt._vn_stereo_rms_partials(opt._cast_input(x), opt._planar_input(opt._cast_input(x)), cands[:2]), 1),
            "threshold": {"min": m, "loop_ms_at_min_minus_1": loop_ms[m - 1], "family_grid_scan_ms_at_min": time_events(fam_k, 1, 3)[0],
                          "family_launches_at_min": launches(fam_k)}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--loop-cands", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    viola_fs, viola = G.wav("viola")
    rng = np.random.default_rng(7)
    long = (rng.standard_normal((30 * 48000, 2)) * 0.3).astype(np.float32)
    xl = torch.from_numpy(long).cuda()
    xv = torch.from_numpy(np.ascontiguousarray(viola, dtype=np.float32)).cuda()
    t0 = time.perf_counter()
    results = []
    for kind, name, x, fs, grid in (("strength", "noise_30s_48k", xl, 48000, 1024), ("seed", "viola", xv, viola_fs, 400),
                                    ("width", "noise_30s_48k", xl, 48000, 400)):
        results.append(run(kind, name, x, fs, grid, args))
        print(json.dumps(results[-1]), file=sys.stderr)
    ten = (rng.standard_normal((600 * 48000, 2)) * 0.3).astype(np.float32)
    sides = []
    for what, x in (("numpy_10min", ten), ("cuda_tensor_10min", torch.from_numpy(ten).cuda()), ("cuda_tensor_30s", xl)):
        sides.append(threshold_sides(x, what))
        print(json.dumps(sides[-1]), file=sys.stderr)
    out = {"bench": "objective_rms", "card": card(), "reps": args.reps, "warmup": args.warmup, "wall_s": time.perf_counter() - t0,
           "results": results, "threshold": sides}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
