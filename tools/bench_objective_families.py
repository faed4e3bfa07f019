#!/usr/bin/env python
"""grid_scan over the velvet-noise stereo and Haas families against the candidate-by-candidate loop (GPU box).

    python tools/bench_objective_families.py [--reps 5] [--warmup 2] [--loop-cands 32] [--out FILE]

Workloads, each on the viola excerpt of tests/golden (44.1 kHz) and on a seeded 30 s 48 kHz stereo clip:
  ms_strength  VelvetNoise(mode='MS', filtered_channels=(0, 1), normalizer=None), log_distribution_strength over [0, 1]
  width        the same filter at strength 1, width over [0, 1]
  haas_ch1_ms  HaasEffect(delayed_channel=1, mode='MS'), delay over [0, 20 ms]
at grids of 400 and 1024 candidates (the Haas sweep at 400).  The input is a CUDA tensor.  For each: the family call
(`grid_scan`, CUDA events around it, host work included), its launches, and the kernel's candidate evaluations per
second (the family partials call alone, evaluations = candidates x clips); for the velvet-noise sweeps the same rate
of the reference's LR family (filtered_channels=(0,), mode 'LR', no normaliser) on the same clip and grid through its
own kernel.  The candidate-by-candidate loop (decorrelate, download, score: the path these candidates took before) is
timed on the first `loop_cands` candidates and reported per candidate and scaled to the grid.  Every score of those
candidates is checked for equality with the loop first.  Each timing: `warmup` untimed calls, then median and best of
`reps`.  Prints one JSON line (and writes it to --out), with the card's name and power limit read in the same run."""
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

from tests import _golden as G  # noqa: E402
from vndecorrelate_b200 import decorrelation as D  # noqa: E402
from vndecorrelate_b200 import optimization as opt  # noqa: E402

KW = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)


def candidates(kind, fs, grid):
    g = np.linspace(0.0, 1.0, grid)
    if kind == "ms_strength":
        return [D.VelvetNoise(sample_rate_hz=fs, normalizer=None, log_distribution_strength=k, seed=1) for k in g]
    if kind == "width":
        return [D.VelvetNoise(sample_rate_hz=fs, normalizer=None, width=w, seed=1) for w in g]
    if kind == "lr_family":
        return [D.VelvetNoise(sample_rate_hz=fs, normalizer=None, log_distribution_strength=k, filtered_channels=(0,), mode="LR", seed=1) for k in g]
    return [D.HaasEffect(sample_rate_hz=fs, delay_time_seconds=0.02 * t, delayed_channel=1, mode="MS") for t in g]


def quiet(fn):
    """grid_scan prints a line per call, as the reference's does: keep it out of the timings' output."""
    def run():
        sys.stdout, saved = open(os.devnull, "w"), sys.stdout
        try:
            return fn()
        finally:
            sys.stdout.close()
            sys.stdout = saved
    return run


def partials_call(kind, x, cands):
    if kind == "lr_family":
        prog = opt._vn_family_program(cands, x.shape[0])
        planar = x.t().contiguous()[None]
        return lambda: opt.vn_objective_partials(planar, prog)
    if kind == "haas_ch1_ms":
        return lambda: opt.haas_effect_objective_partials(x, cands)
    return lambda: opt.vn_stereo_objective_partials(x, cands)


def run(kind, clip_name, x, fs, grid, args) -> dict:
    cands = candidates(kind, fs, grid)
    family = quiet(lambda: opt.grid_scan(x, cands, **KW))
    sub = cands[: args.loop_cands]
    loop = lambda: [opt._score_signal(d.decorrelate(x), KW) for d in sub]  # noqa: E731
    got, want = family()[: len(sub)], loop()
    assert all(g == w and type(g) is type(w) for g, w in zip(got, want)), f"{kind} on {clip_name}: a score differs from the loop"
    f_med, f_best = time_events(family, args.warmup, args.reps)
    l_med, l_best = time_events(loop, 1, max(1, args.reps // 2))
    k_med, k_best = time_events(partials_call(kind, x, cands), args.warmup, args.reps)
    rec = {"workload": kind, "clip": clip_name, "frames": int(x.shape[0]), "grid": grid, "parity_checked_candidates": len(sub),
           "family_ms_median": f_med, "family_ms_best": f_best, "family_launches": launches(family),
           "loop_ms_per_candidate_median": l_med / len(sub), "loop_ms_scaled_to_grid": l_med / len(sub) * grid,
           "loop_launches_per_candidate": launches(loop) / len(sub), "loop_over_family": l_med / len(sub) * grid / f_med,
           "kernel_evaluations_per_s": grid / (k_med * 1e-3)}
    if kind != "haas_ch1_ms":
        lr = candidates("lr_family", fs, grid)
        lr_med, _ = time_events(partials_call("lr_family", x, lr), args.warmup, args.reps)
        rec["lr_family_kernel_evaluations_per_s"] = grid / (lr_med * 1e-3)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--loop-cands", type=int, default=32)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    viola_fs, viola = G.wav("viola")
    long = (np.random.default_rng(7).standard_normal((30 * 48000, 2)) * 0.3).astype(np.float32)
    clips = [("viola", torch.from_numpy(np.ascontiguousarray(viola, dtype=np.float32)).cuda(), viola_fs),
             ("noise_30s_48k", torch.from_numpy(long).cuda(), 48000)]
    t0 = time.perf_counter()
    results = []
    for name, x, fs in clips:
        for kind, grids in (("ms_strength", (400, 1024)), ("width", (400, 1024)), ("haas_ch1_ms", (400,))):
            for grid in grids:
                results.append(run(kind, name, x, fs, grid, args))
                print(json.dumps(results[-1]), file=sys.stderr)
    out = {"bench": "objective_families", "card": card(), "reps": args.reps, "warmup": args.warmup, "wall_s": time.perf_counter() - t0,
           "results": results}
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
