#!/usr/bin/env python
"""optimize_velvet_noise_batch against a loop of optimize_velvet_noise over the same clips, in the same run (GPU box).

    python tools/bench_vn_batch.py [--reps 3] [--warmup 1] [--workloads a,b,c,d] [--out FILE]

Workloads (48 kHz, a 0.03 s filter of 30 impulses, seed 1, seeded coloured stereo noise as in config 5, numpy float32
clips in):
  a  64 clips x 30 s, equal lengths, grid 1024 (config 5's shape)
  b  64 clips of 5-60 s, grid 400
  c  512 clips of 2-6 s, grid 400
  d  256 clips of 0.01-2 s, some shorter than the 1440-frame filter, grid 100
Every clip's strength from the batch is first checked to equal the loop's (==, not approximately).  Then each arm runs
`warmup` untimed calls and `reps` timed ones (host clock around calls that return numpy, so they end in a synchronise);
median and best are reported, with the grid stage and the refinement timed separately inside each call: for the batch,
the grid stage is argument checks + packing + upload + the grid call + scoring; for the loop, the sum over the clips of
the time up to their grid's local-minimum search.  Launches are the library's kernel launches per call.  Prints one
JSON line, with the card's name and power limit read in the same run, and also writes it to FILE when --out is given
(nothing is written otherwise)."""
import argparse
import contextlib
import hashlib
import io
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from oracle import vnd_oracle as O  # noqa: E402
from vndecorrelate_b200 import _native as N  # noqa: E402
from vndecorrelate_b200 import optimization as OPT  # noqa: E402

FS = 48000
SETTINGS = dict(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, seed=1)


def card() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # noqa: BLE001 - recorded, not hidden
        info["power_limit_w"] = f"unavailable ({e})"
    return info


def workload(name: str):
    rng = np.random.default_rng({"a": 1, "b": 2, "c": 3, "d": 4}[name])
    if name == "a":
        lengths, grid = [30 * FS] * 64, 1024
    elif name == "b":
        lengths, grid = rng.integers(5 * FS, 60 * FS + 1, 64).tolist(), 400
    elif name == "c":
        lengths, grid = rng.integers(2 * FS, 6 * FS + 1, 512).tolist(), 400
    else:
        lengths, grid = rng.integers(FS // 100, 2 * FS + 1, 256).tolist(), 100
    return [O.coloured_clip(i, int(n)) for i, n in enumerate(lengths)], grid


def run_batch(clips, grid):
    marks = {}

    class TimedBank(OPT._ClipBank):
        def grid_scores(self, kappas):
            out = super().grid_scores(kappas)
            marks["grid_end"] = time.perf_counter()
            return out

    with contextlib.redirect_stdout(io.StringIO()):
        before = N.launch_count()
        t0 = time.perf_counter()
        kappas, info = OPT.optimize_velvet_noise_batch(input_signals=clips, grid_size=grid, details=True, _bank_factory=TimedBank, **SETTINGS)
        t1 = time.perf_counter()
        launches = N.launch_count() - before
    return kappas, {"total_s": t1 - t0, "grid_s": marks["grid_end"] - t0, "refine_s": t1 - marks["grid_end"], "launches": launches,
                    "calls": info["launches_local"], "evaluations": info["evaluations_local"], "brent_rounds": info["rounds_local"],
                    "minimisers": int(sum(len(m) for m in info["local_minima"]))}


def run_loop(clips, grid):
    acc = {"grid_s": 0.0, "evaluations": 0, "start": 0.0}
    minima, partials = OPT.get_local_minima, OPT.vn_objective_partials

    def timed_minima(*a, **k):  # the single-clip call searches its grid's minima right after scoring it
        acc["grid_s"] += time.perf_counter() - acc["start"]
        return minima(*a, **k)

    def counted_partials(c, prog):
        acc["evaluations"] += prog.channels
        return partials(c, prog)

    OPT.get_local_minima, OPT.vn_objective_partials = timed_minima, counted_partials
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            before = N.launch_count()
            t0 = time.perf_counter()
            out = []
            for c in clips:
                acc["start"] = time.perf_counter()
                out.append(OPT.optimize_velvet_noise(input_signal=c, grid_size=grid, **SETTINGS))
            t1 = time.perf_counter()
            launches = N.launch_count() - before
    finally:
        OPT.get_local_minima, OPT.vn_objective_partials = minima, partials
    return np.array(out, dtype=np.float64), {"total_s": t1 - t0, "grid_s": acc["grid_s"], "refine_s": t1 - t0 - acc["grid_s"], "launches": launches,
                                             "evaluations": acc["evaluations"]}


def stats(runs, key):
    v = [r[key] for r in runs]
    return {"median": float(np.median(v)), "best": float(np.min(v))}


def measure(name, reps, warmup):
    clips, grid = workload(name)
    frames = [len(c) for c in clips]
    got, _ = run_batch(clips, grid)
    want, _ = run_loop(clips, grid)
    equal = bool(np.array_equal(got, want))
    row = {"workload": name, "n_clips": len(clips), "grid": grid, "frames_total": int(sum(frames)), "frames_min": int(min(frames)),
           "frames_max": int(max(frames)), "clips_shorter_than_filter": int(sum(f < 1440 for f in frames)), "per_clip_equal": equal,
           "clips_equal": int(np.sum(got == want)), "kappa_sha256": hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest()}
    if not equal:
        row["mismatch"] = [int(i) for i in np.nonzero(got != want)[0][:16]]
        return row
    for arm, fn in (("batch", run_batch), ("loop", run_loop)):
        for _ in range(warmup):
            fn(clips, grid)
        runs = [fn(clips, grid)[1] for _ in range(reps)]
        row[arm] = {"total_s": stats(runs, "total_s"), "grid_s": stats(runs, "grid_s"), "refine_s": stats(runs, "refine_s"),
                    **{k: runs[-1][k] for k in runs[-1] if k not in ("total_s", "grid_s", "refine_s")}}
    row["loop_over_batch_median"] = row["loop"]["total_s"]["median"] / row["batch"]["total_s"]["median"]
    row["loop_over_batch_best"] = row["loop"]["total_s"]["best"] / row["batch"]["total_s"]["best"]
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default="a,b,c,d")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    res = {"card": card(), **SETTINGS, "reps": a.reps, "warmup": a.warmup, "input": "numpy float32 clips",
           "timer": "host clock around calls that return numpy", "workloads": []}
    for name in a.workloads.split(","):
        res["workloads"].append(measure(name, a.reps, a.warmup))
        print(json.dumps(res["workloads"][-1]), file=sys.stderr, flush=True)
    res["every_clip_equal_to_the_loop"] = all(w["per_clip_equal"] for w in res["workloads"])
    line = json.dumps(res)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
