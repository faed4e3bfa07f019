#!/usr/bin/env python
"""optimize_haas_delay_batch against a loop of optimize_haas_delay over the same clips, in the same run (GPU box).

    python tools/bench_haas_batch.py [--reps 5] [--warmup 1] [--workloads a,b,c,d] [--gpus N] [--out FILE]

Workloads (44.1 kHz, max_delay_seconds=0.03, seeded coloured stereo noise as in config 5, numpy float32 clips in):
  a  64 clips x 30 s, equal lengths, grid 400 (the default)
  b  64 clips of 5-60 s, grid 400
  c  workload a at grid 1024 (config-5 scale)
  d  512 clips of 2-6 s, grid 400
Every clip's delay from the batch is first checked to equal the loop's (==, not approximately).  Then each arm runs
`warmup` untimed calls and `reps` timed ones (host clock around calls that return numpy, so they end in a synchronise);
median and best are reported, with the grid stage and the refinement timed separately inside each call: for the batch,
the grid stage is argument checks + packing + upload + the grid launch + scoring; for the loop, the sum of the
per-clip grid_scan calls.  The grid kernel alone is also timed with CUDA events (one pair launch over all clips x grid
delays) and given as frame-evaluations per second (sum of clip frames x grid / kernel time).  --gpus N additionally
runs workload b over N ranks (NCCL, one process per GPU) and reports the wall time and the sha256 of the delay array
next to that of the one-rank run.  Prints one JSON line, with the card's name and power limit read in the same run, and
also writes it to FILE when --out is given (nothing is written otherwise)."""
import argparse
import contextlib
import hashlib
import io
import json
import os
import socket
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

FS = 44100
MAXD = 0.03
KW = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)


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
    rng = np.random.default_rng({"a": 1, "b": 2, "c": 1, "d": 4}[name])
    if name in ("a", "c"):
        lengths = [30 * FS] * 64
    elif name == "b":
        lengths = rng.integers(5 * FS, 60 * FS + 1, 64).tolist()
    else:
        lengths = rng.integers(2 * FS, 6 * FS + 1, 512).tolist()
    grid = 1024 if name == "c" else 400
    return [O.coloured_clip(i, int(n)) for i, n in enumerate(lengths)], grid


def run_batch(clips, grid):
    marks = {}

    class TimedBank(OPT._HaasClipBank):
        def grid_scores(self, delays):
            out = super().grid_scores(delays)
            marks["grid_end"] = time.perf_counter()
            return out

    with contextlib.redirect_stdout(io.StringIO()):
        t0 = time.perf_counter()
        taus, info = OPT.optimize_haas_delay_batch(input_signals=clips, sample_rate_hz=FS, max_delay_seconds=MAXD, grid_size=grid, details=True,
                                                  _bank_factory=TimedBank)
        t1 = time.perf_counter()
    return taus, {"total_s": t1 - t0, "grid_s": marks["grid_end"] - t0, "refine_s": t1 - marks["grid_end"], "launches": info["launches_local"],
                  "evaluations": info["evaluations_local"], "brent_rounds": info["rounds_local"],
                  "minimisers": int(sum(len(m) for m in info["local_minima"]))}


def run_loop(clips, grid):
    acc = {"grid_s": 0.0, "evaluations": 0}
    grid_scan, partials = OPT.grid_scan, OPT.haas_objective_partials

    def timed_grid_scan(*a, **k):
        s = time.perf_counter()
        r = grid_scan(*a, **k)
        acc["grid_s"] += time.perf_counter() - s
        return r

    def counted_partials(c, delays):
        acc["evaluations"] += len(delays)
        return partials(c, delays)

    OPT.grid_scan, OPT.haas_objective_partials = timed_grid_scan, counted_partials
    try:
        with contextlib.redirect_stdout(io.StringIO()):
            before = N.launch_count()
            t0 = time.perf_counter()
            taus = np.array([OPT.optimize_haas_delay(input_signal=c, sample_rate_hz=FS, max_delay_seconds=MAXD, grid_size=grid) for c in clips])
            t1 = time.perf_counter()
            launches = N.launch_count() - before
    finally:
        OPT.grid_scan, OPT.haas_objective_partials = grid_scan, partials
    return taus, {"total_s": t1 - t0, "grid_s": acc["grid_s"], "refine_s": t1 - t0 - acc["grid_s"], "launches": launches,
                  "evaluations": acc["evaluations"]}


def grid_kernel_ms(clips, grid, reps):
    """The grid stage's one pair launch alone, CUDA events, median of `reps` after one warm-up."""
    bank = OPT._HaasClipBank(clips, KW)
    delays = np.array([round(t * FS) for t in np.linspace(0.0, MAXD, grid).tolist()], dtype=np.int32)
    pc = torch.from_numpy(np.repeat(np.arange(len(clips), dtype=np.int32), grid)).to(bank.device)
    pd = torch.from_numpy(np.tile(delays, len(clips))).to(bank.device)
    OPT.haas_objective_pair_partials(bank.x, bank.offs_dev, pc, pd)
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        OPT.haas_objective_pair_partials(bank.x, bank.offs_dev, pc, pd)
        b.record()
        b.synchronize()
        ms.append(a.elapsed_time(b))
    return float(np.median(ms))


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
           "frames_max": int(max(frames)), "per_clip_equal": equal, "clips_equal": int(np.sum(got == want)),
           "delays_sha256": hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest()}
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
    kms = grid_kernel_ms(clips, grid, max(reps, 5))
    row["grid_kernel_ms"] = kms
    row["grid_kernel_frame_evaluations_per_s"] = sum(frames) * grid / kms * 1e3
    row["grid_stage_frame_evaluations_per_s"] = {"batch": sum(frames) * grid / row["batch"]["grid_s"]["median"],
                                                 "loop": sum(frames) * grid / row["loop"]["grid_s"]["median"]}
    return row


def _rank_main(rank, world, port, result_dir):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["VND_DEVICE"] = str(rank)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        clips, grid = workload("b")
        kw = dict(input_signals=clips, sample_rate_hz=FS, max_delay_seconds=MAXD, grid_size=grid)
        with contextlib.redirect_stdout(io.StringIO()):
            OPT.optimize_haas_delay_batch(**kw)  # warm-up
            walls = []
            for _ in range(3):
                dist.barrier()
                t0 = time.perf_counter()
                taus = OPT.optimize_haas_delay_batch(**kw)
                dist.barrier()
                walls.append(time.perf_counter() - t0)
        if rank == 0:
            json.dump({"wall_s_median": float(np.median(walls)), "wall_s_best": float(np.min(walls)),
                       "delays_sha256": hashlib.sha256(np.ascontiguousarray(taus).tobytes()).hexdigest()}, open(os.path.join(result_dir, "multi.json"), "w"))
    finally:
        dist.destroy_process_group()


def multi_gpu(n, one_rank_sha):
    import tempfile

    import torch.multiprocessing as mp

    visible = torch.cuda.device_count()
    if visible < n:
        return {"gpus": n, "measured": False, "reason": f"not measured: {visible} GPU(s) visible"}
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    with tempfile.TemporaryDirectory() as d:
        mp.spawn(_rank_main, args=(n, port, d), nprocs=n, join=True)
        res = json.load(open(os.path.join(d, "multi.json")))
    return {"gpus": n, "measured": True, "workload": "b", **res, "one_rank_sha256": one_rank_sha, "same_as_one_rank": res["delays_sha256"] == one_rank_sha}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--workloads", default="a,b,c,d")
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    torch.cuda.set_device(0)
    res = {"card": card(), "sample_rate_hz": FS, "max_delay_seconds": MAXD, "reps": a.reps, "warmup": a.warmup, "input": "numpy float32 clips",
           "timer": "host clock around calls that return numpy", "round2_grid_kernel_frame_evaluations_per_s": 2.6e11, "workloads": []}
    for name in a.workloads.split(","):
        res["workloads"].append(measure(name, a.reps, a.warmup))
        print(json.dumps(res["workloads"][-1]), file=sys.stderr, flush=True)
    if a.gpus > 1:
        one = next((w["delays_sha256"] for w in res["workloads"] if w["workload"] == "b"), None)
        if one is None:
            got, _ = run_batch(*workload("b"))
            one = hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest()
        res["multi_gpu"] = multi_gpu(a.gpus, one)
    line = json.dumps(res)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")
    print(line)


if __name__ == "__main__":
    main()
