#!/usr/bin/env python
"""decorrelate_batch against a per-clip loop through the single-clip API, on the same clips in the same run (GPU box).

    python tools/bench_decorrelate_batch.py [--reps 10] [--warmup 3] [--out FILE]

Workloads (all 44.1 kHz stereo float32, seeded):
  a  512 clips of 5-15 s, one default VelvetNoise (MS, rms_normalize); ~1.8 GB in, larger than L2
  b  the same clips with 64 distinct log_distribution_strength values, one VelvetNoise per clip
  c  the config-2 chain (velvet noise + LR Haas, float64 out)
  d  normalizer=None: the one-launch path
  e  8 clips of 10 minutes: few long columns for the order-exact sums of squares
  f  workload a numpy in / numpy out, against a copy ceiling measured in the same run (same bytes up and down, no
     kernel; chunked, uploads and downloads overlapped on two streams)
a-e take CUDA tensors and are timed with CUDA events; f is timed with the host clock around calls that end in a
synchronise.  Each timing: `warmup` untimed calls, then median and best of `reps`.  Parity with the single-clip call
is checked byte for byte on a few clips of every workload before timing.  Prints one JSON line (and writes it to
--out), with the card's name and power limit read in the same run."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from vndecorrelate_b200 import _native as N  # noqa: E402
from vndecorrelate_b200 import decorrelation as D  # noqa: E402
from vndecorrelate_b200 import runtime as R  # noqa: E402

FS = 44100


def dram_bytes_per_output_sample(rms: bool, out_bytes: int, packed_from_list: bool) -> dict:
    """Bytes the library's kernels must move per output sample (2 per row), from the kernel sequence:
    no normaliser: read x, write out; rms: read x, write the float32 scratch | read x and the scratch (sums) | read the
    scratch, write out.  Packing a list of CUDA tensors (torch.cat) adds a read and a write of x."""
    row = 8 + 2 * out_bytes if not rms else 8 + 8 + 8 + 8 + 8 + 2 * out_bytes
    pack = 16 if packed_from_list else 0
    return {"kernels": row / 2, "with_packing": (row + pack) / 2}


def card() -> dict:
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(q[0]), float(q[1])
    except Exception as e:  # noqa: BLE001 - recorded, not hidden
        info["power_limit_w"] = f"unavailable ({e})"
    return info


def time_events(fn, warmup: int, reps: int) -> tuple[float, float]:
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        fn()
        e.record()
        e.synchronize()
        ts.append(s.elapsed_time(e))
    return float(np.median(ts)), float(np.min(ts))


def time_host(fn, warmup: int, reps: int) -> tuple[float, float]:
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts)), float(np.min(ts))


def same(a, b) -> bool:
    a = a.cpu().numpy() if torch.is_tensor(a) else a
    b = b.cpu().numpy() if torch.is_tensor(b) else b
    return a.dtype == b.dtype and a.shape == b.shape and np.ascontiguousarray(a).tobytes() == np.ascontiguousarray(b).tobytes()


def launches(fn) -> int:
    torch.cuda.synchronize()
    before = N.launch_count()
    fn()
    torch.cuda.synchronize()
    return N.launch_count() - before


def run(name, clips, decs, args, *, rms, out_bytes, host=False):
    per = decs if isinstance(decs, list) else [decs] * len(clips)
    batch = lambda: D.decorrelate_batch(clips, decs)  # noqa: E731

    def loop():
        for c, d in zip(clips, per):
            d(c)

    got = batch()
    for i in sorted({0, 1, len(clips) // 2, len(clips) - 1}):
        assert same(got[i], per[i](clips[i])), f"{name}: clip {i} differs from the single-clip call"
    del got
    rows = int(sum(c.shape[0] for c in clips))
    timer = time_host if host else time_events
    b_med, b_best = timer(batch, args.warmup, args.reps)
    l_med, l_best = timer(loop, args.warmup, args.reps)
    rec = {
        "workload": name, "n_clips": len(clips), "rows": rows, "out_dtype": "float64" if out_bytes == 8 else "float32",
        "input": "numpy" if host else "cuda tensors", "timer": "host clock + synchronise" if host else "CUDA events",
        "batch_ms_median": b_med, "batch_ms_best": b_best, "loop_ms_median": l_med, "loop_ms_best": l_best,
        "loop_over_batch_median": l_med / b_med, "loop_over_batch_best": l_best / b_best,
        "batch_gsamples_per_s": 2 * rows / b_med / 1e6, "loop_gsamples_per_s": 2 * rows / l_med / 1e6,
        "launches_per_batch": launches(batch), "launches_per_loop": launches(loop),
        "dram_bytes_per_output_sample": dram_bytes_per_output_sample(rms, out_bytes, not host),
        "parity_checked_clips": 4,
    }
    print(json.dumps(rec), file=sys.stderr, flush=True)
    return rec


def copy_ceiling(nbytes: int, args) -> dict:
    """The same bytes up and down through page-locked buffers, no kernel: 64 MB chunks, uploads on one stream and
    downloads on another, so the two directions overlap as the library's pipeline overlaps them."""
    chunk = 64 << 20
    src = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dst = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    dev = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
    up, down = torch.cuda.Stream(), torch.cuda.Stream()

    def once():
        for o in range(0, nbytes, chunk):
            e = torch.cuda.Event()
            with torch.cuda.stream(up):
                dev[o:o + chunk].copy_(src[o:o + chunk], non_blocking=True)
                e.record(up)
            with torch.cuda.stream(down):
                down.wait_event(e)
                dst[o:o + chunk].copy_(dev[o:o + chunk], non_blocking=True)
        up.synchronize()
        down.synchronize()

    med, best = time_host(once, args.warmup, args.reps)
    return {"bytes_each_way": nbytes, "ms_median": med, "ms_best": best}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip", default="", help="workloads to leave out, e.g. 'f'")
    args = ap.parse_args()
    assert args.reps >= 10 and args.warmup >= 3, "at least 3 warm-ups and 10 timed calls"
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(0)
    rec = {"card": card(), "reps": args.reps, "warmup": args.warmup, "workloads": []}

    rng = np.random.default_rng(2024)
    lengths = rng.integers(5 * FS, 15 * FS + 1, size=512)
    rows = int(lengths.sum())
    offs = np.concatenate([[0], np.cumsum(lengths)])
    g = torch.Generator(device="cuda").manual_seed(1)
    big = torch.randn((rows, 2), generator=g, device="cuda") * 0.3
    clips = [big[int(a):int(b)] for a, b in zip(offs[:-1], offs[1:])]
    vn = D.VelvetNoise(sample_rate_hz=FS, seed=1)
    W = rec["workloads"]
    if "a" not in args.skip:
        W.append(run("a", clips, vn, args, rms=True, out_bytes=4))
    if "b" not in args.skip:
        kappas = np.linspace(0.0, 1.5, 64)
        filters = [D.VelvetNoise(sample_rate_hz=FS, seed=1, log_distribution_strength=float(k)) for k in kappas]
        W.append(run("b", clips, [filters[i % 64] for i in range(len(clips))], args, rms=True, out_bytes=4))
    if "c" not in args.skip:
        chain = (D.SignalChain(sample_rate_hz=FS).velvet_noise(duration_seconds=0.03, num_impulses=30, log_distribution_strength=1.0, seed=1)
                 .haas_effect(delay_time_seconds=0.02, mode="LR"))
        W.append(run("c", clips, chain, args, rms=True, out_bytes=8))
    if "d" not in args.skip:
        W.append(run("d", clips, D.VelvetNoise(sample_rate_hz=FS, seed=1, normalizer=None), args, rms=False, out_bytes=4))
    if "e" not in args.skip:
        long_rows = 8 * 600 * FS
        longs = torch.randn((long_rows, 2), generator=g, device="cuda") * 0.3
        W.append(run("e", [longs[i * 600 * FS:(i + 1) * 600 * FS] for i in range(8)], vn, args, rms=True, out_bytes=4))
        del longs
    if "f" not in args.skip:
        host = big.cpu().numpy()
        del clips, big
        torch.cuda.empty_cache()
        np_clips = [host[int(a):int(b)] for a, b in zip(offs[:-1], offs[1:])]
        R.set_pinned_pool_cap(4 << 30)  # results of both arms on page-locked memory (the default cap is 512 MB)
        f = run("f", np_clips, vn, args, rms=True, out_bytes=4, host=True)
        f["pinned_pool_cap_bytes"] = 4 << 30
        f["copy_ceiling"] = copy_ceiling(rows * 8, args)
        f["batch_over_copy_ceiling_median"] = f["batch_ms_median"] / f["copy_ceiling"]["ms_median"]
        W.append(f)
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
