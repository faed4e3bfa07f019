#!/usr/bin/env python
"""BlockConvolver: live multichannel signals convolved block by block, one launch per step (GPU box).

    python tools/bench_stream_convolve.py [--steps 50] [--warmup 10] [--out profiles/r09_block_convolve.json] [--skip abcde]

Workloads (seeded float32 blocks unless noted; "config 3 filter" = 48 kHz, 0.03 s, 30 impulses, every channel filtered,
LR, normalizer=None, seed 1; "config 4 filter" = 96 kHz, 0.3 s, 300 impulses, the same otherwise):
  a  1 signal x 64 channels, config 3 filter, 512-frame blocks
  b  1 signal x 4096 channels, config 3 filter, 512-frame blocks
  c  1 signal x 1024 channels, config 4 filter, 1024-frame blocks
  d  64 signals x 16 channels, config 3 filter with seed 1 + i for signal i, 256-frame blocks
  e  a with float64 blocks (float64 arithmetic)
For each: every signal checked byte for byte against the one-shot convolve on its concatenated input first; the step,
after ceil(A / L) + 1 untimed priming steps so that every timed step emits L frames per signal (asserted), on CUDA tensors (CUDA events) and on numpy in / numpy out (host clock around a step that ends in a synchronise), median
and best of `steps` steps after `warmup`; the real-time factor (block duration over step time); launches per step; the
"re-convolve" loop a user would otherwise write (per signal: convolve(cat(last A frames, block)), keep the ready rows) on
the same tensor blocks; the one-shot convolve of the same total frames per signal (16 blocks, the offline ceiling, per
block); and the kernel alone (CUDA events around vnd_fir_block_step_dev in steady state) against its byte model: per
signal and channel, the block read, the A frames of look-ahead staged, the float32 output written, and H history frames
read and written, at the compute dtype's size.  Prints one JSON line (and writes it to --out), with the card's name and
power limit read in the same run."""
import argparse
import ctypes as C
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
from bench_decorrelate_batch import card, launches, same, time_events, time_host  # noqa: E402

from vndecorrelate_b200 import _native as N  # noqa: E402
from vndecorrelate_b200 import decorrelation as D  # noqa: E402

WORKLOADS = {  # name: (signals, channels, config, block frames, dtype)
    "a": (1, 64, 3, 512, np.float32),
    "b": (1, 4096, 3, 512, np.float32),
    "c": (1, 1024, 4, 1024, np.float32),
    "d": (64, 16, 3, 256, np.float32),
    "e": (1, 64, 3, 512, np.float64),
}


def filt(config, channels, seed=1):
    fs, dur, imp = (48000, 0.03, 30) if config == 3 else (96000, 0.3, 300)
    return D.VelvetNoise(sample_rate_hz=fs, duration_seconds=dur, num_impulses=imp, num_outs=channels, filtered_channels=tuple(range(channels)),
                         mode="LR", normalizer=None, seed=seed)


def blocks_of(n, L, C_, dtype, rng):
    x = rng.standard_normal((n * L, C_)) * 0.3
    t = torch.from_numpy(x.astype(dtype)).cuda()
    return [t[i * L:(i + 1) * L] for i in range(n)]


def check(filters, n, C_, L, dtype, rng) -> int:
    """Eight steps of L frames, then a final step of L // 3 + 1 frames; every signal against the one-shot convolve."""
    b = D.BlockConvolver(filters, n)
    per = filters if isinstance(filters, list) else [filters] * n
    ins = [[] for _ in range(n)]
    outs = [[] for _ in range(n)]
    for s in range(9):
        blocks = blocks_of(n, L if s < 8 else L // 3 + 1, C_, dtype, rng)
        res = b.process(blocks, final=s == 8)
        for i in range(n):
            ins[i].append(blocks[i])
            outs[i].append(res[i])
    for i in range(n):
        assert same(torch.cat(outs[i]), per[i].convolve(torch.cat(ins[i]))), f"signal {i} differs from the one-shot convolve"
    return n


def primed_blocks(A: int, L: int) -> int:
    """Blocks after which every step of a signal emits L frames: received >= A + L before the step."""
    return -(-A // L) + 1


def kernel_alone(b, L, dtype, args) -> dict:
    """vnd_fir_block_step_dev alone in steady state: every signal has received primed_blocks(max A, L) blocks, so each
    emits all L frames of the one more it gets."""
    n, H, C_ = b.n_signals, b._H, b.num_outs
    st = b._dev
    A = b.latency_frames
    offs = np.arange(n + 1, dtype=np.int64) * L
    recv = np.full(n, primed_blocks(int(A.max()), L) * L, np.int64)
    emit = recv - A
    assert np.all(emit >= L)
    meta = torch.from_numpy(np.concatenate([offs, recv, emit, offs])).cuda()
    m = meta.data_ptr()
    tdt = torch.float64 if dtype == np.float64 else torch.float32
    x = torch.zeros((n * L, C_), dtype=tdt, device="cuda")
    y = torch.empty((n * L, C_), dtype=torch.float32, device="cuda")
    h_in, h_out = st["history"]
    stream = torch.cuda.current_stream().cuda_stream
    lib = N.lib()

    def launch():
        N.check(lib.vnd_fir_block_step_dev(x.data_ptr(), N.VND_F64 if dtype == np.float64 else N.VND_F32, n * L, C_, m, n, m + 8 * (n + 1),
                                           m + 8 * (2 * n + 1), st["prog_of"].data_ptr(), C.byref(st["program"]), h_in.data_ptr(), h_out.data_ptr(),
                                           H, m + 8 * (3 * n + 1), n * L, y.data_ptr(), stream), "vnd_fir_block_step_dev")

    med, best = time_events(launch, args.warmup, args.steps)
    e = np.dtype(dtype).itemsize
    model = int(C_ * (n * L * (e + 4) + int(A.sum()) * e + 2 * n * H * e))
    return {"model_bytes": model, "model": "per signal and channel: block read + A look-ahead frames + float32 out + H history frames read and written",
            "history_frames": H, "kernel_ms_median": med, "kernel_ms_best": best, "kernel_model_tb_per_s_median": model / med / 1e9,
            "kernel_model_tb_per_s_best": model / best / 1e9, "kernel_launches": launches(launch)}


def workload(name, args, rng) -> dict:
    n, C_, config, L, dtype = WORKLOADS[name]
    filters = [filt(config, C_, seed=1 + i) for i in range(n)] if name == "d" else filt(config, C_)
    per = filters if isinstance(filters, list) else [filters] * n
    fs = per[0].sample_rate_hz
    checked = check(filters, n, C_, L, dtype, rng)

    pool = [blocks_of(n, L, C_, dtype, rng) for _ in range(4)]
    np_pool = [[x.cpu().numpy() for x in p] for p in pool]
    prime = primed_blocks(int(D.BlockConvolver(filters, n).latency_frames.max()), L)

    def stepper(blocks_pool):
        """A step function over a BlockConvolver past its latency: each timed step must emit L frames per signal."""
        b = D.BlockConvolver(filters, n)
        for k in range(prime):
            b.process(blocks_pool[k % 4])
        it = iter(range(prime, 10**9))

        def step():
            res = b.process(blocks_pool[next(it) % 4])
            assert all(r.shape[0] == L for r in res), "a timed step emitted fewer than L frames"

        return b, step

    b, step = stepper(pool)
    t_med, t_best = time_events(step, args.warmup, args.steps)
    nl = launches(step)
    _, np_step = stepper(np_pool)
    h_med, h_best = time_host(np_step, args.warmup, args.steps)

    A = [int(a) for a in b.latency_frames]
    hist = [torch.zeros((a, C_), dtype=pool[0][0].dtype, device="cuda") for a in A]
    it3 = iter(range(10**9))

    def loop():
        p = pool[next(it3) % 4]
        for i in range(n):
            x = torch.cat([hist[i], p[i]])
            per[i].convolve(x)[:L]
            hist[i] = x[x.shape[0] - A[i]:]

    l_med, l_best = time_events(loop, args.warmup, args.steps)
    whole = [torch.cat([pool[k % 4][i] for k in range(16)]) for i in range(n)]
    off = lambda: [per[i].convolve(whole[i]) for i in range(n)]  # noqa: E731
    o_med, o_best = time_events(off, args.warmup, max(args.steps // 5, 3))
    block_ms = L / fs * 1e3
    rec = {"workload": name, "n_signals": n, "channels": C_, "filter": f"config {config}", "sample_rate_hz": fs, "block_frames": L,
           "dtype": np.dtype(dtype).name, "latency_frames_max": max(A), "parity_checked_signals": checked, "primed_blocks": prime,
           "tensor_step_ms_median": t_med, "tensor_step_ms_best": t_best, "tensor_timer": "CUDA events",
           "numpy_step_ms_median": h_med, "numpy_step_ms_best": h_best, "numpy_timer": "host clock around a synchronised step",
           "block_ms": block_ms, "realtime_factor_tensor_median": block_ms / t_med, "realtime_factor_numpy_median": block_ms / h_med,
           "launches_per_step": nl, "reconvolve_loop_ms_median": l_med, "reconvolve_loop_ms_best": l_best,
           "reconvolve_over_step_median": l_med / t_med, "launches_per_reconvolve_loop": launches(loop),
           "oneshot_16_blocks_ms_median": o_med, "oneshot_per_block_ms_median": o_med / 16, "kernel": kernel_alone(b, L, dtype, args)}
    print(json.dumps(rec), file=sys.stderr, flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r09_block_convolve.json"))
    ap.add_argument("--skip", default="")
    ap.add_argument("--variant", default="default build", help="what library this run times, recorded in the JSON (e.g. an A/B build)")
    args = ap.parse_args()
    torch.cuda.init()
    rec = {"tool": "bench_stream_convolve", "card": card(), "variant": args.variant, "steps": args.steps, "warmup": args.warmup, "workloads": []}
    rng = np.random.default_rng(0)
    for name in WORKLOADS:
        if name not in args.skip:
            rec["workloads"].append(workload(name, args, rng))
    line = json.dumps(rec)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
