#!/usr/bin/env python
"""BlockDecorrelator: live signals block by block, one launch per step (GPU box).

    python tools/bench_stream_blocks.py [--steps 50] [--warmup 10] [--out profiles/r08_block_step.json] [--skip abcde]

Workloads (48 kHz, stereo float32 blocks, seeded; default VelvetNoise with normalizer=None):
  a  1 signal, 512-frame blocks: step latency with CUDA tensors (CUDA events) and with numpy in / numpy out (host clock
     around a step that ends in a synchronise), and the real-time factor (block duration over step time)
  b  1024 signals x 512-frame blocks: the step, a loop of 1024 single-signal BlockDecorrelators on the same blocks, and
     decorrelate_batch on 1024 clips of the same 512 frames (the offline ceiling: no history, no look-ahead held back).
     The kernel alone (CUDA events around vnd_vn_block_step_dev on packed buffers, in steady state) against its byte
     model: 8 B read and 8 B written per frame, plus the history - H frames of 8 B read and written per signal - and
     the A frames of look-ahead each signal's tile reads from it
  c  1024 signals with ragged blocks of 0-4096 frames, about one in ten signals finishing and restarting at each step
  d  b with a VelvetNoise + LR HaasEffect chain: 2 launches per step
  e  b with one HaasEffect per signal (delays 0-30 ms, channels and modes mixed), Haas alone
Every signal of every workload is checked byte for byte against the one-shot call on its concatenated input before
timing.  Each timing: `warmup` untimed steps, then median and best of `steps` steps.  Prints one JSON line (and writes it
to --out), with the card's name and power limit read in the same run."""
import argparse
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

FS = 48000
BLOCK = 512


def vn(seed=1):
    return D.VelvetNoise(sample_rate_hz=FS, normalizer=None, seed=seed)


def blocks_of(n, lengths, rng, device="cuda"):
    """One float32 stereo block per signal, cut from one packed tensor (so the step reads them in place)."""
    total = int(np.sum(lengths))
    x = torch.from_numpy((rng.standard_normal((max(total, 1), 2)) * 0.3).astype(np.float32)).to(device)
    at, out = 0, []
    for L in lengths:
        out.append(x[at:at + int(L)])
        at += int(L)
    return out


def check(name, dec, n, schedule, finals, rng) -> int:
    """Runs the schedule (lengths per step and signal, final flags) and compares every finished signal with the one-shot
    call on its concatenated input; returns the number of signals checked."""
    b = D.BlockDecorrelator(dec, n)
    decs = dec if isinstance(dec, list) else [dec] * n
    ins = [[] for _ in range(n)]
    outs = [[] for _ in range(n)]
    checked = 0
    for lengths, fin in zip(schedule, finals):
        blocks = blocks_of(n, lengths, rng)
        res = b.process(blocks, final=list(fin))
        for i in range(n):
            ins[i].append(blocks[i])
            outs[i].append(res[i])
            if fin[i]:
                want = decs[i](torch.cat(ins[i]))
                assert same(torch.cat(outs[i]), want), f"{name}: signal {i} differs from the one-shot call"
                ins[i], outs[i] = [], []
                checked += 1
    return checked


def steady(dec, n, args, rng, *, np_in=False, lengths=None):
    """Median and best step time of a BlockDecorrelator fed `lengths` frames per signal (BLOCK by default)."""
    b = D.BlockDecorrelator(dec, n)
    lengths = np.full(n, BLOCK) if lengths is None else lengths
    pool = [blocks_of(n, lengths, rng) for _ in range(4)]
    if np_in:
        pool = [[x.cpu().numpy() for x in p] for p in pool]
    it = iter(range(10**9))
    step = lambda: b.process(pool[next(it) % 4])  # noqa: E731
    timer = time_host if np_in else time_events
    med, best = timer(step, args.warmup, args.steps)
    return med, best, launches(step), b


def kernel_alone(b, args) -> dict:
    """vnd_vn_block_step_dev alone in steady state (every signal has received 16 blocks and gets one more)."""
    n, H = b.n_signals, b._H_vn
    st = b._dev
    lib = N.lib()
    offs = np.arange(n + 1, dtype=np.int64) * BLOCK
    recv = np.full(n, 16 * BLOCK, np.int64)
    emit = np.maximum(recv - b.latency_frames, 0)
    oo = np.arange(n + 1, dtype=np.int64) * BLOCK
    meta = torch.from_numpy(np.concatenate([offs, recv, emit, oo])).cuda()
    m = meta.data_ptr()
    x = torch.zeros((n * BLOCK, 2), dtype=torch.float32, device="cuda")
    y = torch.empty_like(x)
    h_in, h_out = st["vn"]
    stream = torch.cuda.current_stream().cuda_stream
    import ctypes as C

    def launch():
        N.check(lib.vnd_vn_block_step_dev(x.data_ptr(), n * BLOCK, m, n, m + 8 * (n + 1), m + 8 * (2 * n + 1), st["prog_of"].data_ptr(),
                                          C.byref(st["program"]), C.byref(b._ep), h_in.data_ptr(), h_out.data_ptr(), H, m + 8 * (3 * n + 1),
                                          n * BLOCK, y.data_ptr(), stream), "vnd_vn_block_step_dev")

    med, best = time_events(launch, args.warmup, args.steps)
    A = int(b.latency_frames.max())
    model = n * BLOCK * 16 + n * H * 16 + n * A * 8
    return {"model_bytes": model, "model": "16 B per frame + 16 B per history frame + 8 B per look-ahead frame read", "history_frames": H,
            "kernel_ms_median": med, "kernel_ms_best": best, "kernel_model_tb_per_s_median": model / med / 1e9,
            "kernel_model_tb_per_s_best": model / best / 1e9}


def workload_many(name, dec, args, rng, loop_dec=None) -> dict:
    n = 1024
    sched = [np.full(n, BLOCK)] * 5
    fins = [np.zeros(n, bool)] * 4 + [np.ones(n, bool)]
    checked = check(name, dec, n, sched, fins, rng)
    med, best, nl, b = steady(dec, n, args, rng)
    rec = {"workload": name, "n_signals": n, "block_frames": BLOCK, "input": "cuda tensors", "timer": "CUDA events",
           "step_ms_median": med, "step_ms_best": best, "launches_per_step": nl, "parity_checked_signals": checked,
           "frames_per_s_median": n * BLOCK / med * 1e3, "realtime_factor_median": (BLOCK / FS * 1e3) / med}
    if name == "b":
        singles = [D.BlockDecorrelator(dec, 1) for _ in range(n)]
        pool = [blocks_of(n, np.full(n, BLOCK), rng) for _ in range(4)]
        it = iter(range(10**9))

        def loop():
            p = pool[next(it) % 4]
            for s, x in zip(singles, p):
                s.process([x])

        l_med, l_best = time_events(loop, args.warmup, args.steps)
        clips = pool[0]
        off_med, off_best = time_events(lambda: D.decorrelate_batch(clips, dec), args.warmup, args.steps)
        rec.update({"loop_ms_median": l_med, "loop_ms_best": l_best, "loop_over_step_median": l_med / med, "launches_per_loop": launches(loop),
                    "decorrelate_batch_ms_median": off_med, "decorrelate_batch_ms_best": off_best,
                    "step_over_decorrelate_batch_median": med / off_med, "kernel": kernel_alone(b, args)})
    print(json.dumps(rec), file=sys.stderr, flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r08_block_step.json"))
    ap.add_argument("--skip", default="")
    args = ap.parse_args()
    torch.cuda.init()
    rec = {"tool": "bench_stream_blocks", "card": card(), "sample_rate_hz": FS, "steps": args.steps, "warmup": args.warmup, "workloads": []}
    W = rec["workloads"]
    rng = np.random.default_rng(0)
    if "a" not in args.skip:
        dec = vn()
        checked = check("a", dec, 1, [np.full(1, BLOCK)] * 9 + [np.full(1, 77)], [np.zeros(1, bool)] * 9 + [np.ones(1, bool)], rng)
        t_med, t_best, nl, _ = steady(dec, 1, args, rng)
        h_med, h_best, _, _ = steady(dec, 1, args, rng, np_in=True)
        block_ms = BLOCK / FS * 1e3
        a = {"workload": "a", "n_signals": 1, "block_frames": BLOCK, "block_ms": block_ms, "parity_checked_signals": checked,
             "tensor_step_ms_median": t_med, "tensor_step_ms_best": t_best, "tensor_timer": "CUDA events",
             "numpy_step_ms_median": h_med, "numpy_step_ms_best": h_best, "numpy_timer": "host clock around a synchronised step",
             "realtime_factor_tensor_median": block_ms / t_med, "realtime_factor_numpy_median": block_ms / h_med, "launches_per_step": nl}
        print(json.dumps(a), file=sys.stderr, flush=True)
        W.append(a)
    if "b" not in args.skip:
        W.append(workload_many("b", vn(), args, rng))
    if "c" not in args.skip:
        n = 1024
        dec = vn()
        sched = [rng.integers(0, 4097, size=n) for _ in range(12)]
        fins = [rng.random(n) < 0.1 for _ in range(11)] + [np.ones(n, bool)]
        checked = check("c", dec, n, sched, fins, rng)
        b = D.BlockDecorrelator(dec, n)
        pool = [(blocks_of(n, s, rng), list(f)) for s, f in zip(sched[:8], fins[:8])]
        it = iter(range(10**9))

        def step():
            blocks, fin = pool[next(it) % 8]
            b.process(blocks, final=fin)

        med, best = time_events(step, args.warmup, args.steps)
        frames = float(np.mean([s.sum() for s in sched[:8]]))
        c = {"workload": "c", "n_signals": n, "block_frames": "uniform 0-4096", "final_rate": 0.1, "input": "cuda tensors", "timer": "CUDA events",
             "step_ms_median": med, "step_ms_best": best, "mean_frames_per_step": frames, "frames_per_s_median": frames / med * 1e3,
             "launches_per_step": launches(step), "parity_checked_signals": checked}
        print(json.dumps(c), file=sys.stderr, flush=True)
        W.append(c)
    if "d" not in args.skip:
        chain = D.SignalChain(sample_rate_hz=FS).velvet_noise(normalizer=None, seed=1).haas_effect()
        W.append(workload_many("d", chain, args, rng))
    if "e" not in args.skip:
        r = np.random.default_rng(5)
        haases = [D.HaasEffect(sample_rate_hz=FS, delay_time_seconds=float(r.uniform(0, 0.03)), delayed_channel=int(r.integers(-2, 2)),
                               mode="MS" if i % 2 else "LR", width=0.7 if i % 3 == 0 else None) for i in range(1024)]
        W.append(workload_many("e", haases, args, rng))
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
