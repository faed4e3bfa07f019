#!/usr/bin/env python
"""haas_effect_batch against a per-clip loop of HaasEffect.decorrelate, on the same clips in the same run (GPU box).

    python tools/bench_haas_effect_batch.py [--reps 10] [--warmup 3] [--out FILE] [--skip abcde]

Workloads (44.1 kHz stereo float32 clips, seeded; every clip a tensor or array of its own, so the batch packs them):
  a  512 clips of 5-15 s, per-clip delays uniform in [0, 0.03 s], LR; ~1.8 GB in, 3.6 GB out, larger than L2
  b  the clips of a, MS, width 0.7, delayed channels 0 / 1 / -1 / -2 in turn
  c  4096 clips of 0.5-2 s, per-clip delays, LR
  d  the clips and effects of a, numpy in / numpy out, against a copy ceiling measured in the same run (the same bytes
     up and down through page-locked buffers, no kernel, the two directions overlapped)
  e  the clips of a, one VelvetNoise per clip (64 strengths) and the Haas effects of a: decorrelate_batch then
     haas_effect_batch, against a loop of the per-clip SignalChain(VelvetNoise, HaasEffect) - one fused pass per clip
a-c and e take CUDA tensors and are timed with CUDA events; d with the host clock around calls that end in a
synchronise.  a-c also time the kernel alone (CUDA events around the one vnd_haas_batch_dev launch on packed buffers)
and report its model bytes - 8 B read per input frame, 16 B written per output frame - per second, as a fraction of a
device-to-device copy moving the same bytes (half read, half written) timed in the same run.  Each timing: `warmup`
untimed calls, then median and best of `reps`.  Every clip of every workload is checked byte for byte against the
single call before timing.  Prints one JSON line (and writes it to --out), with the card's name and power limit read in
the same run."""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import torch  # noqa: E402
from bench_decorrelate_batch import card, launches, time_events, time_host  # noqa: E402

from vndecorrelate_b200 import _native as N  # noqa: E402
from vndecorrelate_b200 import decorrelation as D  # noqa: E402
from vndecorrelate_b200 import runtime as R  # noqa: E402

FS = 44100


def same_bits(a, b) -> bool:
    if torch.is_tensor(a):
        return a.dtype == b.dtype and a.shape == b.shape and torch.equal(a.contiguous().view(torch.int64), b.contiguous().view(torch.int64))
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(np.ascontiguousarray(a).view(np.uint64), np.ascontiguousarray(b).view(np.uint64))


def check_all(name, got, want_of, n):
    for i in range(n):
        assert same_bits(got[i], want_of(i)), f"{name}: clip {i} differs from the single call"
    return n


def kernel_alone(clips, effects, args) -> dict:
    """The one launch of vnd_haas_batch_dev on buffers packed beforehand, and a device copy of the same bytes."""
    n = len(clips)
    table = D._haas_table(effects, clips, shared=False)
    delays = table["delay"].astype(np.int64)
    lengths = np.array([c.shape[0] for c in clips], dtype=np.int64)
    offsets, out_offsets = D._haas_offsets(lengths, delays)
    rows, out_rows = int(offsets[-1]), int(offsets[-1] + delays.sum())
    xp = D._pack_tensors(clips, rows, clips[0].device)
    out = torch.empty((out_rows, 2), dtype=torch.float64, device="cuda")
    meta = torch.from_numpy(np.concatenate([table.view(np.int64), offsets, out_offsets])).cuda()
    m = meta.data_ptr()
    lib = N.lib()
    stream = torch.cuda.current_stream().cuda_stream

    def launch():
        N.check(lib.vnd_haas_batch_dev(xp.data_ptr(), rows, m + 32 * n, n, m, m + 32 * n + 8 * (n + 1), out_rows, out.data_ptr(), stream),
                "vnd_haas_batch_dev")

    k_med, k_best = time_events(launch, args.warmup, args.reps)
    model = 8 * rows + 16 * out_rows
    src = torch.empty(model // 2, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    c_med, c_best = time_events(lambda: dst.copy_(src), args.warmup, args.reps)
    del src, dst
    return {
        "rows": rows, "out_rows": out_rows, "model_bytes": model, "kernel_ms_median": k_med, "kernel_ms_best": k_best,
        "kernel_model_tb_per_s_median": model / k_med / 1e9, "kernel_model_tb_per_s_best": model / k_best / 1e9,
        "d2d_copy_ms_median": c_med, "d2d_copy_ms_best": c_best, "d2d_copy_tb_per_s_median": model / c_med / 1e9,
        "kernel_over_copy_rate_median": c_med / k_med, "kernel_over_copy_rate_best": c_best / k_best,
    }


def run(name, clips, effects, args, *, host=False, kernel=True):
    batch = lambda: D.haas_effect_batch(clips, effects)  # noqa: E731

    def loop():
        for c, h in zip(clips, effects):
            h.decorrelate(c)

    checked = check_all(name, batch(), lambda i: effects[i].decorrelate(clips[i]), len(clips))
    timer = time_host if host else time_events
    b_med, b_best = timer(batch, args.warmup, args.reps)
    l_med, l_best = timer(loop, args.warmup, args.reps)
    rec = {
        "workload": name, "n_clips": len(clips), "input": "numpy" if host else "cuda tensors",
        "timer": "host clock + synchronise" if host else "CUDA events",
        "batch_ms_median": b_med, "batch_ms_best": b_best, "loop_ms_median": l_med, "loop_ms_best": l_best,
        "loop_over_batch_median": l_med / b_med, "loop_over_batch_best": l_best / b_best,
        "launches_per_batch": launches(batch), "launches_per_loop": launches(loop), "parity_checked_clips": checked,
    }
    if kernel:
        rec["kernel_alone"] = kernel_alone(clips, effects, args)
    print(json.dumps(rec), file=sys.stderr, flush=True)
    return rec


def copy_ceiling(up_bytes: int, down_bytes: int, args) -> dict:
    """up_bytes uploaded and down_bytes downloaded through page-locked buffers, no kernel: 64 MB chunks, uploads on one
    stream and downloads on another, so the two directions overlap as the library's pipeline overlaps them."""
    chunk = 64 << 20
    src = torch.empty(up_bytes, dtype=torch.uint8, pin_memory=True)
    dst = torch.empty(down_bytes, dtype=torch.uint8, pin_memory=True)
    dev_in = torch.empty(up_bytes, dtype=torch.uint8, device="cuda")
    dev_out = torch.empty(down_bytes, dtype=torch.uint8, device="cuda")
    up, down = torch.cuda.Stream(), torch.cuda.Stream()
    n = max(-(-up_bytes // chunk), 1)
    dchunk = -(-down_bytes // n)

    def once():
        for k in range(n):
            e = torch.cuda.Event()
            with torch.cuda.stream(up):
                dev_in[k * chunk:(k + 1) * chunk].copy_(src[k * chunk:(k + 1) * chunk], non_blocking=True)
                e.record(up)
            with torch.cuda.stream(down):
                down.wait_event(e)
                dst[k * dchunk:(k + 1) * dchunk].copy_(dev_out[k * dchunk:(k + 1) * dchunk], non_blocking=True)
        up.synchronize()
        down.synchronize()

    med, best = time_host(once, args.warmup, args.reps)
    return {"bytes_up": up_bytes, "bytes_down": down_bytes, "ms_median": med, "ms_best": best}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None)
    ap.add_argument("--skip", default="", help="workloads to leave out, e.g. 'de'")
    args = ap.parse_args()
    assert args.reps >= 10 and args.warmup >= 3, "at least 3 warm-ups and 10 timed calls"
    assert torch.cuda.is_available(), "this benchmark needs a CUDA device"
    torch.cuda.set_device(0)
    rec = {"card": card(), "reps": args.reps, "warmup": args.warmup, "workloads": []}
    W = rec["workloads"]

    rng = np.random.default_rng(2024)
    lengths = rng.integers(5 * FS, 15 * FS + 1, size=512)
    delays = rng.uniform(0.0, 0.03, size=512)
    g = torch.Generator(device="cuda").manual_seed(1)
    clips = [torch.randn((int(L), 2), generator=g, device="cuda") * 0.3 for L in lengths]
    lr = [D.HaasEffect(sample_rate_hz=FS, delay_time_seconds=float(d), mode="LR") for d in delays]
    if "a" not in args.skip:
        W.append(run("a", clips, lr, args))
    if "b" not in args.skip:
        ms = [D.HaasEffect(sample_rate_hz=FS, delay_time_seconds=float(d), mode="MS", width=0.7, delayed_channel=(0, 1, -1, -2)[i % 4])
              for i, d in enumerate(delays)]
        W.append(run("b", clips, ms, args))
    if "c" not in args.skip:
        c_lengths = rng.integers(FS // 2, 2 * FS + 1, size=4096)
        c_clips = [torch.randn((int(L), 2), generator=g, device="cuda") * 0.3 for L in c_lengths]
        c_eff = [D.HaasEffect(sample_rate_hz=FS, delay_time_seconds=float(d), mode="LR") for d in rng.uniform(0.0, 0.03, size=4096)]
        W.append(run("c", c_clips, c_eff, args))
        del c_clips
    if "e" not in args.skip:
        kappas = np.linspace(0.0, 1.5, 64)
        vns = [D.VelvetNoise(sample_rate_hz=FS, seed=1, log_distribution_strength=float(kappas[i % 64])) for i in range(len(clips))]
        chains = []
        for vn, h in zip(vns, lr):
            ch = D.SignalChain(sample_rate_hz=FS, lazy=False)
            ch._decorrelators = [vn, h]  # the chain a user builds with .velvet_noise(...).haas_effect(...), with these instances
            chains.append(ch)
        batch = lambda: D.haas_effect_batch(D.decorrelate_batch(clips, vns), lr)  # noqa: E731

        def loop():
            for c, ch in zip(clips, chains):
                ch(c)

        checked = check_all("e", batch(), lambda i: chains[i](clips[i]), len(clips))
        b_med, b_best = time_events(batch, args.warmup, args.reps)
        l_med, l_best = time_events(loop, args.warmup, args.reps)
        e = {"workload": "e", "n_clips": len(clips), "input": "cuda tensors", "timer": "CUDA events",
             "batch": "haas_effect_batch(decorrelate_batch(clips, vns), haas_effects)", "loop": "SignalChain(vn_i, haas_i)(clip_i), fused",
             "batch_ms_median": b_med, "batch_ms_best": b_best, "loop_ms_median": l_med, "loop_ms_best": l_best,
             "loop_over_batch_median": l_med / b_med, "loop_over_batch_best": l_best / b_best,
             "launches_per_batch": launches(batch), "launches_per_loop": launches(loop), "parity_checked_clips": checked}
        print(json.dumps(e), file=sys.stderr, flush=True)
        W.append(e)
    if "d" not in args.skip:
        np_clips = [c.cpu().numpy() for c in clips]
        del clips
        torch.cuda.empty_cache()
        R.set_pinned_pool_cap(8 << 30)  # results of both arms on page-locked memory (the default cap is 512 MB)
        d = run("d", np_clips, lr, args, host=True, kernel=False)
        rows = int(sum(c.shape[0] for c in np_clips))
        out_rows = rows + int(sum(h.delay_len_samples for h in lr))
        d["pinned_pool_cap_bytes"] = 8 << 30
        d["copy_ceiling"] = copy_ceiling(rows * 8, out_rows * 16, args)
        d["batch_over_copy_ceiling_median"] = d["batch_ms_median"] / d["copy_ceiling"]["ms_median"]
        W.append(d)
    line = json.dumps(rec)
    print(line)
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
