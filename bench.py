#!/usr/bin/env python
"""Benchmark of the velvet-noise decorrelation hot path (BASELINE.json metric:
"Gsamples/s out (ch x samples) ... + % HBM roofline vs CPU numpy").

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--configs 1,2,3,4,5] [--dump-outputs DIR]

Every timed loop on the GPU (kernels, end-to-end calls and the copy probe) runs K steps; the CPU figures beside
them are bounded samples (one pass, or the best of three), and in --impl reference a step is one such sample of
config 3.  --dump-outputs DIR writes what the timed steps computed in their last step: config 3's
and config 4's output slabs as fixed seeded samples (sample_slab), configs 1 and 2 whole, config 5's strengths and
score matrix; the inputs are seeded, so two builds run with the same arguments can be compared output for output.

The JSON line's headline (`metric`, `value`, `roofline`, `e2e`, `cpu_baseline`) is BASELINE config 3, the one
the metric is quoted on: 4096 channels x 10 min @ 48 kHz fp32 with one 30 ms / 30-impulse velvet filter per
channel, partitioned by channel over the 8 GPUs of a box = 512 channels x 28.8 M samples per GPU (59 GB in +
59 GB out, resident in HBM).  Scaling is WEAK: every rank holds one such shard (N = 8 is the full config), the
tap table is generated once for all 4096 channels and sliced per rank, no data-path collective.  A step is one
pass of the FIR over the rank's shard.

`configs` carries the other four BASELINE configs, each with its own value, roofline, end-to-end figure through
the Python call BASELINE.json names, and the CPU path next to it:

  cfg1  VelvetNoise(0.03 s, 30 impulses, seed 1).decorrelate(viola.wav)          (replicas only)
  cfg2  SignalChain velvet_noise + haas_effect(0.02 s, LR) on guitar.wav, fused     (replicas only)
  cfg4  1024 ch x 10 min @ 96 kHz, 300 impulses / 0.3 s: 128 channels per GPU       (weak scaling)
  cfg5  optimize_velvet_noise: 1024 strengths x 64 clips x 30 s, grid + refinement, clips sharded over the N
        GPUs, ONE NCCL all-gather of the float32 score matrix                       (strong scaling)

`value` numbers are timed with CUDA events, inputs resident in HBM; `e2e` numbers go through the public Python
API with HOST buffers (page-locked numpy arrays in, numpy arrays out), copies inside the timed region;
`cpu_baseline` / `--impl reference` time the reference package itself (baseline/_ref, when present) or the numpy
port of its loops (oracle/vnd_oracle.py, pinned to the reference's golden vectors) on the host cores.
"""

from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

FS = 48000
FRAMES = 28_800_000  # 10 min @ 48 kHz
TOTAL_CHANNELS = 4096
CHANNELS_PER_GPU = 512
METRIC = "Gsamples/s out (ch x samples), velvet-noise sparse FIR, cfg3 shard per GPU"
UNIT = "Gsamples/s"
BYTES_PER_SAMPLE = 8  # algorithmic: 4 B read + 4 B written per output sample (SURVEY.md section 8d)

CFG4_FS, CFG4_FRAMES, CFG4_TOTAL_CHANNELS, CFG4_CHANNELS_PER_GPU = 96000, 57_600_000, 1024, 128
CFG5_CLIPS, CFG5_FRAMES, CFG5_GRID = 64, 1_440_000, 1024
OBJ_KW = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)
AUDIO = os.path.join(ROOT, "tests", "golden", "audio")


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md, 6.65 TB/s)"


def load_wav(name: str) -> np.ndarray:
    from scipy.io import wavfile

    _, x = wavfile.read(os.path.join(AUDIO, name + ".wav"))
    return np.ascontiguousarray(x)


def coloured_clip(index: int, frames: int) -> np.ndarray:
    """Config-5 clip (SURVEY.md section 8d): low-passed mid plus 0.3 x low-passed side, peak 0.5, float32 (frames, 2);
    host-generated so that the CPU and the GPU arm see identical bytes."""
    from scipy.signal import lfilter

    rng = np.random.default_rng(1000 + index)
    m = lfilter([0.02], [1, -0.98], rng.standard_normal(frames))
    s = 0.3 * lfilter([0.02], [1, -0.98], rng.standard_normal(frames))
    x = np.column_stack((m + s, m - s))
    return (x / np.max(np.abs(x)) * 0.5).astype(np.float32)


# --------------------------------------------------------------------------------------------
# clocks sampler (nvidia-smi, during the timed region)
# --------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu_index = gpu_index
        self.proc = None
        self.lines: list[str] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu_index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, power, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [s.strip() for s in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(names, f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(power)), "samples": len(sm),
                "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------
# CPU arm: the reference package (baseline/_ref) when it is there, else the numpy port (oracle)
# --------------------------------------------------------------------------------------------
_REF = None


def reference_modules():
    """(decorrelation, optimization) of the UNMODIFIED reference from baseline/_ref (a git-ignored copy of its
    package that __graft_entry__.build() makes from the checkout BASELINE.json's `reference_path` names), or None."""
    global _REF
    if _REF is None:
        _REF = False
        p = os.path.join(ROOT, "baseline", "_ref")
        if os.path.isdir(os.path.join(p, "vndecorrelate")):
            sys.path.insert(0, p)
            try:
                import vndecorrelate.decorrelation as RD
                import vndecorrelate.optimization as RO

                _REF = (RD, RO)
            except Exception:
                _REF = False
    return _REF or None


def cpu_kind() -> str:
    return "reference" if reference_modules() else "port"


def _silent(fn, *a, **k):
    """The reference prints progress lines; keep stdout for the JSON line."""
    import contextlib
    import io

    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


def _cpu_fir_worker(args):
    """One process: the class-path FIR on a C-order (frames, channels) float32 slab; returns seconds for the FIR alone."""
    seed, channels, frames, fs, dur, nimp = args
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((frames, channels)) * 0.1).astype(np.float32)  # C-order (frames, channels): the reference's layout
    ref = reference_modules()
    if ref:
        vn = ref[0].VelvetNoise(sample_rate_hz=fs, duration_seconds=dur, num_impulses=nimp, num_outs=channels,
                                filtered_channels=tuple(range(channels)), mode="LR", normalizer=None, seed=1)
        t0 = time.perf_counter()
        y = vn.convolve(x)
        dt = time.perf_counter() - t0
    else:
        from oracle import vnd_oracle as O

        taps = O.class_taps(sample_rate_hz=fs, duration_seconds=dur, num_impulses=nimp, num_outs=channels, filtered_channels=tuple(range(channels)), seed=1)
        t0 = time.perf_counter()
        y = O.fir_class_order(x, taps, O.DEFAULT_ENVELOPE, channels)
        dt = time.perf_counter() - t0
    return dt, float(y[0, 0])


def cpu_fir_rate(workers: int, channels_per_worker: int, frames: int, fs=FS, dur=0.03, nimp=30, repeats: int = 1):
    """Gsamples/s of the CPU FIR with `workers` processes (slowest worker's time), best of `repeats`."""
    import multiprocessing as mp

    best = None
    if workers == 1:
        for r in range(repeats):
            dt, _ = _cpu_fir_worker((100 + r, channels_per_worker, frames, fs, dur, nimp))
            best = dt if best is None else min(best, dt)
    else:
        ctx = mp.get_context("fork")
        with ctx.Pool(workers) as pool:
            for r in range(repeats):
                res = pool.map(_cpu_fir_worker, [(100 + r * workers + w, channels_per_worker, frames, fs, dur, nimp) for w in range(workers)])
                dt = max(d for d, _ in res)
                best = dt if best is None else min(best, dt)
    return workers * channels_per_worker * frames / best / 1e9, best


def cpu_cfg1(repeats=3):
    x = load_wav("viola")
    ref = reference_modules()
    if ref:
        vn = ref[0].VelvetNoise(sample_rate_hz=44100, duration_seconds=0.03, num_impulses=30, seed=1)
        fn = lambda: vn.decorrelate(x)  # noqa: E731
    else:
        from oracle import vnd_oracle as O

        taps = O.class_taps(sample_rate_hz=44100, seed=1)
        fn = lambda: O.vn_decorrelate(x, taps)  # noqa: E731
    best = min(_timed(fn) for _ in range(repeats))
    return {"value": x.size / best / 1e6, "unit": "Msamples/s", "ms": best * 1e3, "cores": 1, "kind": cpu_kind(),
            "sample": f"the whole file, {x.shape[0]} x 2 float32, best of {repeats}"}


def cpu_cfg2(repeats=3):
    x = load_wav("guitar")
    ref = reference_modules()
    if ref:
        chain = ref[0].SignalChain(sample_rate_hz=44100).velvet_noise(duration_seconds=0.03, num_impulses=30, log_distribution_strength=1.0,
                                                                      seed=1).haas_effect(delay_time_seconds=0.02, mode="LR")
        fn = lambda: chain(x)  # noqa: E731
    else:
        from oracle import vnd_oracle as O

        taps = O.class_taps(sample_rate_hz=44100, seed=1)
        fn = lambda: O.haas(O.vn_decorrelate(x, taps), sample_rate_hz=44100, delay_time_seconds=0.02)  # noqa: E731
    out = fn()
    best = min(_timed(fn) for _ in range(repeats))
    return {"value": out.size / best / 1e6, "unit": "Msamples/s", "ms": best * 1e3, "cores": 1, "kind": cpu_kind(),
            "sample": f"the whole file, {x.shape[0]} x 2 float32 -> {out.shape[0]} x 2 float64, best of {repeats}"}


def _cpu_obj_worker(args):
    clip_index, kappas, frames = args
    x = coloured_clip(clip_index, frames)
    ref = reference_modules()
    t0 = time.perf_counter()
    if ref:
        RD, RO = ref
        for k in kappas:
            d = RD.VelvetNoise(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, log_distribution_strength=float(k), normalizer=None,
                               filtered_channels=(0,), mode="LR", seed=1)
            _silent(RO.symmetry_aware_objective, x, d, **OBJ_KW)
    else:
        from oracle import vnd_oracle as O

        O.vn_grid_scores(x, kappas, sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, seed=1)
    return time.perf_counter() - t0


def cpu_cfg5(workers: int, kappas_per_worker: int = 8):
    """(clip, strength) objective evaluations per second on 30 s clips: `workers` processes x one clip x a few strengths."""
    import multiprocessing as mp

    ks = np.linspace(0.0, 1.0, kappas_per_worker)
    if workers == 1:
        dt = _cpu_obj_worker((0, ks, CFG5_FRAMES))
    else:
        with mp.get_context("fork").Pool(workers) as pool:
            dt = max(pool.map(_cpu_obj_worker, [(w, ks, CFG5_FRAMES) for w in range(workers)]))
    return {"value": workers * kappas_per_worker / dt, "unit": "evaluations/s", "cores": workers, "kind": cpu_kind(),
            "sample": f"{workers} process(es) x 1 clip x {kappas_per_worker} strengths x {CFG5_FRAMES} frames, symmetry_aware_objective ({dt:.1f} s)"}


def _timed(fn) -> float:
    t0 = time.perf_counter()
    fn()
    return time.perf_counter() - t0


def workload_config(args) -> dict:
    """Identical in both arms (the driver compares the dicts)."""
    return {
        "workload": f"BASELINE configs[2]: {TOTAL_CHANNELS} ch x 10 min @ 48 kHz fp32, 30 ms / 30-impulse velvet FIR per channel; "
                    f"{args.channels_per_gpu} channels x {args.frames} frames per GPU (channel-sharded)",
        "channels_per_gpu": args.channels_per_gpu, "frames": args.frames, "sample_rate_hz": FS, "num_impulses": 30, "duration_seconds": 0.03,
        "partitioning": "channels; one 4096-channel tap table generated once (seed 1) and sliced per rank; no collective",
        "l2": "inputs (tens of GB per GPU) are far larger than the 126 MB L2; no explicit flush",
    }


def run_reference(args) -> None:
    """The reference's own CPU implementation on all host cores, bounded samples of the same workloads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    workers = max(1, cores)
    ch, frames = 4, 960_000  # 20 s @ 48 kHz per worker and step
    sample = f"{workers} processes x {ch} channels x {frames} frames (20 s @ 48 kHz), C-order (frames, channels) fp32, per step"
    warm = args.warmup
    for _ in range(warm):
        cpu_fir_rate(workers, ch, frames)
    t_total = 0.0
    steps = args.steps
    for _ in range(steps):
        _, dt = cpu_fir_rate(workers, ch, frames)
        t_total += dt
    value = workers * ch * frames * steps / t_total / 1e9
    configs = {}
    want = _parse_configs(args.configs)
    try:
        if 1 in want:
            configs["cfg1"] = {"cpu_baseline": cpu_cfg1()}
        if 2 in want:
            configs["cfg2"] = {"cpu_baseline": cpu_cfg2()}
        if 4 in want:
            r4, s4 = cpu_fir_rate(workers, 1, 480_000, fs=CFG4_FS, dur=0.3, nimp=300)
            configs["cfg4"] = {"cpu_baseline": {"value": r4, "unit": UNIT, "cores": workers, "kind": cpu_kind(),
                                                "sample": f"{workers} processes x 1 channel x 480000 frames (5 s @ 96 kHz), 300 impulses / 0.3 s ({s4:.1f} s)"}}
        if 5 in want:
            configs["cfg5"] = {"cpu_baseline": cpu_cfg5(workers, 4)}
    except Exception as exc:  # report, do not hide
        configs["error"] = repr(exc)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": steps, "warmup": warm,
        "ms_per_step": 1e3 * t_total / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": workload_config(args),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": workers, "kind": cpu_kind(), "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "configs": configs,
        "note": "CPU arm: every step is a bounded sample of the workload (the full shard would take hours on the host)",
    }
    print(json.dumps(line))


def _parse_configs(text: str) -> set[int]:
    return {int(t) for t in text.replace(" ", "").split(",") if t}


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
class Env:
    """torch / torch.distributed plumbing of one rank."""

    def __init__(self):
        import torch
        import torch.distributed as dist

        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py --impl b200 needs a CUDA device (there is no CPU fallback)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.stream = torch.cuda.current_stream(self.dev)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, v: float) -> float:
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t[0])

    def sum_over_ranks(self, v: float) -> float:
        if self.world == 1:
            return float(v)
        t = self.torch.tensor([v], dtype=self.torch.float64, device=self.dev)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t[0])

    def timed_events(self, fn, steps: int):
        """Per-step device times (ms) of `fn`, CUDA events on the launching stream, barrier + synchronize on both sides."""
        torch = self.torch
        self.barrier()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
        ev[0].record(self.stream)
        for i in range(steps):
            fn()
            ev[i + 1].record(self.stream)
        torch.cuda.synchronize()
        per_step = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
        total = self.max_over_ranks(ev[0].elapsed_time(ev[-1]))
        self.barrier()
        return per_step, total

    def timed_wall(self, fn, steps: int) -> float:
        """Wall seconds of `steps` calls of a host-API function (max over ranks), synchronised on both sides."""
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        self.torch.cuda.synchronize()
        dt = self.max_over_ranks(time.perf_counter() - t0)
        self.barrier()
        return dt


def device_slab(env: Env, channels: int, frames: int, seed: int):
    """randn(seed) * 0.1 float32 (channels, frames) on the device, generated in channel groups."""
    torch = env.torch
    x = torch.empty((channels, frames), dtype=torch.float32, device=env.dev)
    gen = torch.Generator(device=env.dev).manual_seed(seed)
    grp = max(1, min(channels, (1 << 28) // max(frames, 1)))
    for g0 in range(0, channels, grp):
        x[g0: min(channels, g0 + grp)].normal_(0.0, 1.0, generator=gen).mul_(0.1)
    torch.cuda.synchronize()
    return x


def sample_slab(y, window: int = 1 << 15, points: int = 1 << 19) -> dict:
    """A fixed sample (seed 0) of a device (channels, frames) float32 output, for --dump-outputs: on up to 16 channels
    (the first and the last among them) the first and the last `window` frames and two windows at seeded positions,
    as (channels, 4, window); and `points` samples at seeded positions of the whole slab.  ~10 MB."""
    import torch

    Cy, L = y.shape
    rng = np.random.default_rng(0)
    chans = sorted({0, Cy - 1} | set(rng.choice(Cy, size=min(Cy, 14), replace=False).tolist()))
    W = min(window, L)
    starts = [0, L - W] + rng.integers(0, L - W + 1, 2).tolist()
    windows = torch.stack([torch.stack([y[c, s: s + W] for s in starts]) for c in chans])
    flat = torch.from_numpy(rng.integers(0, Cy * L, min(points, Cy * L))).to(y.device)
    return {"windows": windows.cpu().numpy(), "points": y.reshape(-1)[flat].cpu().numpy()}


def write_outputs(path: str, outputs: dict) -> None:
    """DIR/<name>.npy for every array, float32 or float64, at most 64 MB in all."""
    arrays = {}
    for name, a in outputs.items():
        a = np.ascontiguousarray(a)
        arrays[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    total = sum(a.nbytes for a in arrays.values())
    if total > 64_000_000:
        raise SystemExit(f"bench: --dump-outputs would write {total} bytes, more than 64 MB")
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def oracle_windows(x, y, taps, envelope, windows, halo: int) -> bool:
    """GPU output y[ch, a:b] against the oracle on the excerpt x[ch, a : b + halo] for every (ch, a, b) window."""
    from oracle import vnd_oracle as O

    L = x.shape[1]
    ok = True
    for ch, a, b in windows:
        a, b = max(0, a), min(L, b)
        m = min(L, b + halo)
        col = x[ch, a:m].cpu().numpy()
        want = O.fir_class_order(np.stack((col, col), axis=1), [taps[ch], []], envelope, 2)[: b - a, 0]
        got = y[ch, a:b].cpu().numpy()
        ok = ok and want.tobytes() == got.tobytes()
    return ok


def copy_probe(env: Env, nbytes: int, steps: int) -> dict:
    """Ceiling of any host-buffer path on this box: `nbytes` up and `nbytes` down at the same time between page-locked
    host memory and the device, on two streams, all ranks at once (max over ranks)."""
    torch = env.torch
    n = nbytes // 4
    hx = torch.empty(n, dtype=torch.float32, pin_memory=True)
    hy = torch.empty(n, dtype=torch.float32, pin_memory=True)
    dx = torch.empty(n, dtype=torch.float32, device=env.dev)
    dy = torch.zeros(n, dtype=torch.float32, device=env.dev)
    s_up, s_down = torch.cuda.Stream(env.dev), torch.cuda.Stream(env.dev)

    def once():
        with torch.cuda.stream(s_up):
            dx.copy_(hx, non_blocking=True)
        with torch.cuda.stream(s_down):
            hy.copy_(dy, non_blocking=True)
        s_up.synchronize()
        s_down.synchronize()

    once()
    dt = env.timed_wall(once, steps) / steps
    return {"seconds": dt, "gbs_each_way": nbytes / dt / 1e9, "bytes_each_way": nbytes}


def run_cfg3(env: Env, args, lib, N, R, VelvetNoise, C):
    torch = env.torch
    vn = VelvetNoise(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, num_outs=TOTAL_CHANNELS,
                     filtered_channels=tuple(range(TOTAL_CHANNELS)), mode="LR", normalizer=None, seed=1)
    Cg, L = args.channels_per_gpu, args.frames
    c0 = (env.rank * Cg) % TOTAL_CHANNELS
    if c0 + Cg > TOTAL_CHANNELS:
        c0 = TOTAL_CHANNELS - Cg
    prog = vn.tap_program(L).slice_channels(c0, c0 + Cg)
    x = device_slab(env, Cg, L, 1234 + env.rank)
    y = torch.empty((Cg, L), dtype=torch.float32, device=env.dev)
    sx, sy, ps = R.torch_signal(x.t()), R.torch_signal(y.t()), R.device_program(prog, env.dev)

    def step():
        N.check(lib.vnd_sparse_fir_dev(C.byref(sx), C.byref(sy), C.byref(ps), env.stream.cuda_stream), "vnd_sparse_fir_dev")

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    torch.cuda.synchronize()

    # parity spot check (outside the timed region): the first and the last 2^16 frames (the hand-over from the
    # tensor-memory kernel to the tail kernel lies in the latter) and a window across the first run boundary of the
    # persistent kernel, on the first and the last channel
    parity = "skipped"
    if env.rank == 0:
        from oracle import vnd_oracle as O

        taps_all = O.class_taps(sample_rate_hz=FS, num_outs=TOTAL_CHANNELS, filtered_channels=tuple(range(TOTAL_CHANNELS)), seed=1)
        taps = {ch: taps_all[c0 + ch] for ch in (0, Cg - 1)}
        n = min(L, 1 << 16)
        plan = (C.c_int * 3)()
        boundary = None
        if hasattr(lib, "vnd_debug_fir_plan") and lib.vnd_debug_fir_plan(C.c_longlong(L), Cg, prog.halo, plan) == 0 and plan[1] > 1:
            boundary = plan[0] * plan[2]  # tiles per run x frames per tile
        windows = []
        for ch in (0, Cg - 1):
            windows += [(ch, 0, n), (ch, L - n, L)]
            if boundary:
                windows.append((ch, boundary - (1 << 14), boundary + (1 << 14)))
        if not oracle_windows(x, y, taps, O.DEFAULT_ENVELOPE, windows, prog.halo):
            raise SystemExit("bench: GPU output differs from the oracle; refusing to report a number")
        parity = (f"bit-exact vs oracle on channels 0 and {Cg - 1}: frames [0, {n}), the last {n} (tensor-memory -> tail hand-over)"
                  + (f" and 2^15 frames across the run boundary at frame {boundary}" if boundary else ""))

    sampler = ClockSampler(env.local_rank)
    sampler.start()
    launches0 = N.launch_count()
    per_step, total_ms = env.timed_events(step, args.steps)
    launches = int(env.sum_over_ranks(N.launch_count() - launches0))
    clocks = sampler.stop()
    value = env.world * Cg * L * args.steps / (total_ms * 1e-3) / 1e9
    outputs = {f"cfg3_y_{k}": v for k, v in sample_slab(y).items()} if args.dump_outputs else {}

    kernel_ms = float(np.mean(per_step))
    achieved = BYTES_PER_SAMPLE * Cg * L / (kernel_ms * 1e-3) / 1e9
    peak, peak_src = measured_peak_gbs()
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "fir_tmem_traffic.json")
    if os.path.exists(tpath):
        try:
            traffic = json.load(open(tpath))["dram_bytes_per_sample"] * Cg * L
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "kernel": "fir_tmem_kernel (tensor-memory Hankel rows + tcgen05.ld gathers, FADD2, warp-specialised, tensor-map TMA); the last "
                          "~1.5 tiles of every channel run on fir_window_kernel in a second launch inside the same step",
                "kernel_ms": kernel_ms, "peak_source": peak_src,
                "note": "HBM is not the binding resource: every (output, tap) pair moves one word from on-chip memory to a register. Per lane "
                        "quarter a tile is the sum of the tensor-memory phase (22 taps; bound by the quarter's TMEM read path, ~54 B/clk per "
                        "scheduler) and the shared-memory phase (8 far taps: a per-warp instruction chain), which cannot overlap because the "
                        "quarter's TMEM rows are refilled as a whole. See DESIGN.md section 4 and profiles/r02_summary.md"}

    # end to end through the PYTHON API with host buffers: VelvetNoise.convolve on a page-locked C-order (frames, channels)
    # numpy slab (the reference's layout), numpy result; upload / transposes / kernel / download overlapped inside the call
    e2e = None
    try:
        Ce = min(args.e2e_channels, Cg)
        R.set_pinned_pool_cap(max(2 * Ce * L * 4 + (64 << 20), 512 << 20))
        vne = VelvetNoise(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, num_outs=Ce, filtered_channels=tuple(range(Ce)), mode="LR",
                          normalizer=None, seed=1)
        hx = R.PinnedArray((L, Ce))
        grp = max(1, (1 << 26) // Ce)
        for t0 in range(0, L, grp):  # the same synthetic signal, laid out (frames, channels)
            hx.array[t0: t0 + grp] = x[:Ce, t0: t0 + grp].t().contiguous().cpu().numpy()
        out = vne.convolve(hx.array)  # warm-up: arena, result pool
        from oracle import vnd_oracle as O

        et = O.class_taps(sample_rate_hz=FS, num_outs=Ce, filtered_channels=tuple(range(Ce)), seed=1)
        n = 1 << 14
        head = O.fir_class_order(np.ascontiguousarray(hx.array[: n + 2048]), et, O.DEFAULT_ENVELOPE, Ce)[:n]
        tail = O.fir_class_order(np.ascontiguousarray(hx.array[L - n:]), et, O.DEFAULT_ENVELOPE, Ce)
        same = bool(head.tobytes() == np.ascontiguousarray(out[:n]).tobytes() and tail.tobytes() == np.ascontiguousarray(out[L - n:]).tobytes())
        del out
        e_steps = args.steps
        holder = []

        def e2e_step():
            holder.clear()
            holder.append(vne.convolve(hx.array))

        dt = env.timed_wall(e2e_step, e_steps)
        probe = copy_probe(env, Ce * L * 4, e_steps)
        ceiling = env.world * Ce * L / probe["seconds"] / 1e9
        e2e = {"value": env.world * Ce * L * e_steps / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": Ce * L * 4, "d2h_bytes_per_step": Ce * L * 4,
               "steps": e_steps, "channels": Ce, "frames": L,
               "api": "vndecorrelate_b200.VelvetNoise.convolve(numpy (frames, channels) C-order, page-locked) -> numpy; vnd_sparse_fir_host "
                      "overlaps upload / transpose / kernel / transpose / download in chunks of frames",
               "matches_oracle": same,
               "copy_ceiling": {"value": ceiling, "unit": UNIT, "gbs_each_way_per_gpu": probe["gbs_each_way"],
                                "what": "the same bytes up and down at once between page-locked memory and the device, no kernel, all ranks together"},
               "frac_of_copy_ceiling": (env.world * Ce * L * e_steps / dt / 1e9) / ceiling}
        # the same call on ordinary (pageable) numpy memory, 8 channels: the slab goes through the context's page-locked
        # staging ring (helper threads) instead of being copied by DMA directly
        try:
            Cp = min(8, Ce)
            vnp = VelvetNoise(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, num_outs=Cp, filtered_channels=tuple(range(Cp)), mode="LR",
                              normalizer=None, seed=1)
            px = np.ascontiguousarray(hx.array[:, :Cp])
            holder.clear()
            holder.append(vnp.convolve(px))

            def pageable_step():
                holder.clear()  # the result block goes back to the pool before the next call takes it
                holder.append(vnp.convolve(px))

            dtp = env.timed_wall(pageable_step, args.steps)
            e2e["pageable_input"] = {"value": env.world * Cp * L * args.steps / dtp / 1e9, "unit": UNIT, "channels": Cp,
                                     "note": "ordinary numpy input (staged through page-locked memory by a helper thread), pooled page-locked result"}
            del px
        except Exception as exc:
            e2e["pageable_input"] = {"error": repr(exc)}
        del hx, holder
        R.trim_pinned_pool(0)
    except Exception as exc:  # report, do not hide
        e2e = {"value": None, "unit": UNIT, "error": repr(exc)}
    del x, y
    torch.cuda.empty_cache()
    return dict(value=value, total_ms=total_ms, warm=warm, clocks=clocks, launches=launches, roofline=roofline, e2e=e2e, parity=parity,
                outputs=outputs)


def run_cfg12(env: Env, args, which: int, lib, N, R, api):
    """Single stereo files: latency-bound, replicas only.  value = device-resident (CUDA tensor in / out), e2e = numpy in / out."""
    torch = env.torch
    if which == 1:
        x = load_wav("viola")
        vn = api.VelvetNoise(sample_rate_hz=44100, duration_seconds=0.03, num_impulses=30, seed=1)
        call = vn.decorrelate
        out_bytes = 4
        want_sha = "8ba98663842a1593a8bc6b4d622c04820a33ae7849be10d72752be268a9b3e54"  # SURVEY.md Appendix C (reference output)
        name = "VelvetNoise(sample_rate_hz=44100, duration_seconds=0.03, num_impulses=30, seed=1).decorrelate(viola.wav)"
    else:
        x = load_wav("guitar")
        chain = api.SignalChain(sample_rate_hz=44100).velvet_noise(duration_seconds=0.03, num_impulses=30, log_distribution_strength=1.0,
                                                                   seed=1).haas_effect(delay_time_seconds=0.02, mode="LR")
        call = chain
        out_bytes = 8
        want_sha = "f420f1120b056d083fe976cd8f9aded0c2cee68d33a5976aaf30973df6cf82bb"
        name = "SignalChain(44100).velvet_noise(0.03 s, 30, strength 1.0, seed 1).haas_effect(0.02 s, LR)(guitar.wav), one fused pass"
    got = call(x)
    parity = "sha256 of the output equals the reference's" if hashlib.sha256(np.ascontiguousarray(got).tobytes()).hexdigest() == want_sha else "MISMATCH"
    if parity == "MISMATCH":
        raise SystemExit(f"bench cfg{which}: output differs from the reference's")
    xd = torch.from_numpy(x).to(env.dev)
    for _ in range(5):
        call(xd)
    torch.cuda.synchronize()
    steps = args.steps
    last = [None]

    def step():
        last[0] = call(xd)

    launches0 = N.launch_count()
    per_step, _ = env.timed_events(step, steps)
    launches = (N.launch_count() - launches0) // steps
    ms = float(np.median(per_step))
    samples_out = got.size
    for _ in range(5):
        call(x)
    e_ms = sorted(_timed(lambda: call(x)) for _ in range(steps))[steps // 2] * 1e3
    peak, _ = measured_peak_gbs()
    bytes_algo = x.size * 4 + samples_out * out_bytes
    return {
        "workload": name, "scaling": "replicas only (a single stereo file)", "value": samples_out / (ms * 1e-3) / 1e6, "unit": "Msamples/s",
        "ms": ms, "steps": steps, "kernel_launches_per_call": int(launches),
        "roofline": {"bound": "hbm", "achieved": bytes_algo / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": bytes_algo / (ms * 1e-3) / 1e9 / peak,
                     "traffic": None, "note": f"{bytes_algo / 1e6:.1f} MB per call: latency-bound, the launches of one call take longer than the HBM time"},
        "e2e": {"value": samples_out / (e_ms * 1e-3) / 1e6, "unit": "Msamples/s", "ms": e_ms, "h2d_bytes_per_step": int(x.nbytes), "d2h_bytes_per_step": int(got.nbytes),
                "api": "numpy in -> numpy out through the call above (pageable input, page-locked pooled result)"},
        "parity": parity,
        "outputs": {f"cfg{which}_out": last[0].cpu().numpy()} if args.dump_outputs else {},
    }


def run_cfg4(env: Env, args, lib, N, R, VelvetNoise, C):
    torch = env.torch
    Cg, L = args.cfg4_channels_per_gpu, args.cfg4_frames
    vn = VelvetNoise(sample_rate_hz=CFG4_FS, duration_seconds=0.3, num_impulses=300, num_outs=CFG4_TOTAL_CHANNELS,
                     filtered_channels=tuple(range(CFG4_TOTAL_CHANNELS)), mode="LR", normalizer=None, seed=1)
    c0 = (env.rank * Cg) % CFG4_TOTAL_CHANNELS
    if c0 + Cg > CFG4_TOTAL_CHANNELS:
        c0 = CFG4_TOTAL_CHANNELS - Cg
    prog = vn.tap_program(L).slice_channels(c0, c0 + Cg)
    x = device_slab(env, Cg, L, 4321 + env.rank)
    y = torch.empty((Cg, L), dtype=torch.float32, device=env.dev)
    sx, sy, ps = R.torch_signal(x.t()), R.torch_signal(y.t()), R.device_program(prog, env.dev)

    def step():
        N.check(lib.vnd_sparse_fir_dev(C.byref(sx), C.byref(sy), C.byref(ps), env.stream.cuda_stream), "vnd_sparse_fir_dev")

    for _ in range(3):
        step()
    torch.cuda.synchronize()
    parity = "skipped"
    if env.rank == 0:
        from oracle import vnd_oracle as O

        ta = O.class_taps(sample_rate_hz=CFG4_FS, duration_seconds=0.3, num_impulses=300, num_outs=CFG4_TOTAL_CHANNELS,
                          filtered_channels=tuple(range(CFG4_TOTAL_CHANNELS)), seed=1)
        n = 1 << 15
        taps = {ch: ta[c0 + ch] for ch in (0, Cg - 1)}
        windows = [(ch, a, b) for ch in (0, Cg - 1) for a, b in ((0, n), (L // 2 - n // 2, L // 2 + n // 2), (L - n, L))]
        if not oracle_windows(x, y, taps, O.DEFAULT_ENVELOPE, windows, prog.halo):
            raise SystemExit("bench cfg4: GPU output differs from the oracle")
        parity = f"bit-exact vs oracle on channels 0 and {Cg - 1}: {n} frames at the start, the middle and the end"
    steps = args.steps
    sampler = ClockSampler(env.local_rank)
    sampler.start()
    per_step, total_ms = env.timed_events(step, steps)
    clocks = sampler.stop()
    outputs = {f"cfg4_y_{k}": v for k, v in sample_slab(y).items()} if args.dump_outputs else {}
    value = env.world * Cg * L * steps / (total_ms * 1e-3) / 1e9
    kernel_ms = float(np.mean(per_step))
    peak, _ = measured_peak_gbs()
    achieved = BYTES_PER_SAMPLE * Cg * L / (kernel_ms * 1e-3) / 1e9
    clock_hz = 1.965e9
    lsu_peak = 148 * 128 * clock_hz / 1e9  # GB/s the shared-memory pipes of 148 SMs deliver at the maximum SM clock
    lsu_bytes = 300 * 4 * Cg * L  # one 4-byte word per (output, tap) pair
    res = {
        "workload": f"BASELINE configs[3]: {CFG4_TOTAL_CHANNELS} ch x 10 min @ 96 kHz, 300 impulses over 0.3 s (halo 28 800 samples); "
                    f"{Cg} channels x {L} frames per GPU (channel-sharded, planar)",
        "scaling": "weak", "value": value, "unit": UNIT, "ms": total_ms / steps, "steps": steps, "clocks": clocks,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                     "kernel": "fir_ring_kernel (persistent CTA per SM, ring of six 9216-sample chunks = 221 KB of shared memory, every sample "
                               "fetched once under the taps of the previous step, 12 warps x 24 outputs per lane, two decay segments "
                               "interleaved per warp, packed FADD2); the last four chunks of every channel through fir_tile_kernel"},
        "lsu_pipe": {"achieved": lsu_bytes / (kernel_ms * 1e-3) / 1e9, "peak": lsu_peak, "unit": "GB/s", "frac": lsu_bytes / (kernel_ms * 1e-3) / 1e9 / lsu_peak,
                     "note": "the binding bound: 300 taps x 4 B per output through the 128 B/clk/SM shared-memory pipe = 31 Gsamples/s per GPU at 1965 MHz"},
        "parity": parity, "outputs": outputs,
    }
    # end to end through the Python API on a narrower page-locked slab
    try:
        Ce, Le = 8, min(L, 14_400_000)
        R.set_pinned_pool_cap(max(2 * Ce * Le * 4 + (64 << 20), 512 << 20))
        vne = VelvetNoise(sample_rate_hz=CFG4_FS, duration_seconds=0.3, num_impulses=300, num_outs=Ce, filtered_channels=tuple(range(Ce)), mode="LR",
                          normalizer=None, seed=1)
        hx = R.PinnedArray((Le, Ce))
        hx.array[...] = x[:Ce, :Le].t().contiguous().cpu().numpy()
        vne.convolve(hx.array)
        holder = []

        def e2e_step():
            holder.clear()
            holder.append(vne.convolve(hx.array))

        dt = env.timed_wall(e2e_step, steps)
        res["e2e"] = {"value": env.world * Ce * Le * steps / dt / 1e9, "unit": UNIT, "h2d_bytes_per_step": Ce * Le * 4, "d2h_bytes_per_step": Ce * Le * 4,
                      "channels": Ce, "frames": Le, "api": "VelvetNoise.convolve(numpy (frames, channels) C-order, page-locked) -> numpy"}
        del hx, holder
        R.trim_pinned_pool(0)
    except Exception as exc:
        res["e2e"] = {"value": None, "error": repr(exc)}
    del x, y
    torch.cuda.empty_cache()
    return res


def run_cfg5(env: Env, args, lib, N, R, OPT):
    """optimize_velvet_noise for 64 clips x 1024 strengths x 30 s: grid stage + refinement, clips sharded over the ranks."""
    import contextlib
    import io

    from vndecorrelate_b200 import sharding as S

    torch = env.torch
    n_clips, frames, grid = args.cfg5_clips, args.cfg5_frames, args.cfg5_grid
    lo, hi = S.block_range(n_clips, env.rank, env.world)
    host = np.zeros((n_clips, 2, frames), dtype=np.float32)  # only the rank's block is generated (and ever read)
    for i in range(lo, hi):
        host[i] = coloured_clip(i, frames).T
    kw = dict(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, seed=1, grid_size=grid)
    block = torch.from_numpy(host[lo:hi]).to(env.dev)  # the rank's clips, resident
    resident = None

    def optimise(inputs):
        with contextlib.redirect_stdout(io.StringIO()):
            if inputs is None:
                return OPT.optimize_velvet_noise_batch(local_signals=block, total_clips=n_clips, details=True, **kw)
            return OPT.optimize_velvet_noise_batch(input_signals=inputs, details=True, **kw)

    kappa, info = optimise(resident)  # warm-up (NCCL communicator, arenas)
    steps = args.steps
    launches0 = N.launch_count()
    sampler = ClockSampler(env.local_rank)
    env.barrier()
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(steps):
        kappa, info = optimise(resident)
    torch.cuda.synchronize()
    dt = env.max_over_ranks(time.perf_counter() - t0) / steps
    clocks = sampler.stop()
    outputs = {"cfg5_kappa": np.asarray(kappa), "cfg5_scores": np.asarray(info["scores"])} if args.dump_outputs else {}
    launches = int(env.sum_over_ranks(N.launch_count() - launches0)) // steps
    evals = int(env.sum_over_ranks(info["evaluations_local"]))
    # end to end: host clips in (the rank uploads its block inside the call)
    env.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        kappa_h, info_h = optimise(host)
    torch.cuda.synchronize()
    dt_e2e = env.max_over_ranks(time.perf_counter() - t0) / steps
    same = bool(np.array_equal(kappa, kappa_h) and np.array_equal(info["scores"], info_h["scores"]))

    # grid-stage kernel alone (the dominant kernel): one launch over the rank's clips x all strengths
    from vndecorrelate_b200.taps import kappa_family_program

    prog = kappa_family_program(np.linspace(0.0, 1.0, grid), sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30,
                                envelope=(0.85, 0.55, 0.35, 0.2), seed=1, frames=frames)
    OPT.vn_objective_partials(block, prog)
    sampler = ClockSampler(env.local_rank)
    sampler.start()
    per_step, _ = env.timed_events(lambda: OPT.vn_objective_partials(block, prog), steps)
    k_clocks = sampler.stop()
    k_ms = float(np.mean(per_step))
    k_evals = (hi - lo) * grid
    frame_evals = k_evals * frames
    clock_hz = 1.965e9
    lsu_peak = 148 * 128 * clock_hz / 1e9
    lsu_bytes = frame_evals * 31 * 4  # 30 taps + the unfiltered channel, one word each per frame-evaluation
    peak, _ = measured_peak_gbs()
    hbm_bytes = (hi - lo) * 2 * frames * 4

    # parity: sampled strengths of the first local clip against the oracle, incl. the neighbours of the GPU argmin
    parity = "skipped"
    if env.rank == 0:
        from oracle import vnd_oracle as O

        row = info["scores"][lo]
        am = int(np.argmin(row))
        idx = sorted({0, grid - 1, am, max(0, am - 1), min(grid - 1, am + 1)} | set(np.linspace(0, grid - 1, 6).astype(int).tolist()))
        ks = np.linspace(0.0, 1.0, grid)[idx]
        want = O.vn_grid_scores(host[lo].T.copy(), ks, sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, seed=1)
        err = float(np.max(np.abs(row[idx].astype(np.float64) - np.asarray(want, dtype=np.float64))))
        if err > 5e-4:
            raise SystemExit(f"bench cfg5: scores differ from the oracle by {err}")
        parity = f"{len(idx)} sampled strengths of clip {lo} (incl. the argmin and its neighbours) within {err:.1e} of the oracle (bound 5e-4)"
    digest = hashlib.sha256(np.ascontiguousarray(info["scores"]).tobytes()).hexdigest()
    return {
        "workload": f"BASELINE configs[4]: optimize_velvet_noise, {grid} strengths x {n_clips} synthetic {frames / FS:.0f} s stereo clips @ 48 kHz, "
                    "grid scan + lock-step Brent refinement of every local minimum",
        "scaling": "strong (the clips are sharded over the ranks; one all-gather of the float32 score matrix, one of the refined strengths)",
        "value": evals / dt, "unit": "objective evaluations/s (clip x strength, grid + refinement)", "ms": dt * 1e3, "steps": steps,
        "clips": n_clips, "clips_per_s": n_clips / dt, "evaluations": evals, "kernel_launches": launches, "clocks": clocks,
        "collective": f"NCCL all_gather_into_tensor, {env.world} ranks" if env.world > 1 else "none (one rank)",
        "scores_sha256": digest, "argmin_first8": info["argmin"][:8], "local_minima_first8": [len(m) for m in info["local_minima"][:8]],
        "kappa_first4": [float(k) for k in kappa[:4]],
        "grid_kernel": {"kernel": "vn_objective_kernel", "ms": k_ms, "evaluations_per_s_per_gpu": k_evals / (k_ms * 1e-3),
                        "frame_evaluations_per_s_per_gpu": frame_evals / (k_ms * 1e-3), "clocks": k_clocks},
        "roofline": {"bound": "hbm", "achieved": hbm_bytes / (k_ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s", "frac": hbm_bytes / (k_ms * 1e-3) / 1e9 / peak,
                     "traffic": None, "note": "not the binding bound: every clip is read once per tile and reused by all strengths from shared memory"},
        "lsu_pipe": {"achieved": lsu_bytes / (k_ms * 1e-3) / 1e9, "peak": lsu_peak, "unit": "GB/s", "frac": lsu_bytes / (k_ms * 1e-3) / 1e9 / lsu_peak,
                     "note": "31 shared-memory words per frame-evaluation against 128 B/clk/SM at 1965 MHz"},
        "e2e": {"value": evals / dt_e2e, "unit": "objective evaluations/s", "ms": dt_e2e * 1e3, "h2d_bytes_per_step": int((hi - lo) * 2 * frames * 4),
                "d2h_bytes_per_step": int(evals * 12 * 8 // max(env.world, 1)), "same_result_as_resident": same,
                "api": "vndecorrelate_b200.optimization.optimize_velvet_noise_batch(input_signals=numpy clips, ...)"},
        "parity": parity, "outputs": outputs,
    }


def run_b200(args) -> None:
    import ctypes as C

    from vndecorrelate_b200 import _native as N
    from vndecorrelate_b200 import decorrelation as api
    from vndecorrelate_b200 import optimization as OPT
    from vndecorrelate_b200 import runtime as R

    env = Env()
    lib = N.lib()
    if hasattr(lib, "vnd_debug_fir_plan"):
        lib.vnd_debug_fir_plan.restype = C.c_int
    want = _parse_configs(args.configs)
    main = run_cfg3(env, args, lib, N, R, api.VelvetNoise, C)
    outputs = main.pop("outputs")
    configs = {}
    for which, fn in ((1, lambda: run_cfg12(env, args, 1, lib, N, R, api)), (2, lambda: run_cfg12(env, args, 2, lib, N, R, api)),
                      (4, lambda: run_cfg4(env, args, lib, N, R, api.VelvetNoise, C)), (5, lambda: run_cfg5(env, args, lib, N, R, OPT))):
        if which not in want:
            continue
        try:
            configs[f"cfg{which}"] = fn()
            outputs.update(configs[f"cfg{which}"].pop("outputs"))
        except SystemExit:
            raise
        except Exception as exc:  # report, do not hide
            configs[f"cfg{which}"] = {"error": repr(exc)}
            if env.world > 1:
                raise

    cpu_baseline = None
    if env.rank == 0 and env.world == 1 and not args.no_cpu_baseline:
        ch, fr = 64, 960_000  # ~20 s of CPU work on one core; the strided column access of the C-order layout gets slower with more channels
        rate, secs = cpu_fir_rate(1, ch, fr)
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": 1, "kind": cpu_kind(),
                        "sample": f"{ch} channels x {fr} frames (20 s @ 48 kHz) C-order (frames, channels) fp32, VelvetNoise.convolve, one pass ({secs:.1f} s)"}
        try:
            if "cfg1" in configs:
                configs["cfg1"]["cpu_baseline"] = cpu_cfg1()
            if "cfg2" in configs:
                configs["cfg2"]["cpu_baseline"] = cpu_cfg2()
            if "cfg4" in configs:
                r4, s4 = cpu_fir_rate(1, 2, 480_000, fs=CFG4_FS, dur=0.3, nimp=300)
                configs["cfg4"]["cpu_baseline"] = {"value": r4, "unit": UNIT, "cores": 1, "kind": cpu_kind(),
                                                   "sample": f"2 channels x 480000 frames (5 s @ 96 kHz), 300 impulses / 0.3 s, C-order ({s4:.1f} s)"}
            if "cfg5" in configs:
                configs["cfg5"]["cpu_baseline"] = cpu_cfg5(1, 16)
        except Exception as exc:
            configs["cpu_baseline_error"] = repr(exc)

    if env.rank == 0 and args.dump_outputs:
        write_outputs(args.dump_outputs, outputs)
    if env.rank == 0:
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": env.world, "steps": args.steps, "warmup": main["warm"],
            "ms_per_step": main["total_ms"] / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(args), "clocks": main["clocks"], "e2e": main["e2e"], "gpu_launches": main["launches"],
            "roofline": main["roofline"], "cpu_baseline": cpu_baseline, "parity": main["parity"], "configs": configs,
        }
        print(json.dumps(line))
    if env.world > 1:
        env.dist.destroy_process_group()


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--configs", default="1,2,4,5", help="BASELINE configs reported under `configs` next to the headline (config 3)")
    ap.add_argument("--channels-per-gpu", type=int, default=CHANNELS_PER_GPU)
    ap.add_argument("--frames", type=int, default=FRAMES)
    ap.add_argument("--e2e-channels", type=int, default=32)
    ap.add_argument("--cfg4-channels-per-gpu", type=int, default=CFG4_CHANNELS_PER_GPU)
    ap.add_argument("--cfg4-frames", type=int, default=CFG4_FRAMES)
    ap.add_argument("--cfg5-clips", type=int, default=CFG5_CLIPS)
    ap.add_argument("--cfg5-frames", type=int, default=CFG5_FRAMES)
    ap.add_argument("--cfg5-grid", type=int, default=CFG5_GRID)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed steps computed in their last step (a fixed sample of the "
                    "large slabs) as DIR/<name>.npy, float32 / float64, at most 64 MB; same arguments, same inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU arm (--impl b200)")
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
