"""BlockDecorrelator: live signals decorrelated block by block, one launch per step for all signals, each signal's
concatenated output byte-identical to the one-shot call on its concatenated input.

The CPU tests check the argument handling (every error before any device work, with the signal's index), the step
planner against a frame-by-frame model, and the C ABI's argument checks.  The GPU tests cut signals into blocks in many
ways and compare every signal's concatenated output with the one-shot call.
"""

from __future__ import annotations

import ctypes as C
import os

import numpy as np
import pytest

from tests import _golden as G
from vndecorrelate_b200 import _native as N
from vndecorrelate_b200 import decorrelation as D

gpu = pytest.mark.gpu
FS = 44100


def _vn(**kw):
    base = dict(sample_rate_hz=FS, normalizer=None, seed=3)
    base.update(kw)
    return D.VelvetNoise(**base)


def _haas(**kw):
    base = dict(sample_rate_hz=FS)
    base.update(kw)
    return D.HaasEffect(**base)


def _chain(haas_kw=None, **vn_kw):
    vk = dict(normalizer=None, seed=5)
    vk.update(vn_kw)
    return D.SignalChain(sample_rate_hz=FS).velvet_noise(**vk).haas_effect(**(haas_kw or {}))


def _forbid(monkeypatch):
    def forbidden(*a, **k):
        raise AssertionError("the native library was called")

    monkeypatch.setattr(N, "lib", forbidden)


@pytest.fixture
def no_device(monkeypatch):
    """Call ``no_device()`` after building the objects: from then on any call into the native library fails the test."""
    return lambda: _forbid(monkeypatch)


# ------------------------------------------------------------------ CPU: construction


def test_normalisers_are_rejected_with_a_hint():
    with pytest.raises(NotImplementedError, match="normalizer=None"):
        D.BlockDecorrelator(D.VelvetNoise(sample_rate_hz=FS), 2)
    with pytest.raises(NotImplementedError, match="normalizer=None"):
        D.BlockDecorrelator(D.VelvetNoise(sample_rate_hz=FS, normalizer=lambda x, y: None), 1)


def test_unsupported_chains_and_types_raise_not_implemented():
    with pytest.raises(NotImplementedError, match="HaasEffect, VelvetNoise"):
        D.BlockDecorrelator(D.SignalChain(sample_rate_hz=FS).haas_effect().velvet_noise(normalizer=None), 1)
    with pytest.raises(NotImplementedError):
        D.BlockDecorrelator(D.SignalChain(sample_rate_hz=FS).velvet_noise(normalizer=None).velvet_noise(normalizer=None), 1)
    with pytest.raises(NotImplementedError):
        D.BlockDecorrelator(object(), 1)


def test_per_signal_filters_must_share_the_batch_settings():
    with pytest.raises(ValueError, match="signal 1: BlockDecorrelator needs one width"):
        D.BlockDecorrelator([_vn(width=0.5), _vn(width=0.6)], 2)
    with pytest.raises(ValueError, match="signal 1: every signal needs the same stages"):
        D.BlockDecorrelator([_vn(), _haas()], 2)
    with pytest.raises(ValueError, match="3 decorrelators for 2 signals"):
        D.BlockDecorrelator([_vn()] * 3, 2)


def test_latency_is_the_largest_tap_index():
    vns = [_vn(seed=s) for s in (1, 2)]
    b = D.BlockDecorrelator(vns, 2)
    want = [int(v.velvet_noise.index[v.velvet_noise.filtered].max()) for v in vns]
    assert b.latency_frames.dtype == np.int64 and b.latency_frames.tolist() == want
    assert D.BlockDecorrelator(_haas(), 3).latency_frames.tolist() == [0, 0, 0]


# ------------------------------------------------------------------ CPU: rejections before device work


def test_step_rejections_name_the_signal(no_device):
    b = D.BlockDecorrelator(_vn(), 3)
    no_device()
    ok = np.zeros((8, 2), np.float32)
    with pytest.raises(ValueError, match="2 blocks for 3 signals"):
        b.process([ok, ok])
    with pytest.raises(ValueError, match="2 final flags for 3 signals"):
        b.process([ok, ok, ok], final=[True, False])
    with pytest.raises(ValueError, match=r"signal 1: a block must be \(frames, 2\) or mono \(frames,\), got shape \(8, 3\)"):
        b.process([ok, np.zeros((8, 3), np.float32), ok])
    with pytest.raises(ValueError, match="signal 2: a block must be"):
        b.process([ok, None, np.zeros((2, 2, 2))])
    assert b._received.tolist() == [0, 0, 0]


def test_mixed_and_cpu_tensors_are_rejected(no_device):
    torch = pytest.importorskip("torch")
    b = D.BlockDecorrelator(_haas(), 2)
    no_device()
    with pytest.raises(ValueError, match="signal 1: the blocks of one step must be all numpy arrays or all CUDA tensors"):
        b.process([np.zeros((4, 2), np.float32), torch.zeros((4, 2))])
    with pytest.raises(N.VndError, match="signal 0: CPU torch tensors") as e:
        b.process([torch.zeros((4, 2)), None])
    assert e.value.status == N.VND_EUNSUPPORTED


def test_tensors_on_another_device_are_rejected(no_device):
    torch = pytest.importorskip("torch")

    class Fake:  # a CUDA tensor stand-in whose device differs from the object's
        ndim, shape, is_cuda = 2, (4, 2), True
        device = torch.device("cuda:1")

    b = D.BlockDecorrelator(_haas(), 2, device="cuda:0")
    no_device()
    orig = D.R.is_torch_tensor
    try:
        D.R.is_torch_tensor = lambda x: isinstance(x, Fake) or orig(x)
        with pytest.raises(ValueError, match="signal 1: the block is on cuda:1"):
            b.process([None, Fake()])
    finally:
        D.R.is_torch_tensor = orig


def test_a_signal_keeps_its_layout_until_final(no_device, monkeypatch):
    b = D.BlockDecorrelator(_haas(), 2)
    no_device()
    b._mono[:] = [0, 1]  # as after a stereo block on signal 0 and a mono block on signal 1
    with pytest.raises(ValueError, match="signal 1: a stereo block for a mono signal"):
        b.process([np.zeros((3, 2), np.float32), np.zeros((3, 2), np.float32)])
    with pytest.raises(ValueError, match="signal 0: a mono block for a stereo signal"):
        b.process([np.zeros(3, np.float32), None])


# ------------------------------------------------------------------ CPU: the step planner


def _model(schedule, A, d):
    """Frame-by-frame model of one signal: frame t of the output is ready once every input frame it reads has arrived
    (t + A < T for velvet noise, t < T for the Haas effect), and everything, tail included, at the final step."""
    T = emitted = 0
    out = []
    for L, final in schedule:
        T += L
        if final:
            ready = T + d
        else:
            ready = 0
            while ready < T and ready + A < T:
                ready += 1
        out.append((T, ready - emitted))
        emitted = ready
        if final:
            T = emitted = 0
    return out


@pytest.mark.parametrize("A,d", [(0, 0), (0, 7), (5, 0), (40, 0), (40, 13), (1, 1)])
def test_planner_matches_a_frame_by_frame_model(A, d):
    rng = np.random.default_rng(A * 100 + d)
    n, steps = 6, 40
    lengths = rng.choice([0, 0, 1, 2, A, A + 1, 3 * A + 2, 60], size=(steps, n)).astype(np.int64)
    finals = rng.random((steps, n)) < 0.15
    H = max(A, d)
    rec = np.zeros(n, np.int64)
    emi = np.zeros(n, np.int64)
    lat = np.full(n, A, np.int64)
    tail = np.full(n, d, np.int64)
    got = [[] for _ in range(n)]
    for s in range(steps):
        plan = D.plan_block_step(rec, emi, lengths[s], finals[s], lat, tail, H)
        counts = np.diff(plan.out_offsets)
        assert plan.out_offsets[0] == 0 and np.all(counts >= 0)
        assert np.array_equal(plan.total, rec + lengths[s])
        assert np.array_equal(plan.history_start, plan.total - H)
        for i in range(n):
            got[i].append((int(plan.total[i]), int(counts[i])))
        assert np.all(plan.next_received[finals[s]] == 0) and np.all(plan.next_emitted[finals[s]] == 0)
        rec, emi = plan.next_received, plan.next_emitted
    for i in range(n):
        assert got[i] == _model(list(zip(lengths[:, i].tolist(), finals[:, i].tolist())), A, d)


# ------------------------------------------------------------------ CPU: the C ABI's argument checks


def _vn_step(lib, **over):
    prog = D.BlockDecorrelator(_vn(), 1)._program
    ps = prog.host_struct()
    ep = N.EpilogueStruct(1, 0, 0.0, 0, 0, 0)
    args = dict(x=None, rows=0, offs=8, n=1, recv=8, emit=8, prog_of=8, taps=C.byref(ps), ep=C.byref(ep), h_in=8, h_out=16,
                H=prog.halo, oo=8, out_rows=0, out=None, stream=None)
    args.update(over)
    return lib.vnd_vn_block_step_dev(*args.values())


def test_abi_rejects_illegal_arguments():
    lib = N.lib()
    assert _vn_step(lib) == N.VND_OK  # nothing to do: no launch
    assert _vn_step(lib, rows=-1) == N.VND_EINVAL
    assert _vn_step(lib, n=-1) == N.VND_EINVAL
    assert _vn_step(lib, rows=5, x=None) == N.VND_EINVAL
    assert _vn_step(lib, rows=5, x=4) == N.VND_EINVAL  # misaligned
    assert _vn_step(lib, offs=None) == N.VND_EINVAL
    assert _vn_step(lib, emit=None) == N.VND_EINVAL
    assert _vn_step(lib, out_rows=3, out=None) == N.VND_EINVAL
    assert _vn_step(lib, h_out=8) == N.VND_EINVAL  # one buffer for both
    assert _vn_step(lib, h_in=None) == N.VND_EINVAL
    assert _vn_step(lib, H=3) == N.VND_EINVAL  # shorter than the look-ahead
    assert _vn_step(lib, ep=C.byref(N.EpilogueStruct(0, 0, 0.0, 1, 0, 0))) == N.VND_EINVAL
    assert _vn_step(lib, ep=C.byref(N.EpilogueStruct(0, 0, 0.0, 0, 5, 0))) == N.VND_EINVAL
    assert _vn_step(lib, ep=None) == N.VND_EINVAL
    assert _vn_step(lib, taps=None) == N.VND_EINVAL
    assert _vn_step(lib, n=0, rows=4, x=8) == N.VND_EINVAL

    h = lib.vnd_haas_block_step_dev
    base = dict(x=None, rows=0, offs=16, n=1, recv=16, sig=16, h_in=16, h_out=32, H=4, oo=16, out_rows=0, out=None, stream=None)

    def haas(**over):
        a = dict(base)
        a.update(over)
        return h(*a.values())

    assert haas() == N.VND_OK
    assert haas(sig=None) == N.VND_EINVAL
    assert haas(sig=8) == N.VND_EINVAL  # records are 16-byte aligned
    assert haas(out_rows=2, out=8) == N.VND_EINVAL  # float64 pairs are 16-byte aligned
    assert haas(H=-1) == N.VND_EINVAL
    assert haas(recv=None) == N.VND_EINVAL
    assert haas(h_out=16) == N.VND_EINVAL


def test_abi_rejects_a_filter_too_long_for_the_step_kernel():
    lib = N.lib()
    vn = D.VelvetNoise(sample_rate_hz=48000, normalizer=None, duration_seconds=1.0, num_impulses=60, seed=1)
    prog = vn.tap_program(10**9)
    ps = prog.host_struct()
    ep = N.EpilogueStruct(1, 0, 0.0, 0, 0, 0)
    assert lib.vnd_vn_block_step_dev(None, 0, None, 0, None, None, None, C.byref(ps), C.byref(ep), None, None, prog.halo, None, 0, None,
                                     None) == N.VND_EUNSUPPORTED


# ------------------------------------------------------------------ GPU: byte equality with the one-shot call


def _same(a, b) -> bool:
    if not isinstance(a, np.ndarray):
        a = a.cpu().numpy()
    if not isinstance(b, np.ndarray):
        b = b.cpu().numpy()
    return G.same_bits(a, b)


def _cut(x, sizes):
    """x cut into blocks of the given sizes (the last block takes the rest)."""
    out, at = [], 0
    for s in sizes:
        out.append(x[at:at + s])
        at += s
    out[-1] = x[at - sizes[-1]:]
    return out


def _run(dec, signals, cuts, torch_blocks, extra_final_empty=False):
    """Feeds signal i its blocks cuts[i] (None entries are idle steps), final at its last block; returns each signal's
    concatenated output and checks the ready counts after every non-final step."""
    torch = pytest.importorskip("torch")
    n = len(signals)
    b = D.BlockDecorrelator(dec, n)
    decs = dec if isinstance(dec, list) else [dec] * n
    tails = b._tail
    outs = [[] for _ in range(n)]
    steps = max(len(c) for c in cuts) + (1 if extra_final_empty else 0)
    received = np.zeros(n, np.int64)
    for s in range(steps):
        blocks, fin = [], []
        for i in range(n):
            last = len(cuts[i]) - 1 + (1 if extra_final_empty else 0)
            blk = cuts[i][s] if s < len(cuts[i]) else None
            if blk is not None and torch_blocks:
                blk = torch.from_numpy(np.ascontiguousarray(blk)).cuda()
            blocks.append(blk)
            fin.append(s == last)
        res = b.process(blocks, final=fin)
        for i in range(n):
            if s <= len(cuts[i]) - 1 + (1 if extra_final_empty else 0):
                outs[i].append(res[i])
                received[i] += 0 if blocks[i] is None else blocks[i].shape[0]
                if not fin[i]:
                    total = sum(r.shape[0] for r in outs[i])
                    A = int(b.latency_frames[i])
                    assert total == max(0, int(received[i]) - A), (i, s)
    whole = []
    for i in range(n):
        parts = [r.cpu().numpy() if not isinstance(r, np.ndarray) else r for r in outs[i]]
        got = np.concatenate(parts) if parts else None
        want = decs[i](signals[i])
        assert got.shape[0] == signals[i].shape[0] + int(tails[i])
        whole.append((got, want))
    return whole


def _check(dec, signals, cuts, **kw):
    for torch_blocks in (False, True):
        for i, (got, want) in enumerate(_run(dec, signals, cuts, torch_blocks, **kw)):
            assert _same(got, want), (i, torch_blocks)


def _signal(L, kind="f32", seed=0):
    rng = np.random.default_rng(seed)
    if kind == "mono":
        return (rng.standard_normal(L) * 0.3).astype(np.float32)
    if kind == "int16":
        return rng.integers(-3000, 3000, size=(L, 2)).astype(np.int16)
    if kind == "f64":
        return rng.standard_normal((L, 2)) * 0.2
    return (rng.standard_normal((L, 2)) * 0.3).astype(np.float32)


def _schedules(L, A, seed, ones):
    """Cuts of a signal of L frames: whole, 1-frame blocks over the first `ones` frames, random 0-5000, and blocks of
    A - 1, A and A + 1 frames, A the look-ahead (for the Haas effect alone, its delay)."""
    rng = np.random.default_rng(seed)
    out = [[L]]
    head = min(L, ones)
    out.append([1] * head + [L - head])
    r, left = [], L
    while left > 0:
        s = int(rng.integers(0, 5001))
        r.append(min(s, left))
        left -= r[-1]
    out.append(r + [0])
    for s in (max(A - 1, 1), max(A, 1), A + 1):
        out.append([s] * (L // s) + [L % s])
    return out


DECORRELATORS = {
    "vn-ms": lambda: _vn(),
    "vn-lr": lambda: _vn(mode="LR"),
    "vn-width": lambda: _vn(width=0.6),
    "vn-ch0": lambda: _vn(filtered_channels=(0,), mode="LR"),
    "vn-identity": lambda: _vn(segment_envelope=(1.0,)),
    "haas-lr": lambda: _haas(),
    "haas-ms-width": lambda: _haas(mode="MS", width=0.7, delayed_channel=-1),
    "haas-d0": lambda: _haas(delay_time_seconds=0.0),
    "haas-long": lambda: _haas(delay_time_seconds=0.2),
    "chain-lr": lambda: _chain(),
    "chain-ms-width": lambda: _chain(haas_kw=dict(mode="MS", width=0.4, delayed_channel=1)),
}


@gpu
@pytest.mark.parametrize("name", sorted(DECORRELATORS))
@pytest.mark.parametrize("kind", ["f32", "mono", "int16", "f64"])
def test_every_cut_is_byte_identical_to_the_one_shot_call(name, kind):
    dec = DECORRELATORS[name]()
    one = D.BlockDecorrelator(dec, 1)
    A = int(one.latency_frames[0])
    K = A or int(one._tail[0]) or 64  # the block size whose neighbours matter: the look-ahead, else the Haas delay
    L = 9000
    # 1-frame blocks across the first 3A frames for float32; the other dtypes take the same path after the cast
    ones = 3 * A + 2 if kind == "f32" else 64
    cuts_of = [_cut(_signal(L, kind, seed=k), sizes) for k, sizes in enumerate(_schedules(L, K, len(name), ones))]
    signals = [_signal(L, kind, seed=k) for k in range(len(cuts_of))]
    _check(dec, signals, cuts_of)


@gpu
@pytest.mark.parametrize("name", ["vn-ms", "haas-long", "chain-lr"])
def test_short_empty_and_final_empty_signals(name):
    dec = DECORRELATORS[name]()
    A = int(D.BlockDecorrelator(dec, 1).latency_frames[0])
    signals = [_signal(A // 2, seed=1), _signal(0, seed=2), _signal(A + 3, seed=3), _signal(5, "mono", seed=4)]
    cuts = [_cut(signals[0], [A // 2]), [signals[1]], _cut(signals[2], [2, A]), _cut(signals[3], [1, 1, 3])]
    _check(dec, signals, cuts, extra_final_empty=True)
    _check(dec, signals, cuts)


@gpu
def test_golden_wav_excerpts():
    name = sorted(f[:-4] for f in os.listdir(os.path.join(G.GOLDEN, "audio")) if f.endswith(".wav"))[0]
    fs, data = G.wav(name)
    x = data[: fs * 2]
    for dec in (_vn(sample_rate_hz=fs), _chain(), _haas(sample_rate_hz=fs, mode="MS", width=0.3)):
        _check(dec, [x], [_cut(x, [4096] * (x.shape[0] // 4096 + 1))])


@gpu
def test_per_signal_strengths_seeds_and_haas_settings():
    signals = [_signal(7000 + 37 * i, seed=i) for i in range(5)]
    cuts = [_cut(x, [512] * 20) for x in signals]
    vns = [_vn(seed=10 + i, log_distribution_strength=0.5 + 0.3 * i) for i in range(5)]
    _check(vns, signals, cuts)
    haases = [_haas(delay_time_seconds=0.001 * i, delayed_channel=i % 2, mode="MS" if i % 2 else "LR", width=None if i % 3 else 0.2)
              for i in range(5)]
    _check(haases, signals, cuts)


@gpu
@pytest.mark.parametrize("name", ["vn-ms", "haas-lr", "chain-ms-width"])
def test_many_signals_ragged_idle_and_restarting(name):
    """64 signals with ragged blocks, idle steps, and signals finishing and restarting at different steps: every signal
    matches, and each step makes exactly the launches it needs."""
    torch = pytest.importorskip("torch")
    dec = DECORRELATORS[name]()
    n, steps = 64, 30
    b = D.BlockDecorrelator(dec, n)
    per_step = 2 if name.startswith("chain") else 1
    rng = np.random.default_rng(7)
    pending = [[] for _ in range(n)]  # (blocks, outputs) of the signal's current run
    runs = [[] for _ in range(n)]
    for s in range(steps):
        blocks, fin = [], []
        for i in range(n):
            L = int(rng.choice([0, 0, 1, 300, 512, 1500, 4096]))
            blk = None if L == 0 and rng.random() < 0.5 else _signal(L, "mono" if i % 7 == 0 else "f32", seed=1000 * s + i)
            blocks.append(blk)
            fin.append(bool(rng.random() < 0.12) or s == steps - 1)
        use_t = s % 2 == 1
        if use_t:
            blocks = [None if x is None else torch.from_numpy(x).cuda() for x in blocks]
        before = N.launch_count()
        res = b.process(blocks, final=fin)
        assert N.launch_count() - before == per_step
        for i in range(n):
            x = blocks[i]
            if x is not None:
                pending[i].append((x.cpu().numpy() if use_t else x))
            runs[i].append(res[i].cpu().numpy() if use_t else res[i])
            if fin[i]:
                pend = pending[i] or [np.zeros((0, 2), np.float32)]
                if all(p.shape[0] == 0 for p in pend):
                    pend = [np.zeros((0,) if (i % 7 == 0) else (0, 2), np.float32)]
                got = np.concatenate(runs[i])
                want = dec(np.concatenate([p for p in pend if p.shape[0]] or pend))
                assert _same(got, want), (i, s)
                pending[i], runs[i] = [], []
    # a step where nothing is received and nothing is ready launches nothing
    before = N.launch_count()
    assert all(r.shape[0] == 0 for r in b.process([None] * n))
    assert N.launch_count() == before


@gpu
def test_a_filter_too_long_for_the_step_kernel_raises_at_construction():
    before = N.launch_count()
    with pytest.raises(NotImplementedError, match="does not fit"):
        D.BlockDecorrelator(D.VelvetNoise(sample_rate_hz=48000, normalizer=None, duration_seconds=1.0, num_impulses=60, seed=1), 4)
    assert N.launch_count() == before
