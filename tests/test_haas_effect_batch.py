"""haas_effect_batch: the Haas effect on many clips in one call, each clip with its own settings and each result
byte-identical to ``HaasEffect.decorrelate`` on that clip.

The CPU tests check argument handling, the per-clip settings table, the offsets and the C ABI's argument checks without
a device.  The GPU tests compare every clip's dtype, shape and bytes with the single call - itself pinned to the
reference's fixtures - and with the committed golden cases.
"""

from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from tests import _golden as G
from vndecorrelate_b200 import _native as N
from vndecorrelate_b200 import decorrelation as D
from vndecorrelate_b200.utils.dsp import LayoutMode

gpu = pytest.mark.gpu
FS = 44100


def _haas(delay=0.02, **kw):
    base = dict(sample_rate_hz=FS, delay_time_seconds=delay)
    base.update(kw)
    return D.HaasEffect(**base)


def _clips(lengths, seed=0, mono=(), int16=(), f64=()):
    rng = np.random.default_rng(seed)
    out = []
    for i, L in enumerate(lengths):
        if i in mono:
            out.append((rng.standard_normal(L) * 0.3).astype(np.float32))
        elif i in int16:
            out.append(rng.integers(-3000, 3000, size=(L, 2)).astype(np.int16))
        elif i in f64:
            out.append(rng.standard_normal((L, 2)) * 0.2)
        else:
            out.append((rng.standard_normal((L, 2)) * 0.3).astype(np.float32))
    return out


def _same(a, b) -> bool:
    if not isinstance(a, np.ndarray):
        a = a.cpu().numpy()
    if not isinstance(b, np.ndarray):
        b = b.cpu().numpy()
    return G.same_bits(a, b)


@pytest.fixture
def no_device(monkeypatch):
    """Any call into the native library fails the test: the errors below come before any device work."""

    def forbidden(*a, **k):
        raise AssertionError("the native library was called")

    monkeypatch.setattr(N, "lib", forbidden)


# ------------------------------------------------------------------ CPU: argument handling


def test_bad_shape_raises_value_error_with_the_clip_index(no_device):
    clips = _clips([10, 20]) + [np.zeros((5, 3), np.float32)]
    with pytest.raises(ValueError, match=r"clip 2: could not broadcast input array from shape \(5, 3\)"):
        D.haas_effect_batch(clips, _haas())
    with pytest.raises(ValueError, match="clip 1"):
        D.haas_effect_batch([np.zeros(4, np.float32), np.zeros((2, 2, 2), np.float32)], _haas())


def test_bad_delayed_channel_raises_index_error_with_the_clip_index(no_device):
    with pytest.raises(IndexError, match="clip 1: index 2 is out of bounds for axis 1 with size 2"):
        D.haas_effect_batch(_clips([10, 20, 30]), [_haas(), _haas(delayed_channel=2), _haas(delayed_channel=-3)])
    with pytest.raises(IndexError, match="clip 0"):
        D.haas_effect_batch(_clips([10]), _haas(delayed_channel=5))
    # the single call checks the shape first
    with pytest.raises(ValueError, match="clip 0"):
        D.haas_effect_batch([np.zeros((3, 4), np.float32)], _haas(delayed_channel=5))


def test_negative_delay_raises_value_error_naming_the_clip(no_device):
    with pytest.raises(ValueError, match="clip 1.*-441"):
        D.haas_effect_batch(_clips([10, 20]), [_haas(), _haas(delay=-0.01)])


def test_effect_list_must_match_the_clips(no_device):
    with pytest.raises(ValueError, match="2 Haas effects for 3 clips"):
        D.haas_effect_batch(_clips([10, 20, 30]), [_haas(), _haas()])
    with pytest.raises(TypeError, match="HaasEffect"):
        D.haas_effect_batch(_clips([10]), [D.VelvetNoise(sample_rate_hz=FS, seed=1)])


def test_mixed_and_cpu_tensor_clips_are_rejected(no_device):
    torch = pytest.importorskip("torch")
    with pytest.raises(ValueError, match="all numpy arrays or all CUDA tensors"):
        D.haas_effect_batch([np.zeros((4, 2), np.float32), torch.zeros((4, 2))], _haas())
    with pytest.raises(N.VndError) as e:
        D.haas_effect_batch([torch.zeros((4, 2)), torch.zeros(3)], _haas())
    assert e.value.status == N.VND_EUNSUPPORTED
    with pytest.raises(N.VndError) as e:
        D.haas_effect_batch(torch.zeros((2, 4, 2)), _haas())
    assert e.value.status == N.VND_EUNSUPPORTED


def test_array_form_needs_one_delay_and_a_stereo_shape(no_device):
    x3 = np.zeros((2, 100, 2), np.float32)
    with pytest.raises(ValueError, match="pass clips with different delays as a list"):
        D.haas_effect_batch(x3, [_haas(0.01), _haas(0.02)])
    with pytest.raises(ValueError, match=r"\(n_clips, frames, 2\)"):
        D.haas_effect_batch(np.zeros((2, 100, 3), np.float32), _haas())
    with pytest.raises(ValueError, match=r"\(n_clips, frames, 2\)"):
        D.haas_effect_batch(np.zeros((100, 2), np.float32), _haas())


def test_empty_batch_returns_empty_result(no_device):
    assert D.haas_effect_batch([], _haas()) == []
    assert D.haas_effect_batch([], []) == []
    out = D.haas_effect_batch(np.zeros((0, 50, 2), np.float32), _haas(0.02))
    assert out.shape == (0, 50 + 882, 2) and out.dtype == np.float64


def test_settings_table_from_mixed_effects():
    effects = [
        _haas(0.01, delayed_channel=-1, mode="MS", width=0.4),
        D.HaasEffect(sample_rate_hz=48000, delay_time_seconds=0.02, mode=LayoutMode.LR),
        _haas(0.0, delayed_channel=-2, mode=LayoutMode.MS, width=0.0),
        D.HaasEffect(sample_rate_hz=22050, delay_time_seconds=0.0105, delayed_channel=1, mode="LR", width=1),
    ]
    clips = [np.zeros((5, 2), np.float32), np.zeros(7, np.int16), np.zeros((0, 2)), np.zeros(3, np.float32)]
    t = D._haas_table(effects, clips, shared=False)
    assert t.dtype == N.HAAS_CLIP_DTYPE and t.dtype.itemsize == 32
    assert list(t["delay"]) == [e.delay_len_samples for e in effects] == [441, 960, 0, 232]
    assert list(t["delayed_channel"]) == [1, 0, 0, 1]
    assert list(t["mode_ms"]) == [1, 0, 1, 0]
    assert list(t["mono"]) == [0, 1, 0, 1]
    assert list(t["use_width"]) == [1, 0, 1, 1]
    assert list(t["width"]) == [0.4, 0.0, 0.0, 1.0] and t["width"].dtype == np.float64
    shared = D._haas_table([effects[0]] * 3, clips[:3], shared=True)
    assert list(shared["delay"]) == [441] * 3 and list(shared["mono"]) == [0, 1, 0] and list(shared["width"]) == [0.4] * 3
    offsets, out_offsets = D._haas_offsets(np.array([5, 7, 0, 3]), t["delay"].astype(np.int64))
    assert list(offsets) == [0, 5, 12, 12, 15]
    assert list(out_offsets) == [0, 5 + 441, 12 + 441 + 960, 12 + 441 + 960]


def test_batch_dev_rejects_bad_arguments_without_cuda():
    lib = N.lib()
    x = np.zeros((16, 2), np.float32)
    offs = np.array([0, 16], np.int64)
    oo = np.zeros(1, np.int64)
    table = np.zeros(1, N.HAAS_CLIP_DTYPE)
    out = np.zeros((16, 2), np.float64)

    def call(x_ptr=x.ctypes.data, rows=16, offs_ptr=offs.ctypes.data, n=1, clips=table.ctypes.data, oo_ptr=oo.ctypes.data, out_rows=16,
             out_ptr=out.ctypes.data):
        return lib.vnd_haas_batch_dev(x_ptr, rows, offs_ptr, n, clips, oo_ptr, out_rows, out_ptr, None)

    assert call(x_ptr=None) == N.VND_EINVAL
    assert call(offs_ptr=None) == N.VND_EINVAL
    assert call(clips=None) == N.VND_EINVAL
    assert call(oo_ptr=None) == N.VND_EINVAL
    assert call(out_ptr=None) == N.VND_EINVAL
    assert call(rows=-1) == N.VND_EINVAL
    assert call(n=-1) == N.VND_EINVAL
    assert call(out_rows=-1) == N.VND_EINVAL
    assert call(out_rows=15) == N.VND_EINVAL  # fewer output rows than input rows
    assert call(x_ptr=x.ctypes.data + 4) == N.VND_EINVAL
    assert "8-byte aligned" in lib.vnd_last_error().decode()
    assert call(out_ptr=out.ctypes.data + 8) == N.VND_EINVAL
    assert call(n=0, rows=16, out_rows=16) == N.VND_EINVAL  # rows but no clips
    assert call(x_ptr=None, offs_ptr=None, clips=None, oo_ptr=None, out_ptr=None, n=0, rows=0, out_rows=0) == N.VND_OK  # nothing launched
    assert call(x_ptr=None, rows=0, offs_ptr=offs.ctypes.data, out_ptr=None, out_rows=0) == N.VND_OK  # one empty clip, delay 0
    assert lib.vnd_haas_batch_host(None, x.ctypes.data, 16, offs.ctypes.data, 1, table.ctypes.data, out.ctypes.data) == N.VND_EINVAL


# ------------------------------------------------------------------ GPU: parity with the single call


def _check(clips, effects, got):
    effects = effects if isinstance(effects, list) else [effects] * len(clips)
    assert len(got) == len(clips)
    for i, (x, h, y) in enumerate(zip(clips, effects, got)):
        want = h.decorrelate(x)
        assert _same(y, want), f"clip {i} (length {x.shape[0]}, delay {h.delay_len_samples}) differs from the single call"


RAGGED = [0, 1, 2, 127, 4095, 4096, 4097, 20000, 300_001, 500, 0, 1]


def _mixed_effects(n, seed):
    """Per-clip settings, every delay kind: 0, the clip's length and beyond it, others at random."""
    rng = np.random.default_rng(seed)
    modes = ["LR", "MS", LayoutMode.LR, LayoutMode.MS]
    widths = [None, 0.0, 0.4, 1.0]
    out = []
    for i in range(n):
        out.append(D.HaasEffect(sample_rate_hz=int(rng.choice([44100, 48000])), delay_time_seconds=float(rng.uniform(0, 0.03)),
                                delayed_channel=int(rng.choice([0, 1, -1, -2])), mode=modes[i % 4], width=widths[(i // 4) % 4]))
    return out


def _with_delays(effects, clips):
    """Set clip 0's delay to 0, clip 1's to its length and clip 2's beyond it (in frames of the effect's rate)."""
    for h, L in zip(effects, [None, clips[1].shape[0], clips[2].shape[0] + 1000]):
        h.delay_time_seconds = 0.0 if L is None else L / h.sample_rate_hz
    return effects


@gpu
def test_ragged_numpy_clips_with_mixed_settings():
    clips = _clips(RAGGED, seed=1, mono=(3, 7), int16=(5,), f64=(8,))
    effects = _with_delays(_mixed_effects(len(clips), 1), clips)
    got = D.haas_effect_batch(clips, effects)
    assert all(isinstance(g, np.ndarray) for g in got)
    _check(clips, effects, got)
    shared = _haas(0.0123, delayed_channel=-1, mode="MS", width=0.4)
    _check(clips, shared, D.haas_effect_batch(clips, shared))


@gpu
def test_ragged_cuda_clips_with_mixed_settings():
    import torch

    clips = [torch.from_numpy(np.ascontiguousarray(c)).cuda() for c in _clips(RAGGED, seed=2, mono=(2, 9), int16=(6,), f64=(7,))]
    effects = _with_delays(_mixed_effects(len(clips), 2), clips)
    got = D.haas_effect_batch(clips, effects)
    assert all(g.is_cuda and g.dtype == torch.float64 for g in got)
    _check(clips, effects, got)


@gpu
@pytest.mark.parametrize("mode", ["LR", "MS"])
def test_every_setting_combination_in_one_batch(mode):
    import torch

    lengths = [3000, 1, 0, 777, 5000]
    effects, clips = [], []
    k = 0
    for width in (None, 0.0, 0.4, 1.0):
        for ch in (0, 1, -1, -2):
            for L in lengths:
                effects.append(_haas(0.001 * (k % 7), mode=mode, width=width, delayed_channel=ch))
                clips += _clips([L], seed=k, mono=(0,) if k % 3 == 0 else ())
                k += 1
    _check(clips, effects, D.haas_effect_batch(clips, effects))
    tclips = [torch.from_numpy(c).cuda() for c in clips]
    _check(tclips, effects, D.haas_effect_batch(tclips, effects))


@gpu
def test_array_form():
    import torch

    x3 = (np.random.default_rng(3).standard_normal((6, 30000, 2)) * 0.3).astype(np.float32)
    effects = [_haas(0.02, mode=m, width=w, delayed_channel=c) for m, w, c in
               [("LR", None, 0), ("MS", None, 1), ("LR", 0.3, -1), ("MS", 0.7, -2), ("LR", 1.0, 1), ("MS", 0.0, 0)]]
    got = D.haas_effect_batch(x3, effects)
    assert isinstance(got, np.ndarray) and got.shape == (6, 30000 + 882, 2) and got.dtype == np.float64
    for i in range(6):
        assert _same(got[i], effects[i].decorrelate(x3[i]))
    gt = D.haas_effect_batch(torch.from_numpy(x3).cuda(), effects)
    assert gt.is_cuda and gt.shape == (6, 30000 + 882, 2)
    assert _same(gt, got)
    x16 = (x3 * 1000).astype(np.int16)
    assert _same(D.haas_effect_batch(x16, effects[1])[4], effects[1].decorrelate(x16[4]))


@gpu
def test_golden_haas_cases_in_one_batch():
    cases = G.case_list("haas")
    assert len(cases) == 18
    xs, ys = zip(*(G.case_xy(c) for c in cases))
    effects = [D.HaasEffect(**c["params"]) for c in cases]
    got = D.haas_effect_batch(list(xs), effects)
    for c, y, g in zip(cases, ys, got):
        assert G.same_bits(g, y), f"case {c['id']}"


@gpu
def test_chain_hetero_golden_through_both_batches():
    (c,) = G.case_list("chain_hetero")
    x, y = G.case_xy(c)
    chain = (D.SignalChain(sample_rate_hz=44100)
             .velvet_noise(duration_seconds=0.03, num_impulses=30, width=0.5, seed=5)
             .haas_effect(delay_time_seconds=0.0197, delayed_channel=1, mode="LR"))
    ms = D.HaasEffect(sample_rate_hz=44100, delay_time_seconds=0.0096, delayed_channel=1, mode="MS")
    (z,) = D.haas_effect_batch(D.decorrelate_batch([x], chain), ms)
    assert G.same_bits(z, y)


@gpu
def test_optimised_delays_applied_in_one_batch():
    from vndecorrelate_b200.optimization import optimize_haas_delay_batch

    clips = _clips([8000, 15000, 3000, 12000], seed=13, mono=(2,))
    delays = optimize_haas_delay_batch(input_signals=clips, sample_rate_hz=FS, max_delay_seconds=0.03, grid_size=64)
    effects = [D.HaasEffect(sample_rate_hz=FS, delay_time_seconds=t_i) for t_i in delays]
    _check(clips, effects, D.haas_effect_batch(clips, effects))


def _vn(**kw):
    base = dict(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, seed=1)
    base.update(kw)
    return D.VelvetNoise(**base)


@gpu
@pytest.mark.parametrize("kind", ["lr", "ms", "width"])
@pytest.mark.parametrize("device", ["numpy", "cuda"])
def test_composition_with_decorrelate_batch(kind, device):
    import torch

    clips = _clips([20000, 0, 513, 70000, 1], seed=5, mono=(2,))
    vns = [_vn(seed=s, log_distribution_strength=k) for s, k in zip(range(1, 6), (0.2, 0.5, 1.0, 0.7, 0.1))]
    hs = [_haas(d, delayed_channel=c, mode="MS" if kind == "ms" else "LR", width=0.6 if kind == "width" else None)
          for d, c in zip((0.0, 0.011, 0.02, 0.0297, 0.005), (0, 1, -1, -2, 0))]
    if device == "cuda":
        clips = [torch.from_numpy(c).cuda() for c in clips]
    got = D.haas_effect_batch(D.decorrelate_batch(clips, vns), hs)
    for i, (x, vn, h) in enumerate(zip(clips, vns, hs)):
        chain = D.SignalChain(sample_rate_hz=FS, lazy=False)
        chain._decorrelators = [vn, h]
        assert _same(got[i], chain(x)), i


@gpu
@pytest.mark.parametrize("device", ["numpy", "cuda"])
def test_decorrelate_batch_views_are_read_in_place(monkeypatch, device):
    import torch

    clips = _clips([20000, 0, 513, 70000], seed=6, mono=(2,))
    if device == "cuda":
        clips = [torch.from_numpy(c).cuda() for c in clips]
    vns = [_vn(seed=s) for s in (1, 2, 3, 4)]
    hs = [_haas(d, delayed_channel=c) for d, c in zip((0.02, 0.0, 0.003, 0.0151), (0, 1, 0, 1))]
    ys = D.decorrelate_batch(clips, vns)
    assert D._packed_base(ys, np.concatenate([[0], np.cumsum([y.shape[0] for y in ys])]), device == "cuda") is not None

    def no_packing(*a, **k):
        raise AssertionError("the clips were packed again")

    monkeypatch.setattr(torch, "cat", no_packing)
    monkeypatch.setattr(D, "_pack_clips", no_packing)
    got = D.haas_effect_batch(ys, hs)
    monkeypatch.undo()
    _check(ys, hs, got)


@gpu
def test_launch_count_is_one_per_call():
    import torch

    for n in (4, 400):
        lengths = np.random.default_rng(n).integers(0, 5000, size=n)
        clips = [torch.from_numpy(c).cuda() for c in _clips(lengths, seed=n)]
        effects = _mixed_effects(n, n)
        D.haas_effect_batch(clips, effects)  # warm module loading
        before = N.launch_count()
        D.haas_effect_batch(clips, effects)
        assert N.launch_count() - before == 1, n
    before = N.launch_count()
    assert D.haas_effect_batch([], _haas()) == []
    D.haas_effect_batch(torch.zeros((0, 10, 2), device="cuda"), _haas())
    D.haas_effect_batch([torch.zeros((0, 2), device="cuda")], _haas(0.0))
    assert N.launch_count() == before


@gpu
def test_host_pipeline_matches_one_shot(monkeypatch):
    from vndecorrelate_b200 import runtime as R

    lengths = [int(v) for v in np.random.default_rng(10).integers(20000, 60000, size=40)]
    clips = _clips(lengths, seed=11, mono=(4,))
    effects = _mixed_effects(len(clips), 10)
    monkeypatch.setenv("VND_NO_PIPELINE", "1")
    one_shot = [np.array(y) for y in D.haas_effect_batch(clips, effects)]
    monkeypatch.delenv("VND_NO_PIPELINE")
    monkeypatch.setenv("VND_PIPE_CHUNK_MB", "1")
    piped = D.haas_effect_batch(clips, effects)  # pageable packed input
    for a, b in zip(piped, one_shot):
        assert G.same_bits(a, b)
    _check(clips[:6], effects[:6], piped[:6])
    pinned = R.PinnedArray((24, 50000, 2))  # page-locked input, already packed
    x3 = pinned.array
    x3[...] = (np.random.default_rng(12).standard_normal(x3.shape) * 0.3).astype(np.float32)
    ms = _haas(0.017, mode="MS", width=0.3, delayed_channel=1)
    got = D.haas_effect_batch(x3, ms)
    monkeypatch.setenv("VND_NO_PIPELINE", "1")
    assert G.same_bits(got, D.haas_effect_batch(x3, ms))
    assert _same(got[5], ms.decorrelate(x3[5]))


@gpu
def test_batch_host_rejects_bad_offsets_delays_and_channels():
    from vndecorrelate_b200 import runtime as R

    lib = N.lib()
    x = np.zeros((16, 2), np.float32)
    out = np.zeros((16 + 64, 2), np.float64)
    ctx = R.HostContext.get().handle

    def call(offs, delays=(0, 0), channels=(0, 0)):
        offs = np.asarray(offs, np.int64)
        table = np.zeros(len(delays), N.HAAS_CLIP_DTYPE)
        table["delay"] = delays
        table["delayed_channel"] = channels
        return lib.vnd_haas_batch_host(ctx, x.ctypes.data, 16, offs.ctypes.data, len(table), table.ctypes.data, out.ctypes.data)

    assert call([0, 10, 8, 16], (0, 0, 0), (0, 0, 0)) == N.VND_EINVAL
    assert call([1, 10, 16]) == N.VND_EINVAL
    assert call([0, 10, 15]) == N.VND_EINVAL
    assert call([0, 10, 16], delays=(3, -1)) == N.VND_EINVAL
    assert call([0, 10, 16], channels=(0, 2)) == N.VND_EINVAL
    assert call([0, 10, 16], channels=(-1, 0)) == N.VND_EINVAL
    assert call([0, 10, 16], delays=(32, 32), channels=(1, 0)) == N.VND_OK
