"""grid_scan over velvet-noise stereo candidates (two outputs, no normaliser, any filtered channels, LR or MS, any width)
and over any Haas effect: one launch per family, every score equal (``==``, same dtype) to the one the candidate gets
when it is decorrelated and scored on its own.

The CPU tests check the routing, that every exception comes before any device work with the candidate-by-candidate
type, and the C ABI's argument checks.  The GPU tests compare every score with the per-candidate path.
"""

from __future__ import annotations

import ctypes as C
import re

import numpy as np
import pytest

from oracle import vnd_oracle as O
from tests import _golden as G
from vndecorrelate_b200 import _native as N
from vndecorrelate_b200 import decorrelation as D
from vndecorrelate_b200 import optimization as opt
from vndecorrelate_b200.taps import IDENTITY_ENVELOPE

gpu = pytest.mark.gpu
FS = 44100
KW = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)
LENGTHS = [1, 7, 300, 4095, 4096, 4097, 3 * 4096 + 5]  # 300: shorter than the filters' halo (~1160 frames)


def _vn(mode="MS", fc=(0, 1), width=None, env=(0.85, 0.55, 0.35, 0.2), kappa=1.0, seed=3):
    return D.VelvetNoise(sample_rate_hz=FS, normalizer=None, mode=mode, filtered_channels=fc, width=width, segment_envelope=env,
                         log_distribution_strength=kappa, seed=seed)


def _haas(delay=0.002, ch=0, mode="LR", width=None):
    return D.HaasEffect(sample_rate_hz=FS, delay_time_seconds=delay, delayed_channel=ch, mode=mode, width=width)


def _vn_family(env=(0.85, 0.55, 0.35, 0.2)):
    out = []
    for k, (mode, fc, width) in enumerate([(m, f, w) for m in ("LR", "MS") for f in ((0, 1), (0,), ()) for w in (None, 0.0, 0.3, 1.0)]):
        out.append(_vn(mode=mode, fc=fc, width=width, env=env, kappa=k / 23, seed=k % 5))
    return out


def _signal(frames, seed=0):
    return (np.random.default_rng(seed).standard_normal((frames, 2)) * 0.3).astype(np.float32)


def _one_by_one(x, cands):
    return [opt._score_signal(d.decorrelate(x), KW) for d in cands]


def _assert_same(scores, x, cands):
    ref = _one_by_one(x, cands)
    assert len(scores) == len(ref)
    for j, (s, r) in enumerate(zip(scores, ref)):
        assert type(s) is type(r) and s.dtype == r.dtype, (j, type(s), type(r))
        assert s == r or (np.isnan(s) and np.isnan(r)), (j, s, r)


@pytest.fixture
def no_device(monkeypatch):
    """Any call into the native library fails the test: the errors below come before any device work."""

    def forbidden(*a, **k):
        raise AssertionError("the native library was called")

    monkeypatch.setattr(N, "lib", forbidden)


# ------------------------------------------------------------------ CPU: routing


@pytest.fixture
def routes(monkeypatch):
    """Replaces every device entry point of _scan by a recorder returning zero partials."""
    calls = []

    def rec(name, slots):
        def f(*args):
            if name in ("vn_stereo", "haas_effect"):  # (x, planar x, candidates)
                n = len(args[2])
                calls.append((name, n))
                return np.zeros((n, slots))
            n = args[1].channels if name == "vn" else len(args[1])  # (clip, program) / (clip, delays)
            calls.append((name, n))
            return np.zeros((1, n, slots))
        return f

    monkeypatch.setattr(opt, "_vn_stereo_partials", rec("vn_stereo", N.OBJ_SLOTS))
    monkeypatch.setattr(opt, "_haas_effect_partials", rec("haas_effect", N.HAAS_SLOTS))
    monkeypatch.setattr(opt, "vn_objective_partials", rec("vn", N.OBJ_SLOTS))
    monkeypatch.setattr(opt, "haas_objective_partials", rec("haas", N.HAAS_SLOTS))

    def single(y, kw):
        calls.append(("single", 1))
        return np.float32(0)

    monkeypatch.setattr(opt, "_score_signal", single)
    monkeypatch.setattr(D.VelvetNoise, "decorrelate", lambda self, x: None)
    monkeypatch.setattr(D.HaasEffect, "decorrelate", lambda self, x: None)
    return calls


def test_reference_families_keep_their_kernels(routes):
    x = _signal(100)
    opt.grid_scan(x, [_vn(mode="LR", fc=(0,), kappa=k) for k in (0.1, 0.5)], **KW)
    opt.grid_scan(x, [_haas(d) for d in (0.0, 0.001, 0.002)], **KW)
    assert routes == [("vn", 2), ("haas", 3)]


def test_new_families_and_mixed_lists_are_split(routes):
    x = _signal(100)
    identity = _vn(env=IDENTITY_ENVELOPE)
    user = D.VelvetNoise(sample_rate_hz=FS, normalizer=lambda a, b: None, seed=1)
    rms = D.VelvetNoise(sample_rate_hz=FS, seed=1)
    cands = [_vn(), _haas(ch=1), identity, user, _vn(mode="LR", fc=(0,)), _haas(), rms, _haas(mode="MS", width=0.5)]
    scores = opt.grid_scan(x, cands, **KW)
    assert len(scores) == len(cands)
    assert sorted(routes) == sorted([("vn_stereo", 2), ("vn_stereo", 1), ("haas_effect", 3), ("single", 1), ("single", 1)])
    # a list of the reference's velvet-noise family with two envelopes is no longer scored one by one
    routes.clear()
    opt.grid_scan(x, [_vn(mode="LR", fc=(0,)), _vn(mode="LR", fc=(0,), env=(0.5, 0.25))], **KW)
    assert routes == [("vn_stereo", 2)]


def test_recognition():
    assert opt._is_vn_stereo_candidate(_vn(mode="LR", fc=()))
    assert opt._is_vn_stereo_candidate(_vn(width=0.4))
    assert not opt._is_vn_stereo_candidate(D.VelvetNoise(sample_rate_hz=FS, seed=1))  # rms_normalize
    assert not opt._is_vn_stereo_candidate(D.VelvetNoise(sample_rate_hz=FS, num_outs=3, normalizer=None, filtered_channels=(0, 1, 2), seed=1))
    assert opt._is_haas_effect_candidate(_haas(ch=-2, mode="MS", width=0.2))
    assert not opt._is_haas_effect_candidate(_haas(delay=-0.01))


# ------------------------------------------------------------------ CPU: exceptions before any device work


def test_errors_before_device_work(no_device):
    with pytest.raises(ValueError, match="zero-size array"):
        opt.grid_scan(np.zeros((0, 2), np.float32), [_vn(), _haas()], **KW)
    three = np.zeros((10, 3), np.float32)
    with pytest.raises(ValueError, match=r"Expected shape \(num samples, 2\), but got shape \(10, 3\)"):
        opt.grid_scan(three, [_vn(mode="LR"), _vn(mode="MS")], **KW)  # MS needs exactly two columns
    with pytest.raises(ValueError, match=r"could not broadcast input array from shape \(10, 3\)"):
        opt.grid_scan(three, [_haas(ch=1)], **KW)
    with pytest.raises(IndexError, match="index 2 is out of bounds for axis 1 with size 2"):
        opt.grid_scan(np.zeros((10, 2), np.float32), [_haas(ch=1), _haas(ch=2)], **KW)
    with pytest.raises(IndexError, match="index 1 is out of bounds for axis 1 with size 1"):
        opt.grid_scan(np.zeros((10, 1), np.float32), [_vn(mode="LR")], **KW)
    with pytest.raises(ValueError, match="Input shape invalid"):
        opt.symmetry_aware_objective(np.zeros((4, 2, 2), np.float32), _vn(mode="LR"), **KW)


def test_error_types_match_the_single_path():
    """The checks the family path runs are the single calls' own: same type, same message."""
    for x, d in [(np.zeros((10, 3), np.float32), _vn(mode="MS")), (np.zeros((10, 3), np.float32), _haas(ch=1)), (np.zeros((10, 2), np.float32), _haas(ch=5))]:
        with pytest.raises(Exception) as single:
            d.decorrelate(x)
        with pytest.raises(type(single.value), match=re.escape(str(single.value))):
            opt.grid_scan(x, [d], **KW)


def test_public_helpers_reject_other_candidates(no_device):
    with pytest.raises(ValueError, match="normalizer=None"):
        opt.vn_stereo_objective_partials(_signal(10), [D.VelvetNoise(sample_rate_hz=FS, seed=1)])
    with pytest.raises(ValueError, match="HaasEffect"):
        opt.haas_effect_objective_partials(_signal(10), [_vn()])


# ------------------------------------------------------------------ CPU: C ABI argument checks


def test_abi_checks_arguments_before_any_launch():
    try:
        lib = N.lib()
    except N.VndError:
        pytest.skip("library not built")
    x = np.zeros((2, 8), np.float32)
    out = np.zeros((4, 12))
    prog = opt._batch_program([_vn().tap_program(8), _vn().tap_program(8)])
    ps = prog.host_struct()
    cands = np.zeros(2, dtype=N.VN_STEREO_CAND_DTYPE)
    p = C.c_void_p
    # wrong channel count, empty clip, overlapping channels, null pointers
    assert lib.vnd_vn_stereo_objective_dev(p(x.ctypes.data), 8, 8, C.byref(ps), p(cands.ctypes.data), 1, p(out.ctypes.data), None, 0, None) == N.VND_EINVAL
    assert lib.vnd_vn_stereo_objective_dev(p(x.ctypes.data), 0, 8, C.byref(ps), p(cands.ctypes.data), 2, p(out.ctypes.data), None, 0, None) == N.VND_EINVAL
    assert lib.vnd_vn_stereo_objective_dev(p(x.ctypes.data), 8, 4, C.byref(ps), p(cands.ctypes.data), 2, p(out.ctypes.data), None, 0, None) == N.VND_EINVAL
    assert lib.vnd_vn_stereo_objective_dev(p(x.ctypes.data), 8, 8, C.byref(ps), None, 2, p(out.ctypes.data), None, 0, None) == N.VND_EINVAL
    assert lib.vnd_vn_stereo_objective_dev(None, 8, 8, C.byref(ps), p(cands.ctypes.data), 2, p(out.ctypes.data), None, 0, None) == N.VND_EINVAL
    assert lib.vnd_vn_stereo_objective_host(None, p(x.ctypes.data), 8, 8, C.byref(ps), p(cands.ctypes.data), 2, p(out.ctypes.data)) == N.VND_EINVAL
    recs = np.zeros(2, dtype=N.HAAS_CLIP_DTYPE)
    assert lib.vnd_haas_effect_objective_dev(p(x.ctypes.data), 0, 8, p(recs.ctypes.data), 2, p(out.ctypes.data), None) == N.VND_EINVAL
    assert lib.vnd_haas_effect_objective_dev(p(x.ctypes.data), 8, 4, p(recs.ctypes.data), 2, p(out.ctypes.data), None) == N.VND_EINVAL
    assert lib.vnd_haas_effect_objective_dev(p(x.ctypes.data), 8, 8, p(recs.ctypes.data + 8), 1, p(out.ctypes.data), None) == N.VND_EINVAL
    assert lib.vnd_haas_effect_objective_dev(p(x.ctypes.data), 8, 8, None, 2, p(out.ctypes.data), None) == N.VND_EINVAL
    assert lib.vnd_haas_effect_objective_dev(p(x.ctypes.data), 8, 8, p(recs.ctypes.data), -1, p(out.ctypes.data), None) == N.VND_EINVAL


# ------------------------------------------------------------------ GPU: every score equals the candidate's own


@gpu
@pytest.mark.parametrize("frames", LENGTHS)
@pytest.mark.parametrize("env", ["default", "identity", "long"])
def test_vn_stereo_scores_equal_the_single_path(frames, env):
    envelope = {"default": (0.85, 0.55, 0.35, 0.2), "identity": IDENTITY_ENVELOPE, "long": tuple(np.linspace(1.0, 0.05, 1000))}[env]
    cands = _vn_family(envelope)
    x = _signal(frames, seed=frames)
    _assert_same(opt.grid_scan(x, cands, **KW), x, cands)


@gpu
def test_vn_stereo_scores_on_viola_and_other_inputs():
    _, viola = G.wav("viola")
    cands = _vn_family()
    _assert_same(opt.grid_scan(viola, cands, **KW), viola, cands)
    rng = np.random.default_rng(5)
    mono = (rng.standard_normal(5000) * 0.3).astype(np.float32)
    i16 = rng.integers(-3000, 3000, size=(5000, 2)).astype(np.int16)
    f64 = rng.standard_normal((5000, 2)) * 0.2
    lr3 = (rng.standard_normal((5000, 3)) * 0.3).astype(np.float32)
    for x in (mono, i16, f64):
        _assert_same(opt.grid_scan(x, cands, **KW), x, cands)
    lr = [d for d in cands if d.mode == "LR"]
    _assert_same(opt.grid_scan(lr3, lr, **KW), lr3, lr)


@gpu
def test_vn_stereo_mixed_widths_envelope_kinds_and_tensors():
    import torch

    x = _signal(9000, seed=2)
    cands = [_vn(width=w, kappa=w or 0.5) for w in (None, 0.7, 0.0, None, 0.25)] + [_vn(env=IDENTITY_ENVELOPE, mode="LR", width=0.5)]
    _assert_same(opt.grid_scan(x, cands, **KW), x, cands)
    xt = torch.from_numpy(x).cuda()
    _assert_same(opt.grid_scan(xt, cands, **KW), xt, cands)
    p = opt.vn_stereo_objective_partials(xt, cands[:5])
    assert isinstance(p, torch.Tensor) and p.is_cuda and p.shape == (5, N.OBJ_SLOTS)
    assert np.array_equal(p.cpu().numpy(), opt.vn_stereo_objective_partials(x, cands[:5]))


@gpu
@pytest.mark.parametrize("frames", [1, 7, 4096, 3 * 4096 + 5])
def test_haas_scores_equal_the_single_path(frames):
    import torch

    x = _signal(frames, seed=frames + 1)
    mono = x[:, 0].copy()
    cands = [_haas(delay=d, ch=ch, mode=m, width=w) for d in (0.0, 0.001, 2 * frames / FS + 0.001) for ch in (0, 1, -1, -2) for m in ("LR", "MS")
             for w in (None, 0.6)]
    for inp in (x, mono, torch.from_numpy(x).cuda()):
        _assert_same(opt.grid_scan(inp, cands, **KW), inp, cands)


@gpu
def test_mixed_lists_keep_their_order():
    x = _signal(6000, seed=9)
    user = D.VelvetNoise(sample_rate_hz=FS, normalizer=lambda a, b: None, seed=1)
    cands = [_vn(), _haas(ch=1), user, _vn(mode="LR", fc=(0,)), _haas(), D.VelvetNoise(sample_rate_hz=FS, seed=2), _vn(env=IDENTITY_ENVELOPE),
             _haas(mode="MS", width=0.5)]
    scores = opt.grid_scan(x, cands, **KW)
    ref = np.array(_one_by_one(x, cands))
    assert scores.dtype == ref.dtype and np.array_equal(scores, ref)


@gpu
def test_scores_against_the_oracle():
    x = _signal(20000, seed=4)
    vns = [_vn(mode="MS", width=0.4), _vn(mode="LR", fc=())]
    for d, s in zip(vns, opt.grid_scan(x, vns, **KW)):
        assert abs(float(s) - float(O.objective(np.asarray(d.decorrelate(x), dtype=np.float32), **KW))) <= 5e-4
    hs = [_haas(ch=1, mode="MS", width=0.3), _haas(ch=-2, delay=0.004)]
    for h, s in zip(hs, opt.grid_scan(x, hs, **KW)):
        y = O.haas(x, sample_rate_hz=FS, delay_time_seconds=h.delay_time_seconds, delayed_channel=h.delayed_channel % 2, ms_mode=h.mode == "MS",
                   width=h.width)
        assert abs(float(s) - float(O.objective(y, **KW))) <= 1e-9 * max(1.0, abs(float(s)))


@gpu
def test_one_launch_per_family():
    x = _signal(20000, seed=6)
    before = N.launch_count()
    opt.grid_scan(x, _vn_family(), **KW)
    assert N.launch_count() - before == 2  # objective + combine
    before = N.launch_count()
    opt.grid_scan(x, [_haas(delay=d / 1000, ch=1, mode="MS") for d in range(40)], **KW)
    assert N.launch_count() - before == 1
