"""grid_scan over velvet-noise stereo candidates with the default normaliser ``rms_normalize`` (two outputs, any filtered
channels, LR or MS, any width): groups of at least ``_RMS_FAMILY_MIN`` candidates of one envelope kind are scored in
three launches, every score equal (``==``, same dtype) to the one the candidate gets when it is decorrelated and scored
on its own.

The CPU tests check the routing, the recognition, that every exception comes before any device work with the
candidate-by-candidate type and message, and the C ABI's argument checks.  The GPU tests compare every score, partials
row and gain with the per-candidate path and the oracle's arithmetic.
"""

from __future__ import annotations

import ctypes as C
from functools import partial

import numpy as np
import pytest

from oracle import vnd_oracle as O
from tests import _golden as G
from vndecorrelate_b200 import _native as N
from vndecorrelate_b200 import decorrelation as D
from vndecorrelate_b200 import optimization as opt
from vndecorrelate_b200.taps import IDENTITY_ENVELOPE, TapProgram
from vndecorrelate_b200.utils.dsp import rms_normalize

gpu = pytest.mark.gpu
FS = 44100
KW = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)
OBJ_TILE = 4096  # the objective kernel's tile; the sums kernel's input tile (2048) and sub-tile (256) divide it
LENGTHS = [1, 7, 300, OBJ_TILE - 1, OBJ_TILE, OBJ_TILE + 1, 3 * OBJ_TILE + 5, 2047, 2048, 2049]  # 300: shorter than the halo
ENVELOPES = {"default": (0.85, 0.55, 0.35, 0.2), "identity": IDENTITY_ENVELOPE, "long": tuple(np.linspace(1.0, 0.05, 1000))}


def _rms(mode="MS", fc=(0, 1), width=None, env=(0.85, 0.55, 0.35, 0.2), kappa=1.0, seed=3, **kw):
    return D.VelvetNoise(sample_rate_hz=FS, mode=mode, filtered_channels=fc, width=width, segment_envelope=env, log_distribution_strength=kappa,
                         seed=seed, **kw)


def _family(env=(0.85, 0.55, 0.35, 0.2)):
    out = []
    for k, (mode, fc, width) in enumerate([(m, f, w) for m in ("LR", "MS") for f in ((0, 1), (0,), ()) for w in (None, 0.0, 0.3, 1.0)]):
        out.append(_rms(mode=mode, fc=fc, width=width, env=env, kappa=k / 23, seed=k % 5))
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


def _identity_partials(y):
    prog = TapProgram(opt._IDENTITY_PROGRAM_WORDS, np.array([0, 5], dtype=np.int32), 1, N.ORDER_SEGMENTED, 0, 1, 5)
    y = y.cpu().numpy() if hasattr(y, "cpu") else np.asarray(y)
    return opt.vn_objective_partials(y[:, :2], prog)[0, 0]


def _same_bits(a, b):
    return np.array_equal(np.atleast_1d(np.asarray(a)).view(np.uint8), np.atleast_1d(np.asarray(b)).view(np.uint8))


@pytest.fixture
def no_device(monkeypatch):
    """Any call into the native library fails the test: the errors below come before any device work."""

    def forbidden(*a, **k):
        raise AssertionError("the native library was called")

    monkeypatch.setattr(N, "lib", forbidden)


# ------------------------------------------------------------------ CPU: routing


@pytest.fixture
def routes(monkeypatch):
    """Replaces every device entry point of _scan, the rms family's included, by a recorder returning zero partials."""
    calls = []

    def family(name, slots):
        def f(x, xp, cands):
            calls.append((name, len(cands)))
            z = np.zeros((len(cands), slots))
            return (z, np.zeros((len(cands), 2), np.float32)) if name == "vn_rms" else z
        return f

    def reference(name, slots):
        def f(clip, arg):
            n = arg.channels if name == "vn" else len(arg)
            calls.append((name, n))
            return np.zeros((1, n, slots))
        return f

    monkeypatch.setattr(opt, "_vn_stereo_partials", family("vn_stereo", N.OBJ_SLOTS))
    monkeypatch.setattr(opt, "_vn_stereo_rms_partials", family("vn_rms", N.OBJ_SLOTS))
    monkeypatch.setattr(opt, "_haas_effect_partials", family("haas_effect", N.HAAS_SLOTS))
    monkeypatch.setattr(opt, "vn_objective_partials", reference("vn", N.OBJ_SLOTS))
    monkeypatch.setattr(opt, "haas_objective_partials", reference("haas", N.HAAS_SLOTS))

    def single(y, kw):
        calls.append(("single", 1))
        return np.float32(0)

    monkeypatch.setattr(opt, "_score_signal", single)
    monkeypatch.setattr(D.VelvetNoise, "decorrelate", lambda self, x: None)
    monkeypatch.setattr(D.HaasEffect, "decorrelate", lambda self, x: None)
    return calls


def test_threshold_is_a_candidate_count_of_at_least_two():
    assert isinstance(opt._RMS_FAMILY_MIN, int) and opt._RMS_FAMILY_MIN >= 2


def test_groups_at_the_threshold_take_the_family_route(routes):
    x = _signal(100)
    m = opt._RMS_FAMILY_MIN
    opt.grid_scan(x, [_rms(kappa=k / 7) for k in range(m)], **KW)
    assert routes == [("vn_rms", m)]
    routes.clear()
    cands = [_rms(kappa=k / 7) for k in range(m)] + [_rms(env=IDENTITY_ENVELOPE, seed=k) for k in range(m)]
    opt.grid_scan(x, cands, **KW)
    assert sorted(routes) == [("vn_rms", m), ("vn_rms", m)]  # one call per envelope kind
    routes.clear()
    opt.grid_scan(x, [_rms(kappa=k / 7) for k in range(m - 1)], **KW)
    assert routes == [("single", 1)] * (m - 1)


def test_a_lone_rms_candidate_goes_one_by_one(routes):
    x = _signal(100)
    opt.grid_scan(x, [_rms()], **KW)
    assert routes == [("single", 1)]
    routes.clear()
    opt.symmetry_aware_objective(x, _rms(), **KW)
    assert routes == [("single", 1)]


def test_mixed_lists_are_split_and_scattered_in_order(routes, monkeypatch):
    m = opt._RMS_FAMILY_MIN
    x = _signal(100)
    user = D.VelvetNoise(sample_rate_hz=FS, normalizer=lambda a, b: None, seed=1)
    rms = [_rms(kappa=k / 9, seed=k) for k in range(m)]
    rms_id = [_rms(env=IDENTITY_ENVELOPE, seed=k) for k in range(m - 1)]  # one short of a group: one by one
    cands = [rms[0], _rms(normalizer=None), D.HaasEffect(sample_rate_hz=FS, delayed_channel=1), user] + rms[1:] + rms_id
    cands += [_rms(normalizer=None, env=IDENTITY_ENVELOPE)]
    opt.grid_scan(x, cands, **KW)
    want = [("vn_stereo", 1), ("vn_stereo", 1), ("vn_rms", m), ("haas_effect", 1)] + [("single", 1)] * (1 + len(rms_id))
    assert sorted(routes) == sorted(want)
    # every score lands at its candidate's position
    monkeypatch.setattr(opt, "vn_scores_from_partials", lambda p, **kw: np.asarray(p)[:, 0].astype(np.float32))

    def tagged(x, xp, c):
        return np.array([[float(id(d) % 1000)] + [0.0] * (N.OBJ_SLOTS - 1) for d in c]), np.zeros((len(c), 2), np.float32)

    monkeypatch.setattr(opt, "_vn_stereo_rms_partials", tagged)
    scores = opt.grid_scan(x, cands, **KW)
    for d, s in zip(cands, scores):
        if opt._is_vn_rms_candidate(d) and d in rms:
            assert s == np.float32(id(d) % 1000)


def test_planar_input_goes_one_by_one(routes):
    x = np.asfortranarray(_signal(100))
    opt.grid_scan(x, [_rms(kappa=k / 7) for k in range(max(2, opt._RMS_FAMILY_MIN))], **KW)
    assert set(routes) == {("single", 1)}


def test_recognition():
    assert opt._is_vn_rms_candidate(_rms())
    assert opt._is_vn_rms_candidate(_rms(mode="LR", fc=(), width=0.3))
    assert opt._is_vn_rms_candidate(_rms(fc=(1, 0)))
    assert not opt._is_vn_rms_candidate(_rms(normalizer=None))
    assert not opt._is_vn_rms_candidate(D.VelvetNoise(sample_rate_hz=FS, num_outs=3, filtered_channels=(0, 1, 2), seed=1))
    assert not opt._is_vn_rms_candidate(_rms(fc=(0, 0)))
    assert not opt._is_vn_rms_candidate(_rms(fc=(0, 2)))
    assert not opt._is_vn_rms_candidate(_rms(normalizer=partial(rms_normalize, mode="STEREO")))
    assert not opt._is_vn_rms_candidate(_rms(normalizer=partial(rms_normalize)))
    assert not opt._is_vn_rms_candidate(D.HaasEffect(sample_rate_hz=FS))
    assert not opt._is_vn_stereo_candidate(_rms())


# ------------------------------------------------------------------ CPU: exceptions before any device work


def test_errors_before_device_work(no_device):
    n = max(2, opt._RMS_FAMILY_MIN)
    three = np.zeros((10, 3), np.float32)
    with pytest.raises(ValueError, match=r"operands could not be broadcast together with shapes \(10,2\) \(3,\)"):
        opt.grid_scan(three, [_rms(mode="LR", kappa=k / 5) for k in range(n)], **KW)
    with pytest.raises(IndexError, match="index 1 is out of bounds for axis 1 with size 1"):
        opt.grid_scan(np.zeros((10, 1), np.float32), [_rms(mode="LR", kappa=k / 5) for k in range(n)], **KW)
    with pytest.raises(ValueError, match=r"Expected shape \(num samples, 2\), but got shape \(10, 3\)"):
        opt.grid_scan(three, [_rms(mode="MS", kappa=k / 5) for k in range(n)], **KW)


def test_public_helper_rejects_other_candidates(no_device):
    x = _signal(10)
    with pytest.raises(ValueError, match="normalizer=rms_normalize"):
        opt.vn_stereo_rms_objective_partials(x, [_rms(), _rms(normalizer=None)])
    with pytest.raises(ValueError, match="identity"):
        opt.vn_stereo_rms_objective_partials(x, [_rms(), _rms(env=IDENTITY_ENVELOPE)])
    with pytest.raises(ValueError, match="pairwise"):
        opt.vn_stereo_rms_objective_partials(np.asfortranarray(x), [_rms()])
    with pytest.raises(ValueError, match="operands could not be broadcast"):
        opt.vn_stereo_rms_objective_partials(np.zeros((10, 3), np.float32), [_rms(mode="LR")])
    assert "vn_stereo_rms_objective_partials" in opt.__all__


# ------------------------------------------------------------------ CPU: C ABI argument checks


def test_abi_checks_arguments_before_any_launch():
    try:
        lib = N.lib()
    except N.VndError:
        pytest.skip("library not built")
    x = np.zeros((2, 8), np.float32)
    out = np.zeros((4, 12))
    gains = np.zeros((2, 2), np.float32)
    prog = opt._batch_program([_rms().tap_program(8), _rms().tap_program(8)])
    ps = prog.host_struct()
    asc = prog.host_struct()
    asc.order = N.ORDER_ASCENDING
    cands = np.zeros(2, dtype=N.VN_STEREO_CAND_DTYPE)
    p = C.c_void_p
    X, CD, G_, O_ = p(x.ctypes.data), p(cands.ctypes.data), p(gains.ctypes.data), p(out.ctypes.data)
    bad = [  # (x, frames, chan_stride, program, cands, n_cand, gains, partials)
        (X, 8, 8, C.byref(ps), CD, 1, G_, O_),       # the program has 4 channels, one candidate needs 2
        (X, 8, 8, C.byref(asc), CD, 2, G_, O_),      # not SEGMENTED
        (X, 0, 8, C.byref(ps), CD, 2, G_, O_),       # empty clip
        (X, -3, 8, C.byref(ps), CD, 2, G_, O_),
        (X, 8, 4, C.byref(ps), CD, 2, G_, O_),       # overlapping channels
        (None, 8, 8, C.byref(ps), CD, 2, G_, O_),
        (X, 8, 8, None, CD, 2, G_, O_),
        (X, 8, 8, C.byref(ps), None, 2, G_, O_),
        (X, 8, 8, C.byref(ps), CD, 2, None, O_),
        (X, 8, 8, C.byref(ps), CD, 2, G_, None),
    ]
    before = N.launch_count()
    for args in bad:
        assert lib.vnd_vn_stereo_rms_objective_dev(*args, None, 0, None) == N.VND_EINVAL, args
        assert lib.vnd_vn_stereo_rms_objective_host(None, *args) == N.VND_EINVAL, args
    assert N.launch_count() == before
    nbytes = C.c_size_t()
    assert lib.vnd_vn_stereo_rms_objective_workspace(-1, 2, C.byref(nbytes)) == N.VND_EINVAL
    assert lib.vnd_vn_stereo_rms_objective_workspace(8, 2, None) == N.VND_EINVAL


# ------------------------------------------------------------------ GPU: every score equals the candidate's own


@gpu
@pytest.mark.parametrize("frames", LENGTHS)
@pytest.mark.parametrize("env", ["default", "identity", "long"])
def test_scores_equal_the_single_path(frames, env):
    cands = _family(ENVELOPES[env])
    x = _signal(frames, seed=frames)
    _assert_same(opt.grid_scan(x, cands, **KW), x, cands)


@gpu
def test_strength_and_seed_sweeps():
    x = _signal(30000, seed=11)
    strengths = [D.VelvetNoise(sample_rate_hz=FS, log_distribution_strength=k, seed=1) for k in np.linspace(0.0, 3.0, 40)]
    _assert_same(opt.grid_scan(x, strengths, **KW), x, strengths)
    seeds = [D.VelvetNoise(sample_rate_hz=FS, seed=s) for s in range(40)]
    _assert_same(opt.grid_scan(x, seeds, **KW), x, seeds)


@gpu
def test_excerpts_and_input_kinds():
    import torch

    cands = _family()
    for name in ("viola", "guitar", "vocal"):
        _, clip = G.wav(name)
        clip = clip[: 3 * FS]
        _assert_same(opt.grid_scan(clip, cands, **KW), clip, cands)
    rng = np.random.default_rng(5)
    mono = (rng.standard_normal(5000) * 0.3).astype(np.float32)
    i16 = rng.integers(-3000, 3000, size=(5000, 2)).astype(np.int16)
    f64 = rng.standard_normal((5000, 2)) * 0.2
    planar = np.asfortranarray(_signal(5000, seed=8))
    for x in (mono, i16, f64, planar):
        _assert_same(opt.grid_scan(x, cands, **KW), x, cands)
    x = _signal(9000, seed=2)
    xt = torch.from_numpy(x).cuda()
    _assert_same(opt.grid_scan(xt, cands, **KW), xt, cands)
    _assert_same(opt.grid_scan(xt.t().contiguous().t(), cands, **KW), xt.t().contiguous().t(), cands)  # planar tensor
    p, g = opt.vn_stereo_rms_objective_partials(xt, cands[:5])
    assert isinstance(p, torch.Tensor) and p.is_cuda and p.shape == (5, N.OBJ_SLOTS) and p.dtype == torch.float64
    assert isinstance(g, torch.Tensor) and g.is_cuda and g.shape == (5, 2) and g.dtype == torch.float32
    pn, gn = opt.vn_stereo_rms_objective_partials(x, cands[:5])
    assert isinstance(pn, np.ndarray) and _same_bits(p.cpu().numpy(), pn) and _same_bits(g.cpu().numpy(), gn)


@gpu
def test_extreme_signals():
    cands = _family()
    rng = np.random.default_rng(12)
    silent = np.zeros((6000, 2), np.float32)
    _assert_same(opt.grid_scan(silent, cands, **KW), silent, cands)
    assert not np.any(opt.vn_stereo_rms_objective_partials(silent, cands)[1])
    apart = _signal(6000, seed=3)
    apart[:, 1] *= 1e-3  # 60 dB
    subnormal = (rng.standard_normal((6000, 2)) * 3e-21).astype(np.float32)  # squares below FLT_MIN
    bad = _signal(6000, seed=4)
    bad[100, 0] = np.nan
    bad[4500, 1] = np.inf
    inf_only = _signal(6000, seed=5)
    inf_only[2000, 0] = -np.inf
    for x in (apart, subnormal, bad, inf_only):
        with np.errstate(all="ignore"):
            _assert_same(opt.grid_scan(x, cands, **KW), x, cands)


# ------------------------------------------------------------------ GPU: partials and gains bit for bit


@gpu
def test_partials_and_gains_bit_for_bit():
    for frames in (7, 5000, 3 * OBJ_TILE + 5):
        x = _signal(frames, seed=frames + 3)
        cands = _family()
        parts, gains = opt.vn_stereo_rms_objective_partials(x, cands)
        n = np.float64(frames)
        for j, d in enumerate(cands):
            y = d.decorrelate(x)
            assert _same_bits(parts[j], _identity_partials(y)), (frames, j)
            raw = np.asarray(_rms(mode=d.mode, fc=d.filtered_channels, width=d.width, env=d.segment_envelope, kappa=d.log_distribution_strength,
                                  seed=d.seed, normalizer=None).decorrelate(x))
            for c in range(2):  # rms_match's dtype chain on seq_sumsq_f32 sums (rms_gain_f32)
                mx = np.float32(np.float64(O.seq_sumsq_f32(x[:, c])) / n)
                my = np.float32(np.float64(O.seq_sumsq_f32(raw[:, c])) / n)
                want = np.float32(np.sqrt(mx) / np.sqrt(np.float32(my + np.float32(1e-10))))
                assert _same_bits(gains[j, c], want), (frames, j, c, gains[j, c], want)


@gpu
def test_rows_do_not_depend_on_grouping():
    x = _signal(7000, seed=21)
    rng = np.random.default_rng(0)
    cands = [_rms(mode=("LR", "MS")[k % 2], fc=((0, 1), (0,), ())[k % 3], width=(None, 0.3)[k % 2], kappa=float(rng.uniform(0, 3)), seed=k % 7)
             for k in range(400)]
    parts, gains = opt.vn_stereo_rms_objective_partials(x, cands)
    perm = rng.permutation(len(cands))
    p2, g2 = opt.vn_stereo_rms_objective_partials(x, [cands[i] for i in perm])
    assert _same_bits(p2, parts[perm]) and _same_bits(g2, gains[perm])
    for size in (2, 15, 16, 31, 400):
        for lo in range(0, len(cands), size):
            p3, g3 = opt.vn_stereo_rms_objective_partials(x, cands[lo:lo + size])
            assert _same_bits(p3, parts[lo:lo + size]) and _same_bits(g3, gains[lo:lo + size]), (size, lo)


# ------------------------------------------------------------------ GPU: launches, kernels, fallback, oracle


@gpu
@pytest.mark.parametrize("k", [2, 40, 1000])
def test_three_launches(k):
    import torch
    from tests.test_fir_kernels import launched

    x = _signal(20000, seed=6)
    cands = [D.VelvetNoise(sample_rate_hz=FS, log_distribution_strength=i / k, seed=1 + i % 3) for i in range(k)]
    before = N.launch_count()
    opt.vn_stereo_rms_objective_partials(x, cands)
    assert N.launch_count() - before == 3
    xt = torch.from_numpy(x).cuda()
    want = {"vn_rms_sums_kernel", "vn_stereo_objective_kernel<true>", "obj_combine_kernel"}
    for _ in range(3):  # the profiler now and then loses a session's records (tests/test_fir_kernels.py)
        names, _ = launched(lambda: opt.vn_stereo_rms_objective_partials(xt, cands))
        if names:
            break
    assert want <= names and not any(n.startswith("vn_stereo_kernel") or "sumsq" in n or "place" in n for n in names), names


@gpu
def test_halo_fallback():
    x = _signal(40000, seed=13)
    cands = [_rms(kappa=k / 3, seed=k) for k in range(3)]
    long = [D.VelvetNoise(sample_rate_hz=FS, duration_seconds=0.6, seed=k) for k in range(max(2, opt._RMS_FAMILY_MIN))]
    with pytest.raises(N.VndError, match="does not fit") as e:
        opt.vn_stereo_rms_objective_partials(x, long)
    assert e.value.status == N.VND_EUNSUPPORTED
    _assert_same(opt.grid_scan(x, long + cands, **KW), x, long + cands)


@gpu
def test_scores_against_the_oracle():
    x = _signal(20000, seed=4)
    cands = [_rms(mode="MS", width=0.4), _rms(mode="LR", fc=()), _rms(), _rms(mode="LR", fc=(0,), width=0.8)]
    for d, s in zip(cands, opt.grid_scan(x, cands, **KW)):
        taps = O.class_taps(sample_rate_hz=FS, num_segments=len(d.segment_envelope), log_distribution_strength=d.log_distribution_strength,
                            filtered_channels=d.filtered_channels, seed=d.seed)
        y = O.vn_decorrelate(x, taps, envelope=d.segment_envelope, ms_mode=d.mode == "MS", width=d.width)
        assert abs(float(s) - float(O.objective(y, **KW))) <= 5e-4
