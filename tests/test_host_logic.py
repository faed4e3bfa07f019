"""CPU-only tests of the host side: tap generation and program packing against the reference
fixtures, the reference-facing API contracts (names, errors, laziness), and the C ABI surface
(library loads, every declared symbol is exported, no compute without a GPU)."""

from __future__ import annotations

import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle import vnd_oracle as O
from tests import _golden as G
from vndecorrelate_b200 import _native as N
from vndecorrelate_b200 import taps as T

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _has_gpu() -> bool:
    n = C.c_int(0)
    return N.lib().vnd_device_count(C.byref(n)) == 0 and n.value > 0


# ------------------------------------------------------------------ tap tables


def _table(**kw):
    base = dict(sample_rate_hz=44100, duration_seconds=0.03, num_impulses=30, num_outs=2, num_segments=4,
                log_distribution_strength=1.0, filtered_channels=(0, 1), seed=1)
    base.update(kw)
    return T.generate_tap_table(**base)


def test_tables_match_reference():
    t = _table()
    assert np.array_equal(t.rows(), G.tables()["cfg1"])
    t3 = _table(sample_rate_hz=48000, num_outs=4096, filtered_channels=tuple(range(4096)))
    assert G.sha(t3.rows()) == G.hashes()["tables"]["cfg3"]["sha256"]
    t4 = _table(sample_rate_hz=96000, duration_seconds=0.3, num_impulses=300, num_outs=4, filtered_channels=(0, 1, 2, 3))
    assert G.sha(t4.rows()) == G.hashes()["tables"]["cfg4_4ch"]["sha256"]
    for k in (0.0, 0.123, 0.5, 1.0):
        tk = _table(sample_rate_hz=48000, log_distribution_strength=k, filtered_channels=(0,))
        assert np.array_equal(tk.rows(), G.tables()[f"cand_{k}"])
        assert tk[1] == []


def test_cfg5_candidate_tables_hash():
    import hashlib

    h = hashlib.sha256()
    for k in np.linspace(0.0, 1.0, 1024):
        h.update(_table(sample_rate_hz=48000, log_distribution_strength=k, filtered_channels=(0,)).rows().tobytes())
    assert h.hexdigest() == G.hashes()["tables"]["cfg5_1024_candidates"]["sha256_concat"]


def test_table_is_sliced_not_regenerated_per_shard():
    """Channel c of a 2-channel generator is NOT channel c of a wider one with the same seed
    (decorrelation.py:510-520), so shards must slice one table."""
    narrow = _table()
    wide = _table(num_outs=4, filtered_channels=(0, 1, 2, 3))
    assert not np.array_equal(narrow.index[0], wide.index[0])
    prog = T.segmented_program(wide, O.DEFAULT_ENVELOPE, 10000)
    part = prog.slice_channels(2, 4)
    full_rows = wide.rows()
    assert part.channels == 2 and part.offsets[0] == 0
    want = T.segmented_program(
        T.TapTable(wide.fir_length_samples, 30, 4, wide.filtered[2:], wide.index[2:], wide.positive[2:], wide.segment), O.DEFAULT_ENVELOPE, 10000)
    assert np.array_equal(part.words, want.words) and np.array_equal(part.offsets, want.offsets)
    assert len(full_rows) == 120


def test_filtered_channel_quirk():
    with pytest.raises(IndexError):
        _table(filtered_channels=(1,))


@pytest.mark.parametrize("name", ["gen_cfg1", "gen_g3", "gen_trunc"])
def test_generate_velvet_noise(name):
    meta = G.hashes()["tables"][name]
    kw = dict(meta["kwargs"])
    if "segment_envelope" in kw:
        kw["segment_envelope"] = tuple(kw["segment_envelope"])
    f = T.generate_dense_fir(**kw)
    assert list(f.shape) == meta["shape"] and f.dtype == np.float32
    assert np.array_equal(np.argwhere(f != 0).astype(np.int32), G.tables()[name + "_nz"])
    assert np.array_equal(f[f != 0], G.tables()[name + "_val"])


# ------------------------------------------------------------------ program packing (interpreted on the CPU)


def _interpret(prog: T.TapProgram, x: np.ndarray) -> np.ndarray:
    """Executes a tap program the way the kernels are specified to (include/vnd_b200.h), in numpy,
    so that the packing can be checked against the oracle without a GPU."""
    n = len(x)
    y = np.zeros((n, prog.channels), dtype=np.float32)
    for c in range(prog.channels):
        w = prog.words[prog.offsets[c] : prog.offsets[c + 1]]
        if len(w) == 0:
            y[:, c] = x[:, c]
            continue
        if prog.order == N.ORDER_SEGMENTED:
            S = int(w[0])
            tp = 1 + 3 * S
            for s in range(S):
                nn, npos, gbits = int(w[1 + 3 * s]), int(w[2 + 3 * s]), w[3 + 3 * s : 4 + 3 * s]
                acc = np.zeros(n, dtype=np.float32)
                for i in w[tp : tp + nn]:
                    acc[: n - i] -= x[i:, c]
                tp += nn
                for i in w[tp : tp + npos]:
                    acc[: n - i] += x[i:, c]
                tp += npos
                if prog.apply_gain:
                    acc *= gbits.view(np.float32)[0]
                y[:, c] += acc
        else:
            K = int(w[0])
            for k in range(K):
                i = int(w[1 + 3 * k])
                coef = np.array([w[2 + 3 * k], w[3 + 3 * k]], dtype=np.int32).view(np.float64)[0]
                v = np.float32(coef) if prog.order == N.ORDER_ASCENDING else coef
                y[: n - i, c] += x[i:, c] * v
    return y


@pytest.mark.parametrize("c", G.case_list("vn_convolve"), ids=lambda c: f"case{c['id']}")
def test_segmented_program_semantics(c):
    x, y = G.case_xy(c)
    p = c["params"]
    t = _table(num_outs=p["num_outs"], filtered_channels=tuple(p["filtered_channels"]), seed=p["seed"])
    prog = T.segmented_program(t, O.DEFAULT_ENVELOPE, len(x))
    assert prog.halo <= len(x) and prog.channels == p["num_outs"]
    assert G.same_bits(_interpret(prog, x), y)


@pytest.mark.parametrize("c", G.case_list("fn_convolve"), ids=lambda c: f"case{c['id']}")
def test_ascending_program_semantics(c):
    x, y = G.case_xy(c)
    fir = G.cases()[1][c["params"]["fir"]]
    prog = T.ascending_program(fir, len(x))
    assert prog.order == (N.ORDER_ASCENDING if fir.dtype == np.float32 else N.ORDER_ASCENDING_F64)
    assert G.same_bits(_interpret(prog, x), y)


def test_program_drops_empty_segments_and_long_taps():
    t = _table(duration_seconds=0.5, num_impulses=15)  # 22 050-sample filter
    prog = T.segmented_program(t, O.DEFAULT_ENVELOPE, 1000)
    assert prog.halo <= 1000
    w = prog.words[: prog.offsets[1]]
    S = int(w[0])
    assert S < 4 and all(int(w[1 + 3 * s]) + int(w[2 + 3 * s]) > 0 for s in range(S))
    ident = T.segmented_program(t, (1.0,), 30000)
    assert ident.apply_gain == 0
    one = _table(duration_seconds=0.5, num_impulses=15, num_segments=1)
    lst = T.segmented_program(one, [1.0], 30000)  # a list is not the identity tuple: multiplied by 1.0
    assert lst.apply_gain == 1
    with pytest.raises(IndexError):
        T.segmented_program(t, (0.5, 0.25), 30000)


def test_candidate_program_layout():
    tables = [_table(sample_rate_hz=48000, log_distribution_strength=k, filtered_channels=(0,)) for k in (0.0, 0.5, 1.0)]
    prog = T.candidate_program(tables, O.DEFAULT_ENVELOPE, 48000)
    assert prog.channels == 3 and prog.offsets[-1] == prog.words.size
    for i, t in enumerate(tables):
        one = T.segmented_program(T.TapTable(t.fir_length_samples, 30, 4, t.filtered[:1], t.index[:1], t.positive[:1], t.segment), O.DEFAULT_ENVELOPE, 48000)
        assert np.array_equal(prog.words[prog.offsets[i] : prog.offsets[i + 1]], one.words)


# ------------------------------------------------------------------ reference-facing API contracts (no device needed)


def test_velvet_noise_contracts():
    from vndecorrelate_b200.decorrelation import VelvetNoise

    vn = VelvetNoise(sample_rate_hz=44100, seed=1)
    assert vn._generate() == vn._velvet_noise  # tests/test_decorrelation.py:56-68
    assert VelvetNoise(sample_rate_hz=44100, seed=2)._velvet_noise != vn._velvet_noise
    assert VelvetNoise(sample_rate_hz=44100, log_distribution_strength=0.0, seed=1)._velvet_noise != vn._velvet_noise
    before = vn._velvet_noise
    _ = vn.FIR
    assert vn.velvet_noise is before  # generated once, tests/test_decorrelation.py:161-169
    assert VelvetNoise(duration_seconds=0.03, num_impulses=30, sample_rate_hz=44100).density == 1000
    v = VelvetNoise(sample_rate_hz=44100, duration_seconds=0.055, num_impulses=45, seed=6)
    assert 818.19 > v.density > 818.18
    assert v.FIR.shape == (2426, 2) and np.count_nonzero(v.FIR[:, 0]) == 45
    assert G.same_bits(v.FIR, G.tables()["fir_prop_055_45_seed6"])
    with pytest.raises(ValueError):
        VelvetNoise(duration_seconds=0.03, num_impulses=700, sample_rate_hz=44100)
    vn.num_impulses = 20  # triggers regeneration on next access (decorrelation.py:368-379)
    assert vn.velvet_noise.num_impulses == 20
    assert VelvetNoise(sample_rate_hz=44100, segment_envelope=()).segment_envelope == (1.0,)
    with pytest.raises(ValueError):  # MS mode needs a stereo pair (utils/dsp.py:57-58)
        VelvetNoise(sample_rate_hz=44100, num_outs=4, filtered_channels=(0, 1, 2, 3)).decorrelate(np.zeros((10, 4), np.float32))


def test_signal_chain_contracts():
    from vndecorrelate_b200.decorrelation import HaasEffect, SignalChain, VelvetNoise, _fusable

    with pytest.raises(TypeError):
        SignalChain(sample_rate_hz=44100, _decorrelators=[])
    with pytest.raises(TypeError):
        SignalChain(sample_rate_hz=44100).velvet_noise(sample_rate_hz=48000)
    chain = SignalChain(sample_rate_hz=44100).velvet_noise(seed=1).haas_effect(delay_time_seconds=0.02)
    assert all(callable(d) and not isinstance(d, (VelvetNoise, HaasEffect)) for d in chain._decorrelators)  # lazy
    chain._init_decorrelators()
    assert isinstance(chain._decorrelators[0], VelvetNoise) and isinstance(chain._decorrelators[1], HaasEffect)
    assert _fusable(*chain._decorrelators)
    assert not _fusable(chain._decorrelators[0], HaasEffect(sample_rate_hz=44100, mode="MS"))
    assert not _fusable(chain._decorrelators[0], HaasEffect(sample_rate_hz=44100, width=0.5))
    hot = SignalChain(sample_rate_hz=44100, lazy=False).velvet_noise(seed=1)
    assert isinstance(hot._decorrelators[0], VelvetNoise)
    bad = SignalChain(sample_rate_hz=44100).velvet_noise(num_outs=2)  # error surfaces at first call, as in the reference
    with pytest.raises(TypeError):
        bad(np.zeros(10))
    with pytest.raises(NotImplementedError):
        SignalChain(sample_rate_hz=44100).white_noise(duration_seconds=0.03)
    assert HaasEffect(sample_rate_hz=44100, delay_time_seconds=0.02).delay_len_samples == 882


def test_function_path_contracts():
    from vndecorrelate_b200.decorrelation import convolve_velvet_noise, generate_velvet_noise

    fir = generate_velvet_noise(duration_seconds=0.03, num_impulses=30, seed=1)
    assert fir.shape == (1323, 2) and fir.dtype == np.float32
    with pytest.raises(IndexError):  # 1-D input, decorrelation.py:650
        convolve_velvet_noise(np.zeros(100, np.float32), fir)
    with pytest.raises(ValueError):  # channel mismatch, utils/dsp.py:305-310
        convolve_velvet_noise(np.zeros((100, 3), np.float32), fir)


def test_local_minima_rule():
    from vndecorrelate_b200.optimization import get_local_minima

    assert get_local_minima(np.array([3.0, 1.0, 2.0, 0.5, 4.0]), 5) == [1, 3]
    assert get_local_minima(np.array([0.0, 1.0, 2.0, 3.0]), 4) == [0]  # no interior minimum -> argmin
    assert get_local_minima(np.array([1.0, 1.0, 1.0]), 3) == [0]  # strict comparisons


def test_score_combination_matches_reference_dtype_chain():
    """The scalar combination applied to partial sums computed from the reference's own terms
    reproduces the reference's float32 score (viola, SURVEY.md Appendix C)."""
    from vndecorrelate_b200.optimization import _vn_score

    for row in G.objective()["viola_vn"]:
        p = np.zeros(12)
        p[0] = row["sum_r"]
        p[1], p[2], p[3] = row["centroid"] * row["sum_r"], row["spread"] * row["sum_r"], row["m3"] * row["sum_r"]
        p[4], p[5] = row["dot_lr"], row["norm_l"] ** 2
        p[6], p[7] = np.tan(np.float64(row["max_abs_theta"])), 1.0  # a frame whose angle is the recorded maximum
        p[8], p[9] = 0.0, 1.0
        got = _vn_score(p, angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)
        assert isinstance(got, np.float32)
        assert abs(float(got) - row["objective"]) <= 2e-4


# ------------------------------------------------------------------ C ABI surface


def _declared_functions():
    text = open(os.path.join(ROOT, "include", "vnd_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(vnd_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    names = _declared_functions()
    assert len(names) >= 25
    lib = N.lib()
    for n in names:
        assert hasattr(lib, n), f"{n} is declared in include/vnd_b200.h but not exported"
    assert set(names) == set(N.SIGNATURES), set(names) ^ set(N.SIGNATURES)
    assert lib.vnd_abi_version() == 1
    assert b"sm_100a" in lib.vnd_version()
    assert lib.vnd_status_string(N.VND_EPROGRAM) == b"malformed tap program"


def test_struct_layouts_match_header():
    assert C.sizeof(N.SignalStruct) == 40
    assert C.sizeof(N.TapProgramStruct) == 48
    assert C.sizeof(N.EpilogueStruct) == 32


def test_argument_errors_do_not_need_a_device():
    lib = N.lib()
    n = C.c_size_t()
    assert lib.vnd_vn_decorrelate_workspace(-1, 2, C.byref(N.EpilogueStruct()), C.byref(n)) == N.VND_EINVAL
    assert b"negative" in lib.vnd_last_error()
    assert lib.vnd_ctx_create(0, None) == N.VND_EINVAL


@pytest.mark.skipif(_has_gpu(), reason="this checks the behaviour WITHOUT a device")
def test_no_gpu_means_loud_failure_not_fallback():
    from vndecorrelate_b200.decorrelation import VelvetNoise

    h = C.c_void_p()
    assert N.lib().vnd_ctx_create(0, C.byref(h)) == N.VND_ECUDA
    assert b"no CPU fallback" in N.lib().vnd_last_error()
    with pytest.raises(N.VndError):
        VelvetNoise(sample_rate_hz=44100, seed=1).decorrelate(np.zeros((100, 2), np.float32))


# ------------------------------------------------------------------ lock-step Brent refinement


def _lockstep(lows, highs, f):
    """optimization._BrentBatch run to the end on the objectives ``f(i, x)`` (minimiser ``i`` at abscissa ``x``): its
    results, the abscissae each minimiser was evaluated at, and the size of every round."""
    from vndecorrelate_b200.optimization import _BrentBatch

    eng = _BrentBatch(lows, highs, 1e-4)
    seen, sizes = [[] for _ in range(len(lows))], []
    while True:
        idx, xs = eng.pending()
        if len(idx) == 0:
            return eng.results(), seen, sizes
        sizes.append(len(idx))
        for i, x in zip(idx, xs.tolist()):
            seen[i].append(x)
        eng.feed(idx, np.array([f(i, x) for i, x in zip(idx, xs.tolist())]))


def test_lockstep_minimize_equals_scipy_one_at_a_time():
    """The lock-step engine runs scipy's own bounded minimiser per interval, so abscissae, values and
    evaluation counts must equal the sequential loop of the reference (optimization.py:131-155),
    including on a piecewise-constant objective like the velvet-noise one; and the refinement built on it picks, clip
    by clip and whatever the number of lanes, what optimize_local_minima picks."""
    from scipy.optimize import minimize_scalar

    from vndecorrelate_b200.optimization import _refine_minima, optimize_local_minima

    def f(x):
        return np.float32(np.floor(40.0 * np.sin(7.0 * x) ** 2) / 40.0 + 0.3 * (x - 0.55) ** 2)

    bounds = [(0.0, 0.1), (0.1, 0.35), (0.3, 0.5), (0.45, 0.7), (0.7, 1.0), (0.2, 0.2000001)]
    (x, fun, nfev, _), _, calls = _lockstep([lo for lo, _ in bounds], [hi for _, hi in bounds], lambda i, x: f(x))
    for i, (lo, hi) in enumerate(bounds):
        want = minimize_scalar(fun=f, bounds=(lo, hi), method="bounded", options={"xatol": 1e-4})
        assert x[i] == want.x and fun[i] == want.fun and nfev[i] == want.nfev
    assert calls[0] == len(bounds) and sum(calls) == nfev.sum()  # every batch holds all live minimisers
    assert len(calls) == nfev.max()

    # selection rule of the reference: bounds from the grid neighbours, first strictly best wins
    grid = np.linspace(0.0, 1.0, 21)
    fc = [lambda x, c=c: f(x + 0.07 * c) for c in range(5)]  # one objective per clip
    minima = []
    for g in fc:
        scores = np.array([g(x) for x in grid])
        minima.append([i for i in range(1, 20) if scores[i] < scores[i - 1] and scores[i] < scores[i + 1]])
        assert minima[-1]
    want = [optimize_local_minima(m, grid, 21, g) for m, g in zip(minima, fc)]
    for lanes in (1, 2, 3):
        got, rounds = _refine_minima(minima, grid, lambda clip_ids, xs: [fc[c](x) for c, x in zip(clip_ids, xs.tolist())], lanes=lanes)
        assert got.tolist() == want and rounds >= 1
    got, rounds = _refine_minima([], grid, lambda clip_ids, xs: [])
    assert got.shape == (0,) and rounds == 0


def test_lockstep_minimize_propagates_errors():
    from vndecorrelate_b200.optimization import _refine_minima

    def bad(clip_ids, xs):
        raise ValueError("boom")

    for lanes in (1, 2):
        with pytest.raises(ValueError, match="boom"):
            _refine_minima([[2], [5]], np.linspace(0.0, 1.0, 8), bad, lanes=lanes)


def test_pinned_output_pool_falls_back_without_a_device():
    """runtime.pinned_empty backs small results by page-locked memory; without a CUDA device (this container) the
    allocation fails and it must hand out an ordinary array and leave the pool's accounting untouched."""
    from vndecorrelate_b200 import runtime as R

    before = R._POOL_BYTES[0]
    a = R.pinned_empty((100, 2), np.float64)
    assert a.shape == (100, 2) and a.dtype == np.float64 and a.flags.writeable
    a[:] = 1.0
    try:
        import torch

        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if not has_gpu:
        assert R._POOL_BYTES[0] == before
    assert R.pinned_empty((0, 2), np.float32).shape == (0, 2)


def test_kappa_family_program_equals_table_by_table_packing():
    """taps.kappa_family_program (one vectorised pass for the candidates of optimize_velvet_noise) must produce the
    very program candidate_program builds from one VelvetNoise per candidate, or decline (None)."""
    from vndecorrelate_b200 import taps as T
    from vndecorrelate_b200.decorrelation import VelvetNoise

    rng = np.random.default_rng(0)
    identical = declined = 0
    for trial in range(48):
        fs = int(rng.choice([44100, 48000, 96000]))
        dur = float(rng.choice([0.004, 0.01, 0.03, 0.06]))
        n_imp = int(rng.choice([5, 16, 30]))
        env = [(0.85, 0.55, 0.35, 0.2), (1.0,), (0.9, -0.5), (0.5, 0.4, 0.3, 0.2, 0.1, 0.05)][trial % 4]
        seed = int(rng.integers(0, 100))
        kappas = rng.uniform(0, 1, 9)
        kappas[0], kappas[1] = 0.0, 1.0
        frames = int(rng.choice([100, 2000, 100000]))
        cands = [VelvetNoise(sample_rate_hz=fs, duration_seconds=dur, num_impulses=n_imp, log_distribution_strength=float(k), normalizer=None,
                             filtered_channels=(0,), mode="LR", seed=seed, segment_envelope=env) for k in kappas]
        want = T.candidate_program([d.velvet_noise for d in cands], cands[0].segment_envelope, frames)
        got = T.kappa_family_program(kappas, sample_rate_hz=fs, duration_seconds=dur, num_impulses=n_imp, envelope=cands[0].segment_envelope,
                                     seed=seed, frames=frames)
        if got is None:
            declined += 1
            continue
        identical += 1
        assert np.array_equal(got.words, want.words) and np.array_equal(got.offsets, want.offsets)
        assert (got.channels, got.order, got.apply_gain, got.halo, got.max_channel_words) == (
            want.channels, want.order, want.apply_gain, want.halo, want.max_channel_words)
    assert identical >= 10 and declined >= 1  # both branches exercised


def test_bounded_brent_batch_is_scipys_minimiser():
    """optimization._BrentBatch (the lock-step refinement) against scipy.optimize.minimize_scalar(method="bounded"),
    the routine the reference calls (optimization.py:144-149): same abscissae in the same order, same minimum, same
    value and dtype, same evaluation count and status - for float32-valued objectives (what the velvet-noise score is),
    float64-valued ones (Haas), plateaus with ties, and Python floats; the 25 objectives of a kind in one batch."""
    from scipy.optimize import minimize_scalar

    def make(kind, seed):
        c = np.random.default_rng(seed).uniform(0, 1, 4)
        if kind == 0:
            return lambda x: np.float32((x - c[0]) ** 2 + 0.01 * np.sin(50 * x * c[1]))
        if kind == 1:
            return lambda x: np.float32(np.abs(x - c[0]) + 0.3 * np.cos(37 * x))
        if kind == 2:
            return lambda x: float(np.sin(20 * x * c[2]) + x * c[3])
        if kind == 3:
            return lambda x: np.float32(np.round(np.sin(30 * x) * 8) / 8)
        return lambda x: np.float64(np.cos(11 * x * c[0]) * np.exp(-x) + c[1] * x * x)

    rng = np.random.default_rng(1)
    for kind in range(5):
        fs, lows, highs, wants, seen_ref = [], [], [], [], []
        for seed in range(25):
            f = make(kind, seed)
            lo = np.float64(rng.uniform(0, 0.5))
            hi = lo + np.float64(rng.uniform(1e-3, 0.5))
            seen_ref.append([])
            wants.append(minimize_scalar(fun=lambda x, f=f, s=seen_ref[-1]: (s.append(float(x)), f(x))[1], bounds=(lo, hi), method="bounded",
                                         options={"xatol": 1e-4}))
            fs.append(f)
            lows.append(lo)
            highs.append(hi)
        (x, fun, nfev, status), seen, _ = _lockstep(lows, highs, lambda i, x: fs[i](x))
        for i, want in enumerate(wants):
            assert seen[i] == seen_ref[i]
            assert x[i] == want.x
            assert fun[i] == want.fun and type(fun[i]) is type(want.fun)
            assert (nfev[i], status[i], status[i] == 0) == (want.nfev, want.status, want.success)


def test_lockstep_minimize_batches_all_minimisers():
    bounds = [(i / 64, (i + 2) / 64) for i in range(0, 62, 3)]
    (x, _, _, status), _, calls = _lockstep([lo for lo, _ in bounds], [hi for _, hi in bounds], lambda i, x: np.float32((x - 0.4) ** 2))
    assert len(x) == len(bounds) and np.all(status == 0)
    assert calls[0] == len(bounds) and calls == sorted(calls, reverse=True)  # everybody in the first round, finished ones drop out
    (x, fun, nfev, status), _, calls = _lockstep([], [], lambda i, x: np.float32(x))
    assert len(x) == len(fun) == len(nfev) == len(status) == 0 and calls == []


def test_vectorised_scores_equal_the_one_row_chain_bit_for_bit():
    """optimization._vn_scores_rows (all (clip, candidate) pairs at once) against _vn_score (one pair, the reference's
    scalar dtype chain, SURVEY.md A.5): identical float32 bits, including rows with and without a frame on the
    negative half plane and rows that exceed the angle limit."""
    import vndecorrelate_b200.optimization as OPT
    from vndecorrelate_b200 import _native as N

    kw = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)
    rng = np.random.default_rng(3)
    n = 6000
    p = np.zeros((n, N.OBJ_SLOTS))
    sr = rng.uniform(1e2, 1e6, n)
    p[:, 0] = sr
    p[:, 1] = sr * rng.normal(0, 0.3, n)
    p[:, 2] = sr * rng.uniform(0, 0.8, n)
    p[:, 3] = sr * rng.normal(0, 0.2, n)
    p[:, 5] = rng.uniform(1, 1e5, n)
    p[:, 4] = p[:, 5] * rng.uniform(-1, 1, n)
    p[:, 6] = np.float32(rng.uniform(0, 2, n))
    p[:, 7] = np.float32(rng.uniform(1e-6, 1, n))
    p[:, 8] = np.float32(rng.uniform(0, 2, n))
    p[:, 9] = np.float32(rng.uniform(1e-6, 1, n))
    untouched = rng.random(n) < 0.2
    p[untouched, 8], p[untouched, 9] = 0.0, 1.0
    want = np.array([OPT._vn_score(r, **kw) for r in p], dtype=np.float32)
    got = OPT.vn_scores_from_partials(p.reshape(60, 100, -1), **kw)
    assert got.dtype == np.float32 and got.shape == (60, 100)
    assert np.array_equal(got.reshape(-1).view(np.uint32), want.view(np.uint32))


def test_pinned_output_pool_recycles_blocks(monkeypatch):
    """The pool's life-cycle with a stand-in allocator (malloc instead of cudaHostAlloc): a block stays out while
    any view of the array lives, comes back when the last one dies, and is handed out again."""
    import ctypes as C
    import gc

    from vndecorrelate_b200 import _native as N
    from vndecorrelate_b200 import runtime as R

    libc = C.CDLL(None)
    libc.malloc.restype = C.c_void_p
    libc.malloc.argtypes = [C.c_size_t]

    freed = []

    class FakeLib:
        def vnd_ctx_host_alloc(self, handle, nbytes, out):
            C.cast(out, C.POINTER(C.c_void_p))[0] = libc.malloc(nbytes)
            return 0

        def vnd_host_free(self, ptr):
            freed.append(ptr.value)
            return 0

    class FakeCtx:
        handle = None

    monkeypatch.setattr(N, "lib", lambda: FakeLib())
    monkeypatch.setattr(R.HostContext, "get", classmethod(lambda cls, device=None: FakeCtx()))
    monkeypatch.setattr(R, "_POOL_FREE", {})
    monkeypatch.setattr(R, "_POOL_BYTES", [0])
    monkeypatch.setattr(R, "_POOL_CAP", [512 << 20])
    monkeypatch.setattr(R, "_POOL_WARNED", [False])
    a = R.pinned_empty((1000, 2), np.float32)
    assert a.flags.writeable and not a.flags.owndata and R._POOL_BYTES[0] == 1 << 16
    a[:] = 1.5
    ptr = a.ctypes.data
    view = a[10:20]
    del a
    gc.collect()
    assert sum(len(v) for v in R._POOL_FREE.values()) == 0 and float(view[0, 0]) == 1.5  # the view keeps the block
    del view
    gc.collect()
    assert sum(len(v) for v in R._POOL_FREE.values()) == 1
    b = R.pinned_empty((500, 4), np.float32)  # same block size: recycled, no new allocation
    assert b.ctypes.data == ptr and R._POOL_BYTES[0] == 1 << 16
    # at the cap: an idle block of another size class is released to make room ...
    del b
    gc.collect()
    R.set_pinned_pool_cap(1 << 17)
    c = R.pinned_empty((1 << 15,), np.float32)  # 128 KB: needs the 64 KB block gone
    assert not c.flags.owndata and freed == [ptr] and R._POOL_BYTES[0] == 1 << 17
    # ... and when nothing can be released the result is ordinary memory, with one warning
    with pytest.warns(ResourceWarning):
        d = R.pinned_empty((1000,), np.float32)
    assert d.flags.owndata and R._POOL_BYTES[0] == 1 << 17
    # a forked child forgets the parent's blocks instead of recycling their pointers
    R._pinned_pool_after_fork()
    assert R._POOL_FREE == {} and R._POOL_BYTES[0] == 0


def test_random_tap_tables_match_reference():
    """240 random (sample rate, duration, impulses, strength, seed, outputs, envelope) tuples: the class-path tap rows
    and the dense FIR of the function path hash to what the UNMODIFIED reference produced
    (tests/golden/make_golden_r02.py::random_tables)."""
    import json
    import os

    recs = json.load(open(os.path.join(G.GOLDEN, "tables_random.json")))
    assert len(recs) >= 200
    for rec in recs:
        p = rec["params"]
        t = T.generate_tap_table(sample_rate_hz=p["sample_rate_hz"], duration_seconds=p["duration_seconds"], num_impulses=p["num_impulses"],
                                 num_outs=p["num_outs"], num_segments=len(p["segment_envelope"]), log_distribution_strength=p["log_distribution_strength"],
                                 filtered_channels=tuple(p["filtered_channels"]), seed=p["seed"])
        rows = t.rows()
        assert rows.shape[0] == rec["class_rows_count"] and G.sha(rows) == rec["class_rows_sha256"], p
        fir = T.generate_dense_fir(duration_seconds=p["duration_seconds"], num_impulses=p["num_impulses"], num_outs=p["num_outs"],
                                   sample_rate_hz=p["sample_rate_hz"], segment_envelope=tuple(p["segment_envelope"]),
                                   log_distribution_strength=p["log_distribution_strength"], seed=p["seed"])
        assert list(fir.shape) == rec["dense_shape"] and G.sha(fir) == rec["dense_sha256"], p


def test_interval_grid_family_is_bitwise_the_single_strength_grid():
    """taps._interval_grid_family (one vectorised pass for all strengths of a sweep or of a Brent round) against the
    single-strength function, 20 000 strengths incl. the end points and Brent-like values."""
    rng = np.random.default_rng(3)
    ks = np.concatenate([np.linspace(0.0, 1.0, 1024), rng.uniform(0.0, 1.0, 20000), [0.0, 1.0, 1e-300, 0.5, 0.3201472263050255]])
    for n_imp, fir_len in ((30, 1440), (15, 1323), (300, 28800)):
        sub = ks if n_imp == 30 else ks[:3000]
        w, s = T._interval_grid_family(sub, n_imp, fir_len)
        for i in range(0, len(sub), 7):
            w1, s1 = T._interval_grid(float(sub[i]), n_imp, fir_len)
            assert np.array_equal(w1, w[i]) and np.array_equal(s1, s[i])


def test_array_brent_equals_scipy_abscissa_by_abscissa():
    """optimization._BrentBatch (every minimiser of every clip advanced by array arithmetic) against scipy's bounded
    minimiser run one objective at a time, on 2000 float32-valued, piecewise-constant noisy objectives (the shape the
    rounded-tap objective has) and 300 float64 ones: same abscissae in the same order, same x / fun / nfev / status, fun
    in the objective's dtype."""
    from scipy.optimize import minimize_scalar

    rng = np.random.default_rng(0)

    def make(dtype):
        c, s, step = rng.uniform(0, 1), rng.uniform(0.1, 50), rng.choice([0, 1e-3, 1e-2, 5e-2])
        off, tab = rng.uniform(600, 620), rng.standard_normal(4096) * rng.uniform(0, 1e-3)

        def f(x):
            xx = np.floor(x / step) * step if step > 0 else x
            return dtype(off + s * (xx - c) ** 2 + tab[int(abs(x) * 1e6) % 4096])

        return f

    for dtype, n in ((np.float32, 2000), (np.float64, 300)):
        fs = [make(dtype) for _ in range(n)]
        lo = rng.uniform(0, 0.9, n)
        hi = lo + rng.uniform(1e-3, 0.2, n)
        (x, fun, nfev, status), seen, _ = _lockstep(lo, hi, lambda i, x: fs[i](x))
        assert fun.dtype == dtype
        for i in range(n):
            seq = []
            want = minimize_scalar(fun=lambda v: (seq.append(float(v)), fs[i](v))[1], bounds=(lo[i], hi[i]), method="bounded",
                                   options={"xatol": 1e-4})
            assert seq == seen[i], i
            assert want.x == x[i] and want.fun == fun[i] and type(want.fun) is type(fun[i]) and want.nfev == nfev[i] and want.status == status[i], i


def test_fir_kernels_have_no_contracted_multiply_add():
    """Floating-point contract (DESIGN.md section 6): the reference rounds after every numpy ufunc, so no FIR / post-processing
    kernel may contain a multiply-add with a real addend.  ptxas was seen contracting a packed `mul.rn.f32x2` followed by
    `add.rn.f32x2` into FFMA2 (one rounding instead of two) despite -fmad=false when both landed in one basic block
    (vnd_fir_tmem.cu, compute_main); the only contraction that is harmless is `x * g + 0`.  Checked on the SASS of the built
    library (cuobjdump ships with the CUDA toolkit the library was built with)."""
    import shutil
    import subprocess

    cuobjdump = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    if not os.path.exists(cuobjdump):
        pytest.skip("no cuobjdump")
    sass = subprocess.run([cuobjdump, "-sass", N.LIB_PATH], capture_output=True, text=True, check=True).stdout
    functions = re.split(r"\n\s*Function : ", sass)[1:]
    checked = 0
    for f in functions:
        name = f.split("\n", 1)[0]
        if not re.search(r"fir_|vn_stereo|haas_kernel|place_kernel|stereo_ops", name) or "objective" in name:
            continue
        checked += 1
        bad = [ln.strip() for ln in f.split("\n") if re.search(r"\b[FD]FMA2?\b", ln) and not re.search(r"RZ(\.F32)?\s*;", ln)]
        assert not bad, f"{name}: contracted multiply-add(s), e.g. {bad[0]}"
    assert checked >= 10
