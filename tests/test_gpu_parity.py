"""Parity of the CUDA path (through the Python API and so through the C ABI) with the reference.

Every comparison is against (a) fixtures produced by the unmodified reference
(tests/golden/make_golden.py) or (b) the CPU oracle (oracle/vnd_oracle.py, itself pinned to those
fixtures) on the same seeded inputs.  Sample values are compared BIT-EXACTLY (dtype, shape and
bytes) — stricter than the 1e-6-of-full-scale the spec allows for fp32 — except the objective
scores, whose tolerance is written next to each assertion.  Needs a CUDA device: ``-m gpu``.
"""

from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from oracle import vnd_oracle as O
from tests import _golden as G
from tests.test_fir_kernels import DIRECT, RING, TILE, TMEM, WIN, predict_route, routed

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    import vndecorrelate_b200.decorrelation as D

    return D


def _vn_kwargs(p, extra=None):
    kw = {k: v for k, v in p.items() if k not in ("new_envelope_len",)}
    if "filtered_channels" in kw:
        kw["filtered_channels"] = tuple(kw["filtered_channels"])
    if "segment_envelope" in kw:
        kw["segment_envelope"] = tuple(kw["segment_envelope"])
    kw.update(extra or {})
    return kw


# ------------------------------------------------------------------ golden cases (numpy in/out)


@pytest.mark.parametrize("c", G.case_list("vn_convolve"), ids=lambda c: f"case{c['id']}")
def test_vn_convolve_cases(api, c):
    x, y = G.case_xy(c)
    got = api.VelvetNoise(**_vn_kwargs(c["params"])).convolve(x)
    assert G.same_bits(np.ascontiguousarray(got), y)


@pytest.mark.parametrize("c", G.case_list("vn_decorrelate"), ids=lambda c: f"case{c['id']}")
def test_vn_decorrelate_cases(api, c):
    x, y = G.case_xy(c)
    kw = _vn_kwargs(c["params"])
    if c["normalizer_none"]:
        kw["normalizer"] = None
    else:
        kw.pop("normalizer", None)
    got = api.VelvetNoise(**kw).decorrelate(x)
    assert G.same_bits(got, y)


def test_vn_envelope_swapped_after_construction(api):
    (c,) = G.case_list("vn_decorrelate_env_swap")
    x, y = G.case_xy(c)
    p = c["params"]
    vn = api.VelvetNoise(num_impulses=15, duration_seconds=0.5, sample_rate_hz=44100, segment_envelope=(1.0, 0.5, 0.25), seed=4)
    vn.segment_envelope = [1.0] * p["new_envelope_len"]
    assert G.same_bits(vn(x), y)


@pytest.mark.parametrize("c", G.case_list("haas"), ids=lambda c: f"case{c['id']}")
def test_haas_cases(api, c):
    x, y = G.case_xy(c)
    got = api.HaasEffect(**c["params"]).decorrelate(x)
    assert G.same_bits(got, y)


def test_chain_cases(api):
    (c,) = G.case_list("chain_cfg2")
    x, y = G.case_xy(c)
    chain = (api.SignalChain(sample_rate_hz=44100)
             .velvet_noise(duration_seconds=0.03, num_impulses=30, log_distribution_strength=1.0, seed=1)
             .haas_effect(delay_time_seconds=0.02, mode="LR"))
    assert G.same_bits(chain(x), y)
    (c,) = G.case_list("chain_example")
    x, y = G.case_xy(c)
    chain = (api.SignalChain(sample_rate_hz=44100)
             .velvet_noise(duration_seconds=0.02, num_impulses=30, seed=1, log_distribution_strength=1.0, mode="MS", filtered_channels=(0, 1))
             .haas_effect(delay_time_seconds=0.02, delayed_channel=1, mode="LR"))
    assert G.same_bits(chain(x), y)
    (c,) = G.case_list("chain_hetero")
    x, y = G.case_xy(c)
    chain = (api.SignalChain(sample_rate_hz=44100)
             .velvet_noise(duration_seconds=0.03, num_impulses=30, width=0.5, seed=5)
             .haas_effect(delay_time_seconds=0.0197, delayed_channel=1, mode="LR")
             .haas_effect(delay_time_seconds=0.0096, delayed_channel=1, mode="MS"))
    assert G.same_bits(chain(x), y)


@pytest.mark.parametrize("c", G.case_list("fn_convolve"), ids=lambda c: f"case{c['id']}")
def test_fn_convolve_cases(api, c):
    x, y = G.case_xy(c)
    fir = G.cases()[1][c["params"]["fir"]]
    got = api.convolve_velvet_noise(x, fir)
    assert G.same_bits(np.ascontiguousarray(got), y)


def test_reference_equality_test_of_both_paths(api):
    """tests/test_decorrelation.py:172-197 of the reference, on float64 input, atol 1e-6."""
    rng = np.random.default_rng(5)
    x = rng.random((10000, 2))
    kw = dict(duration_seconds=0.03, num_impulses=30, num_outs=2, sample_rate_hz=44100, segment_envelope=(0.85, 0.55, 0.35, 0.2),
              log_distribution_strength=1.0, seed=1)
    a = api.convolve_velvet_noise(x, api.generate_velvet_noise(**kw))
    b = api.VelvetNoise(**kw).convolve(x)
    assert a.shape == b.shape and np.allclose(a, b, atol=1e-6)
    assert np.allclose(api.VelvetNoise(**kw).FIR, api.generate_velvet_noise(**kw), atol=1e-6)  # :71-93


def test_helpers(api):
    from vndecorrelate_b200.utils import dsp

    (c,) = G.case_list("encode")
    xy, y = G.case_xy(c)
    t = xy[1].copy()
    dsp.encode_signal_to_side_channel(xy[0], t)
    assert G.same_bits(t, y)
    (c,) = G.case_list("width")
    x, y = G.case_xy(c)
    t = x.copy()
    dsp.apply_stereo_width(t, c["params"]["width"])
    assert G.same_bits(t, y)
    for c in G.case_list("rms"):
        xy, y = G.case_xy(c)
        t = xy[1].copy()
        dsp.rms_normalize(xy[0], t)
        assert G.same_bits(t, y)
    # float64 helpers and the LR<->MS round trip against the oracle
    rng = np.random.default_rng(3)
    a = rng.standard_normal((1001, 2))
    for fn, ofn in ((dsp.LR_to_MS, O.lr_to_ms), (dsp.MS_to_LR, O.ms_to_lr)):
        u, v = a.copy(), a.copy()
        fn(u)
        ofn(v)
        assert G.same_bits(u, v)
    u, v = a.copy(), a.copy()
    dsp.apply_stereo_width(u, 0.37)
    O.stereo_width(v, 0.37)
    assert G.same_bits(u, v)
    b = rng.standard_normal((1001, 2))
    u, v = b.copy(), b.copy()
    dsp.rms_normalize(a, u)
    O.rms_match(a, v)
    assert G.same_bits(u, v)


def _dsp_cases(kind):
    return [c for c in G.dsp_extra()[0] if c["kind"] == kind]


@pytest.mark.parametrize("c", _dsp_cases("rms_normalize") + _dsp_cases("peak_normalize"), ids=lambda c: f"{c['kind']}{c['id']}")
def test_normalisers_every_mode(api, c):
    """rms_normalize (STEREO, DUAL_MONO, 1-D) and peak_normalize against the reference's outputs
    (tests/golden/make_golden_r02.py::dsp_extra): same bytes - the axis=None statistics are summed in numpy's pairwise
    order on the device."""
    from vndecorrelate_b200.utils import dsp

    dtype = np.dtype(c["dtype"]).type
    x, y = G.dsp_inputs("rms_normalize", c["seed"], c["n"], dtype)
    mode = dsp.NormalizeMode(c["params"]["mode"])
    if c["kind"] == "rms_normalize":
        if c["params"]["ndim"] == 1:
            out = y[:, 0].copy()
            dsp.rms_normalize(x[:, 0].copy(), out)
        else:
            out = y.copy()
            dsp.rms_normalize(x, out, mode=mode)
    else:
        if c["params"]["ndim"] == 1:
            out = y[:, 1].copy()
            dsp.peak_normalize(out)
        else:
            out = y.copy()
            dsp.peak_normalize(out, mode=mode)
    assert G.sha(out) == c["sha256"]["y"], (c["params"], c["n"], c["dtype"])


@pytest.mark.parametrize("c", _dsp_cases("polar_coordinates"), ids=lambda c: f"polar{c['id']}")
def test_polar_coordinates(api, c):
    """polar_coordinates (utils/dsp.py:374-422) against the reference: radii and weights bit for bit (pairwise-order sum),
    angles within 2 float32 ulp / 4 float64 ulp of numpy's arctan2 at magnitude pi/2."""
    from vndecorrelate_b200.utils import dsp

    dtype = np.dtype(c["dtype"]).type
    l, r = G.dsp_inputs("polar_coordinates", c["seed"], c["n"], dtype)
    p = c["params"]
    rad, th, w = dsp.polar_coordinates(l, r, mode=p["mode"], semicircular=p["semicircular"], normalize=p["normalize"])
    assert rad.dtype == dtype and th.dtype == dtype and w.dtype == dtype and rad.shape == (c["n"],)
    assert G.sha(rad) == c["sha256"]["radii"]
    assert G.sha(w) == c["sha256"]["weights"]
    want_th = G.dsp_extra()[1][f"c{c['id']}_thetas"]
    tol = 4e-7 if dtype == np.float32 else 1e-15
    assert np.max(np.abs(th[:: c["stride"]].astype(np.float64) - want_th.astype(np.float64))) <= tol
    two = dsp.polar_coordinates(l, r, mode=p["mode"], semicircular=p["semicircular"], normalize=p["normalize"], compute_weights=False)
    assert len(two) == 2 and G.sha(two[0]) == c["sha256"]["radii"]


@pytest.mark.parametrize("frames", [100, 4099, 250_774])
def test_rms_order_follows_the_layout_like_numpy(api, frames):
    """numpy sums np.mean(np.square(a), axis=0) along the axis of the smallest stride: frame by frame (a sequential running
    sum) for a C-order (frames, 2) array, pairwise per column for a Fortran-ordered / planar one - 6e-5 apart in float32 on a
    250 k-frame file.  decorrelate() and rms_normalize() must follow the layout of each array the way the reference does."""
    from vndecorrelate_b200.utils import dsp

    rng = np.random.default_rng(frames)
    xc = (rng.standard_normal((frames, 2)) * 0.3).astype(np.float32)
    xf = np.asfortranarray(xc)                  # same values, planar in memory (what `planar_array.T` gives a user)
    taps = O.class_taps(sample_rate_hz=44100, seed=1)
    vn = api.VelvetNoise(sample_rate_hz=44100, duration_seconds=0.03, num_impulses=30, seed=1)
    want_c, want_f = O.vn_decorrelate(xc, taps), O.vn_decorrelate(xf, taps)
    assert G.same_bits(vn.decorrelate(xc), want_c)
    assert G.same_bits(vn.decorrelate(xf), want_f)
    if frames > 100000:
        assert not np.array_equal(want_c, want_f)  # the two orders really differ at this length
    import torch

    got_t = vn.decorrelate(torch.from_numpy(np.ascontiguousarray(xc.T)).cuda().t())  # planar CUDA tensor, (frames, 2) view
    assert G.same_bits(got_t.cpu().numpy(), want_f)
    # the helper itself, every combination of layouts, float32 and float64
    for dt in (np.float32, np.float64):
        y0 = (rng.standard_normal((frames, 2)) * 0.1).astype(dt)
        for x in (xc.astype(dt), np.asfortranarray(xc.astype(dt))):
            for y in (y0.copy(), np.asfortranarray(y0)):
                want = y.copy(order="K")
                O.rms_match(x, want)
                got = y.copy(order="K")
                dsp.rms_normalize(x, got)
                assert G.same_bits(np.ascontiguousarray(got), np.ascontiguousarray(want)), (dt, x.flags.f_contiguous, y.flags.f_contiguous)
                want = y.copy(order="K")  # STEREO mode: axis=None statistics run over the array in memory order
                O.rms_match(x, want, stereo_mode=True)
                got = y.copy(order="K")
                dsp.rms_normalize(x, got, mode=dsp.NormalizeMode.STEREO)
                assert G.same_bits(np.ascontiguousarray(got), np.ascontiguousarray(want)), ("stereo", dt, x.flags.f_contiguous, y.flags.f_contiguous)


def test_rms_normalize_reference_known_answers(api):
    """The reference's own test of rms_normalize (tests/test_dsp.py:119-142), float64: 1-D, DUAL_MONO, STEREO (known value
    0.55893258) and a 1-D input against a 2-D output in STEREO mode."""
    from vndecorrelate_b200.utils import dsp

    x = np.array([0.707, 0.707, 0.707])
    y = np.array([1.0, 1.0, 1.0])
    dsp.rms_normalize(x, y)
    assert np.allclose(x, y)
    x = np.array([[0.707, 0.3535], [0.707, 0.3535]])
    y = np.array([[1.0, 1.0], [1.0, 1.0]])
    dsp.rms_normalize(x, y, mode=dsp.NormalizeMode.DUAL_MONO)
    assert np.allclose(x, y)
    y = np.array([[1.0, 1.0], [1.0, 1.0]])
    dsp.rms_normalize(x, y, mode=dsp.NormalizeMode.STEREO)
    assert np.allclose(np.array([0.55893258, 0.55893258]), y)
    x = np.array([0.707, 0.707, 0.707])
    y = np.array([[1.0, 1.0], [1.0, 1.0]])
    want = y.copy()
    O.rms_match(x, want, stereo_mode=True)
    dsp.rms_normalize(x, y, mode=dsp.NormalizeMode.STEREO)
    assert x[0] == pytest.approx(y[0, 0]) and G.same_bits(y, want)


# ------------------------------------------------------------------ full-size wav goldens


def test_cfg1_viola_full(api):
    fs, x = G.wav("viola")
    vn = api.VelvetNoise(sample_rate_hz=fs, duration_seconds=0.03, num_impulses=30, seed=1)
    assert np.array_equal(vn.velvet_noise.rows(), G.tables()["cfg1"])
    assert G.sha(vn.convolve(x)) == G.hashes()["cfg1_convolve_viola"]
    y = vn.decorrelate(x)
    assert y.dtype == np.float32 and y.shape == x.shape
    assert G.sha(y) == G.hashes()["cfg1_decorrelate_viola"]


def test_cfg2_guitar_full(api):
    fs, x = G.wav("guitar")
    chain = (api.SignalChain(sample_rate_hz=fs)
             .velvet_noise(duration_seconds=0.03, num_impulses=30, log_distribution_strength=1.0, seed=1)
             .haas_effect(delay_time_seconds=0.02, mode="LR"))
    y = chain(x)
    h = G.hashes()["cfg2_chain_guitar"]
    assert list(y.shape) == h["shape"] and str(y.dtype) == h["dtype"]
    assert G.sha(y) == h["sha256"]


@pytest.mark.parametrize("name", ["viola", "vocal", "guitar"])
def test_reference_example_chain_goldens(api, name):
    """viola/vocal: the outputs the reference commits (audio/*_decorrelated.wav)."""
    fs, x = G.wav(name)
    chain = (api.SignalChain(sample_rate_hz=fs)
             .velvet_noise(duration_seconds=0.02, num_impulses=30, seed=1, log_distribution_strength=1.0, mode="MS", filtered_channels=(0, 1))
             .haas_effect(delay_time_seconds=0.02, delayed_channel=1, mode="LR"))
    y = chain(x)
    h = G.hashes()["example_chain"][name]
    assert list(y.shape) == h["shape"] and y.dtype == np.float64
    assert G.sha(y) == h["sha256"]


# ------------------------------------------------------------------ CUDA tensors, planar slabs, big halos


def test_torch_tensors_match_numpy_path(api):
    import torch

    fs, x = G.wav("vocal")
    xt = torch.from_numpy(x).cuda()
    vn = api.VelvetNoise(sample_rate_hz=fs, seed=1)
    y_np = vn.decorrelate(x)
    y_t = vn.decorrelate(xt)
    assert y_t.is_cuda and y_t.dtype == torch.float32
    assert G.same_bits(y_t.cpu().numpy(), y_np)
    assert G.same_bits(vn.convolve(xt).cpu().numpy(), vn.convolve(x))
    chain = api.SignalChain(sample_rate_hz=fs).velvet_noise(seed=1).haas_effect(delay_time_seconds=0.02)
    assert G.same_bits(chain(xt).cpu().numpy(), chain(x))
    h = api.HaasEffect(sample_rate_hz=fs, mode="MS", delayed_channel=1, width=0.4)
    assert G.same_bits(h(xt).cpu().numpy(), h(x))
    mono = xt[:, 0].contiguous()
    assert G.same_bits(vn.decorrelate(mono).cpu().numpy(), vn.decorrelate(x[:, 0].copy()))


@pytest.mark.parametrize("frames", [1, 255, 8191, 8192, 8193, 8447, 8448, 8449, 2 * 8448 - 1, 2 * 8448 + 1057, 3 * 8192 + 5, 5 * 8448])
def test_planar_slab_tile_edges(api, frames):
    """cfg3-style planar slab (time contiguous per channel, the TMA bulk-copy path) around the
    tile boundaries of the kernel, against the oracle."""
    import torch

    C = 6
    vn = api.VelvetNoise(sample_rate_hz=48000, duration_seconds=0.03, num_impulses=30, num_outs=C, filtered_channels=tuple(range(C)),
                         mode="LR", normalizer=None, seed=1)
    g = torch.Generator(device="cuda").manual_seed(1234)
    slab = torch.randn((C, frames), generator=g, device="cuda") * 0.1
    prog = vn.tap_program(frames)
    aligned = frames % 4 == 0  # the channel stride of the slab: bulk copies need a multiple of 16 bytes
    route = predict_route(frames, prog.halo, prog.max_channel_words, bulk=aligned, y_ok=aligned)
    y = routed(lambda: vn.convolve(slab.t()), route, f"{frames} frames")  # (frames, C) view of a planar slab
    assert y.shape == (frames, C) and y.stride(0) == 1 or frames == 1
    taps = O.class_taps(sample_rate_hz=48000, num_outs=C, filtered_channels=tuple(range(C)), seed=1)
    want = O.fir_class_order(np.ascontiguousarray(slab.cpu().numpy().T), taps, O.DEFAULT_ENVELOPE, C)
    assert G.same_bits(np.ascontiguousarray(y.cpu().numpy()), want)


@pytest.mark.parametrize("kappa,envelope", [(0.0, (0.85, 0.55, 0.35, 0.2)), (0.4, (1.0,)), (1.0, (0.9, -0.5)), (1.0, (0.85, 0.55, 0.35, 0.2))])
def test_planar_slab_filter_shapes(api, kappa, envelope):
    """Uniform and log-distributed impulses, identity / negative / default envelopes, and an output
    slab whose base is not 16-byte aligned (no bulk store) on the register-window kernel."""
    import torch

    C, frames = 5, 40000
    vn = api.VelvetNoise(sample_rate_hz=48000, num_outs=C, filtered_channels=(0, 1, 2, 3), mode="LR", normalizer=None,
                         log_distribution_strength=kappa, segment_envelope=envelope, seed=3)
    slab = torch.randn((C, frames), device="cuda") * 0.1
    slab[2, 100:5000] = 0.0  # runs of exact zeros (signed-zero handling of the negated accumulation)
    slab[2, 5000:5100] = -0.0
    # the same slab through a view that starts 4 bytes into a buffer: TMA-ineligible input and output
    buf = torch.empty(C * frames + 1, device="cuda")
    view = buf[1:].view(C, frames)
    view.copy_(slab)
    y = routed(lambda: vn.convolve(slab.t()), {WIN}, "aligned slab")
    y2 = vn.convolve(view.t())
    taps = O.class_taps(sample_rate_hz=48000, num_outs=C, filtered_channels=(0, 1, 2, 3), num_segments=len(envelope),
                        log_distribution_strength=kappa, seed=3)
    want = O.fir_class_order(np.ascontiguousarray(slab.cpu().numpy().T), taps, envelope, C)
    assert G.same_bits(np.ascontiguousarray(y.cpu().numpy()), want)
    assert torch.equal(y2, y)


@pytest.mark.parametrize(
    "frames,kappa,envelope,duration,route",
    [
        # four frames short of the shortest slab the kernel takes (frames stay a multiple of four, so that the channel stride
        # of the slab allows the bulk copies): the window kernel instead
        (-4, 1.0, (0.85, 0.55, 0.35, 0.2), 0.03, {WIN}),
        (0, 1.0, (0.85, 0.55, 0.35, 0.2), 0.03, {TMEM, TILE("float", 0, 256)}),  # the shortest slab it takes: 4 interior tiles
        (4, 1.0, (0.85, 0.55, 0.35, 0.2), 0.03, {TMEM, TILE("float", 0, 256)}),
        (200004, 0.0, (0.85, 0.55, 0.35, 0.2), 0.03, {TMEM, TILE("float", 0, 256)}),  # uniform impulses: most taps far
        (150000, 0.4, (1.0,), 0.03, {TMEM, TILE("float", 0, 256)}),  # identity envelope (no gain multiply), one segment
        (131072 + 9000, 1.0, (0.9, -0.5), 0.03, {TMEM, WIN}),
        (300000, 1.0, (0.85, 0.55, 0.35, 0.2), 0.048, {TMEM, WIN}),  # 2 009-sample halo: the largest it takes
        (300000, 1.0, (0.85, 0.55, 0.35, 0.2), 0.0485, {WIN}),  # 2 030-sample halo: past it
        (180000, 1.0, (0.85, 0.55, 0.35, 0.2), 0.004, {TMEM, WIN}),  # every tap inside the TMEM window
    ],
)
def test_planar_slab_tmem_kernel(api, frames, kappa, envelope, duration, route):
    """Long planar slabs take the tensor-memory kernel for the interior tiles and the window or tile kernel
    for the tail of each channel; the kernels launched are asserted and the whole output must equal the oracle bit for bit."""
    import torch

    C = 5
    filtered = (0, 1, 2, 3)  # channel 4 is copied through
    vn = api.VelvetNoise(sample_rate_hz=48000, duration_seconds=duration, num_impulses=30, num_outs=C, filtered_channels=filtered,
                         mode="LR", normalizer=None, log_distribution_strength=kappa, segment_envelope=envelope, seed=5)
    if frames <= 4:  # relative to the kernel's minimum: (128 + halo blocks) x 96 samples staged per tile + 3 more tiles of 12288
        halo = (vn.tap_program(1 << 20).halo + 3) & ~3
        frames += max(128 + -(-(halo + 4) // 96), 134) * 96 + 3 * 12288
    g = torch.Generator(device="cuda").manual_seed(99)
    slab = torch.randn((C, frames), generator=g, device="cuda") * 0.1
    slab[1, 20000:26000] = 0.0
    slab[1, 26000:26100] = -0.0
    y = routed(lambda: vn.convolve(slab.t()), route, f"{frames} frames")
    taps = O.class_taps(sample_rate_hz=48000, duration_seconds=duration, num_impulses=30, num_outs=C, filtered_channels=filtered,
                        num_segments=len(envelope), log_distribution_strength=kappa, seed=5)
    want = O.fir_class_order(np.ascontiguousarray(slab.cpu().numpy().T), taps, envelope, C)
    got = np.ascontiguousarray(y.cpu().numpy())
    if not G.same_bits(got, want):
        bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
        raise AssertionError(f"{len(bad)} samples differ; first at (frame, channel) {bad[0]}, last {bad[-1]}")


def test_randomised_decorrelate_against_the_oracle(api):
    """120 seeded random (sample rate, duration, impulses, strength, envelope, mode, width, normaliser, filtered channels,
    length, mono / stereo, dtype, seed) combinations of ``VelvetNoise.decorrelate`` (tests/_random_cases.py) on numpy input,
    and on CUDA tensors for the float32 ones: dtype, shape and every bit must equal the oracle's, which
    tests/test_oracle_golden.py pins to the reference's hashes of the same cases; where the reference raises (filters that
    are not sparse), so must the library.  Lengths include 1, 2, 7 and 33 frames (shorter than any filter)."""
    import json
    import os

    import torch

    from tests import _random_cases as RC

    golden = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "random_decorrelate.json")))["cases"]
    errors = {"ValueError": ValueError, "IndexError": IndexError, "TypeError": TypeError}
    for (i, p, x), ref in zip(RC.cases(), golden):
        kw = RC.vn_kwargs(p)
        if "error" in ref:
            with pytest.raises(errors[ref["error"]]):
                api.VelvetNoise(**kw).decorrelate(x)
            continue
        vn = api.VelvetNoise(**kw)
        want = RC.oracle_output(O, p, x)
        got = vn.decorrelate(x)
        assert got.dtype == want.dtype and got.shape == want.shape, (i, p, x.shape, x.dtype)
        if not G.same_bits(np.ascontiguousarray(got), want):
            bad = np.argwhere(np.ascontiguousarray(got).view(np.uint32) != want.view(np.uint32))
            raise AssertionError(f"case {i} {p} input {x.shape} {x.dtype}: {len(bad)} samples differ, first {bad[0]}")
        if x.dtype == np.float32:
            got_t = vn.decorrelate(torch.from_numpy(x).cuda())
            assert G.same_bits(np.ascontiguousarray(got_t.cpu().numpy()), want), (i, p, "tensor path")


@pytest.mark.parametrize("family", ["convolve", "chain", "function"])
def test_more_randomised_families_against_the_oracle(api, family):
    """The three further families of tests/_random_cases.py (60 cases each): multichannel ``convolve`` on C- and
    Fortran-order numpy arrays and on the matching CUDA tensors, ``SignalChain`` velvet noise + Haas, and
    ``convolve_velvet_noise(generate_velvet_noise(...))``.  Bits, dtype and shape equal the oracle's (pinned to the
    reference's hashes on the CPU side); the reference's exceptions are raised where it raises."""
    import json
    import os

    import torch

    from tests import _random_cases as RC

    rows = json.load(open(os.path.join(os.path.dirname(__file__), "golden", "random_decorrelate.json")))["more"][family]
    errors = {"ValueError": ValueError, "IndexError": IndexError, "TypeError": TypeError}
    oracle = {"convolve": RC.oracle_convolve, "chain": RC.oracle_chain, "function": RC.oracle_function}[family]

    def run(p, x):
        if family == "convolve":
            return api.VelvetNoise(**RC.convolve_kwargs(p)).convolve(x)
        if family == "chain":
            return RC.run_chain(api.SignalChain, p, x)
        return api.convolve_velvet_noise(x, api.generate_velvet_noise(**RC.function_kwargs(p)))

    for (i, p, x), ref in zip(RC.more_cases(family), rows):
        if "error" in ref:
            with pytest.raises(errors[ref["error"]]):
                run(p, x)
            continue
        want = oracle(O, p, x)
        got = run(p, x)
        assert got.dtype == want.dtype and got.shape == want.shape, (family, i, p, x.shape, x.dtype)
        if not G.same_bits(np.ascontiguousarray(got), want):
            bad = np.argwhere(np.ascontiguousarray(got).view(np.uint8) != want.view(np.uint8))
            raise AssertionError(f"{family} case {i} {p} input {x.shape} {x.dtype}: bytes differ, first at {bad[0]}")
        if family == "convolve" and x.dtype == np.float32:  # the same view of the data as a CUDA tensor
            xt = torch.from_numpy(np.ascontiguousarray(x.T)).cuda().t() if x.flags.f_contiguous and not x.flags.c_contiguous \
                else torch.from_numpy(np.ascontiguousarray(x)).cuda()
            got_t = run(p, xt)
            assert G.same_bits(np.ascontiguousarray(got_t.cpu().numpy()), want), (family, i, p, "tensor path")


def test_many_channels_every_sample(api):
    """600 channels x 65 000 frames (more runs than four waves of persistent CTAs, one tap table sliced over all of them):
    EVERY output sample of every channel against the oracle, not just windows of the first and the last channel as in
    bench.py's spot check."""
    import torch

    Cn, frames = 600, 65000
    vn = api.VelvetNoise(sample_rate_hz=48000, duration_seconds=0.03, num_impulses=30, num_outs=Cn, filtered_channels=tuple(range(Cn)), mode="LR",
                         normalizer=None, seed=3)
    g = torch.Generator(device="cuda").manual_seed(123)
    slab = torch.randn((Cn, frames), generator=g, device="cuda") * 0.1
    y = vn.convolve(slab.t())
    taps = O.class_taps(sample_rate_hz=48000, duration_seconds=0.03, num_impulses=30, num_outs=Cn, filtered_channels=tuple(range(Cn)), seed=3)
    want = O.fir_class_order(np.ascontiguousarray(slab.cpu().numpy().T), taps, O.DEFAULT_ENVELOPE, Cn)
    got = np.ascontiguousarray(y.cpu().numpy())
    if not G.same_bits(got, want):
        bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
        raise AssertionError(f"{len(bad)} samples differ; first at (frame, channel) {bad[0]}, channels {np.unique(bad[:, 1])[:10]}")


def test_planar_slab_unaligned_falls_back(api):
    """A channel stride that is not a multiple of 4 samples cannot use the bulk copy."""
    import torch

    C, frames = 3, 10001
    vn = api.VelvetNoise(sample_rate_hz=48000, num_outs=C, filtered_channels=tuple(range(C)), mode="LR", normalizer=None, seed=2)
    slab = torch.randn((C, frames), device="cuda") * 0.1
    y = vn.convolve(slab.t())
    taps = O.class_taps(sample_rate_hz=48000, num_outs=C, filtered_channels=tuple(range(C)), seed=2)
    want = O.fir_class_order(np.ascontiguousarray(slab.cpu().numpy().T), taps, O.DEFAULT_ENVELOPE, C)
    assert G.same_bits(np.ascontiguousarray(y.cpu().numpy()), want)


def test_wide_interleaved_numpy_slab(api):
    """(frames, 64) C-order numpy input: transposed on the device around the planar kernel."""
    rng = np.random.default_rng(8)
    C, frames = 64, 20011
    x = (rng.standard_normal((frames, C)) * 0.1).astype(np.float32)
    vn = api.VelvetNoise(sample_rate_hz=48000, num_outs=C, filtered_channels=tuple(range(C)), mode="LR", normalizer=None, seed=1)
    taps = O.class_taps(sample_rate_hz=48000, num_outs=C, filtered_channels=tuple(range(C)), seed=1)
    assert G.same_bits(vn.convolve(x), O.fir_class_order(x, taps, O.DEFAULT_ENVELOPE, C))
    # LR decorrelate with the RMS normaliser on more than two channels (unfused composition)
    vn4 = api.VelvetNoise(sample_rate_hz=48000, num_outs=4, filtered_channels=(0, 1, 2, 3), mode="LR", seed=1)
    t4 = O.class_taps(sample_rate_hz=48000, num_outs=4, filtered_channels=(0, 1, 2, 3), seed=1)
    x4 = np.ascontiguousarray(x[:, :4])
    assert G.same_bits(vn4.decorrelate(x4), O.vn_decorrelate(x4, t4, num_outs=4, ms_mode=False))


def test_cfg4_long_filter_large_halo(api):
    """300 impulses over 0.3 s at 96 kHz: a 28 800-sample halo, one CTA per SM."""
    import torch

    C, frames = 4, 150001
    vn = api.VelvetNoise(sample_rate_hz=96000, duration_seconds=0.3, num_impulses=300, num_outs=C, filtered_channels=(0, 1, 2, 3),
                         mode="LR", normalizer=None, seed=1)
    assert G.sha(vn.velvet_noise.rows()) == G.hashes()["tables"]["cfg4_4ch"]["sha256"]
    slab = torch.randn((C, frames), device="cuda") * 0.1
    y = vn.convolve(slab.t())
    taps = O.class_taps(sample_rate_hz=96000, duration_seconds=0.3, num_impulses=300, num_outs=C, filtered_channels=(0, 1, 2, 3), seed=1)
    want = O.fir_class_order(np.ascontiguousarray(slab.cpu().numpy().T), taps, O.DEFAULT_ENVELOPE, C)
    assert G.same_bits(np.ascontiguousarray(y.cpu().numpy()), want)


_RING_TAIL = {RING, TILE("float", 0, 1024)}
_ENV5 = (0.9, -0.5, 0.25, 0.3, 0.1)


@pytest.mark.parametrize(
    "fs,duration,n_imp,envelope,frames,filtered,route",
    [
        # BASELINE config 4's filter (28 420-sample halo), several runs per channel, channel 3 copied
        (96000, 0.3, 300, (0.85, 0.55, 0.35, 0.2), 700004, (0, 1, 2), _RING_TAIL),
        (96000, 0.35, 120, (1.0,), 400000, (0, 1, 2, 3), _RING_TAIL),        # identity envelope (no gain multiply), 32 534-sample halo
        (96000, 0.36, 100, (0.9, -0.5, 0.25), 9216 * 30, (0, 1), _RING_TAIL),  # three segments (one single-stream pass), whole steps
        (96000, 0.34, 100, _ENV5, 125776, (0, 1, 2, 3), _RING_TAIL),          # five segments; the shortest slab it takes: 4 x halo
        (96000, 0.34, 100, _ENV5, 125772, (0, 1, 2, 3), {TILE("float", 0, 1024)}),  # four frames short of it: the tile kernel only
    ],
)
def test_ring_kernel_long_filters(api, fs, duration, n_imp, envelope, frames, filtered, route):
    """Long filters on long planar slabs: the interior of every channel goes through the ring-buffer kernel
    (vnd_fir_ring.cu: persistent CTAs, every sample fetched once), the tail through the tile kernels; the kernels launched
    are asserted and every output sample must equal the oracle's.  Frames are multiples of four, so that the channel
    stride of the slab allows the bulk copies."""
    import torch

    Cn = 4
    vn = api.VelvetNoise(sample_rate_hz=fs, duration_seconds=duration, num_impulses=n_imp, num_outs=Cn, filtered_channels=filtered, mode="LR",
                         normalizer=None, segment_envelope=envelope, seed=9)
    g = torch.Generator(device="cuda").manual_seed(31)
    slab = torch.randn((Cn, frames), generator=g, device="cuda") * 0.1
    slab[0, 1000:9000] = 0.0
    slab[0, 9000:9100] = -0.0
    y = routed(lambda: vn.convolve(slab.t()), route, f"{frames} frames")
    taps = O.class_taps(sample_rate_hz=fs, duration_seconds=duration, num_impulses=n_imp, num_outs=Cn, num_segments=len(envelope),
                        filtered_channels=filtered, seed=9)
    want = O.fir_class_order(np.ascontiguousarray(slab.cpu().numpy().T), taps, envelope, Cn)
    got = np.ascontiguousarray(y.cpu().numpy())
    if not G.same_bits(got, want):
        bad = np.argwhere(got.view(np.uint32) != want.view(np.uint32))
        raise AssertionError(f"{len(bad)} samples differ; first at (frame, channel) {bad[0]}, last {bad[-1]}")


def test_filter_longer_than_shared_memory_uses_direct_kernel(api):
    rng = np.random.default_rng(4)
    x = (rng.standard_normal((300000, 2)) * 0.1).astype(np.float32)
    vn = api.VelvetNoise(sample_rate_hz=96000, duration_seconds=2.5, num_impulses=40, seed=3)  # 240 000-sample halo
    taps = O.class_taps(sample_rate_hz=96000, duration_seconds=2.5, num_impulses=40, seed=3)
    y = routed(lambda: vn.convolve(x), {DIRECT("float", 0)})
    assert G.same_bits(y, O.fir_class_order(x, taps, O.DEFAULT_ENVELOPE, 2))
    assert G.same_bits(vn.decorrelate(x), O.vn_decorrelate(x, taps))


def test_size_independent_properties_full_slab(api):
    """Properties that hold bit-exactly at any size: scaling by a power of two commutes with the
    FIR, and a time shift of the input shifts the output (away from the end)."""
    import torch

    C, frames = 16, 4_000_000
    vn = api.VelvetNoise(sample_rate_hz=48000, num_outs=C, filtered_channels=tuple(range(C)), mode="LR", normalizer=None, seed=1)
    slab = torch.randn((C, frames), device="cuda") * 0.1
    y = vn.convolve(slab.t())
    y2 = vn.convolve((slab * 2.0).t())
    assert torch.equal(y2, y * 2.0)
    k = 4096 + 12
    ys = vn.convolve(slab[:, k:].t())
    halo = vn.tap_program(frames).halo
    assert torch.equal(ys[: frames - k - halo], y[k : frames - halo])
    # sub-slab against the oracle: first and last 2^17 samples of two channels
    n = 1 << 17
    taps = O.class_taps(sample_rate_hz=48000, num_outs=C, filtered_channels=tuple(range(C)), seed=1)
    for ch in (0, C - 1):
        col = slab[ch].cpu().numpy()
        sub_taps = [[] if i != ch else taps[ch] for i in range(C)]
        head = O.fir_class_order(np.repeat(col[: n + halo, None], C, axis=1), sub_taps, O.DEFAULT_ENVELOPE, C)[:n, ch]
        assert np.array_equal(head, y[:n, ch].cpu().numpy())
        tail = O.fir_class_order(np.repeat(col[-n:, None], C, axis=1), sub_taps, O.DEFAULT_ENVELOPE, C)[:, ch]
        assert np.array_equal(tail, y[-n:, ch].cpu().numpy())


def test_streaming_host_path(api):
    """vnd_sparse_fir_stream_host (pinned and pageable) equals the one-shot planar call."""
    import ctypes as C_

    from vndecorrelate_b200 import _native as N
    from vndecorrelate_b200 import runtime as R

    C, frames = 12, 200003
    vn = api.VelvetNoise(sample_rate_hz=48000, num_outs=C, filtered_channels=tuple(range(C)), mode="LR", normalizer=None, seed=1)
    prog = vn.tap_program(frames)
    rng = np.random.default_rng(2)
    x = (rng.standard_normal((C, frames)) * 0.1).astype(np.float32)
    want = np.ascontiguousarray(vn.convolve(x.T).T)
    ctx = R.HostContext.get()
    for pinned in (False, True):
        if pinned:
            px, py = R.PinnedArray((C, frames)), R.PinnedArray((C, frames))
            px.array[...] = x
            xin, yout = px.array, py.array
        else:
            xin, yout = x, np.empty_like(x)
        ps = prog.host_struct()
        N.check(N.lib().vnd_sparse_fir_stream_host(ctx.handle, xin.ctypes.data, yout.ctypes.data, frames, C, C_.byref(ps), 5), "stream")
        assert G.same_bits(np.array(yout), want)


@pytest.mark.parametrize("layout", ["interleaved", "planar", "stereo", "extra_channels"])
@pytest.mark.parametrize("pinned", [False, True])
def test_overlapped_host_path_equals_one_shot(api, monkeypatch, layout, pinned):
    """numpy slabs of 8 MB and more go through the overlapped pipeline of vnd_sparse_fir_host (chunks of frames with
    the filter's halo for C-order input, channel groups for planar input; pageable buffers staged by helper threads,
    page-locked ones copied by DMA): same bytes as the one-shot path (VND_NO_PIPELINE) and as the oracle."""
    from vndecorrelate_b200 import runtime as R

    rng = np.random.default_rng(11)
    if layout == "stereo":
        C, Cin, frames = 2, 2, 1_500_003
    elif layout == "extra_channels":
        C, Cin, frames = 2, 3, 1_000_001
    else:
        C, Cin, frames = 12, 12, 300_007
    vn = api.VelvetNoise(sample_rate_hz=48000, num_outs=C, filtered_channels=tuple(range(C)), mode="LR", normalizer=None, seed=1)
    shape = (Cin, frames) if layout == "planar" else (frames, Cin)
    data = (rng.standard_normal(shape) * 0.1).astype(np.float32)
    if pinned:
        holder = R.PinnedArray(shape)
        holder.array[...] = data
        data = holder.array
    x = data.T if layout == "planar" else data
    monkeypatch.setenv("VND_NO_PIPELINE", "1")
    want = np.array(vn.convolve(x))
    monkeypatch.delenv("VND_NO_PIPELINE")
    for chunk_mb in ("1", "3", "64"):  # many small stages, odd stage sizes, the default
        monkeypatch.setenv("VND_PIPE_CHUNK_MB", chunk_mb)
        got = vn.convolve(x)
        assert got.shape == (frames, C) and got.dtype == np.float32
        assert G.same_bits(np.ascontiguousarray(got), np.ascontiguousarray(want)), (layout, pinned, chunk_mb)
    n = 20000  # and against the oracle at both ends of the slab
    taps = O.class_taps(sample_rate_hz=48000, num_outs=C, filtered_channels=tuple(range(C)), seed=1)
    head = O.fir_class_order(np.ascontiguousarray(x[: n + 2000, :C]), taps, O.DEFAULT_ENVELOPE, C)[:n]
    tail = O.fir_class_order(np.ascontiguousarray(x[-n:, :C]), taps, O.DEFAULT_ENVELOPE, C)
    assert G.same_bits(np.ascontiguousarray(want[:n]), head) and G.same_bits(np.ascontiguousarray(want[-n + 2000:]), tail[2000:])


# ------------------------------------------------------------------ objective and sweeps


def test_objective_known_answers_viola(api):
    from vndecorrelate_b200.optimization import symmetry_aware_objective

    fs, x = G.wav("viola")
    okw = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)
    for row in G.objective()["viola_vn"]:
        d = api.VelvetNoise(sample_rate_hz=fs, duration_seconds=0.03, num_impulses=30, log_distribution_strength=row["kappa"],
                            normalizer=None, filtered_channels=(0,), mode="LR", seed=1)
        got = symmetry_aware_objective(x, d, **okw)
        assert isinstance(got, np.float32)
        # float32 scores near 619 have an ulp of 6.1e-5; the reference's own value moves by up to
        # ~2e-4 with the last ulp of numpy's float32 arctan2 (SURVEY.md H5)
        assert abs(float(got) - row["objective"]) <= 5e-4, (row["kappa"], float(got), row["objective"])
    for row in G.objective()["viola_haas"]:
        got = symmetry_aware_objective(x, api.HaasEffect(sample_rate_hz=fs, delay_time_seconds=row["tau"], mode="LR"), **okw)
        assert isinstance(got, np.float64)
        assert abs(float(got) - row["objective"]) <= 1e-9 * max(1.0, abs(row["objective"]))


def test_objective_partials_against_reference_terms(api):
    """The kernel's sums against the reference's own intermediate values on viola."""
    from vndecorrelate_b200.optimization import _max_abs_theta_f32, vn_objective_partials
    from vndecorrelate_b200.taps import candidate_program

    fs, x = G.wav("viola")
    rows = G.objective()["viola_vn"]
    ds = [api.VelvetNoise(sample_rate_hz=fs, duration_seconds=0.03, num_impulses=30, log_distribution_strength=r["kappa"],
                          normalizer=None, filtered_channels=(0,), mode="LR", seed=1) for r in rows]
    prog = candidate_program([d.velvet_noise for d in ds], ds[0].segment_envelope, x.shape[0])
    p = vn_objective_partials(x, prog)[0]
    for r, q in zip(rows, p):
        assert abs(q[0] - r["sum_r"]) <= 2e-6 * r["sum_r"]  # the reference's value is a float32 pairwise sum
        assert abs(q[2] / q[0] - r["spread"]) <= 2e-6
        assert abs(q[1] / q[0] - r["centroid"]) <= 2e-6
        assert abs(q[3] / q[0] - r["m3"]) <= 2e-6
        assert abs(q[4] - r["dot_lr"]) <= 1e-5 * max(1.0, abs(r["dot_lr"]))
        assert abs(np.sqrt(q[5]) - r["norm_l"]) <= 1e-5 * r["norm_l"]
        assert float(_max_abs_theta_f32(q)) == pytest.approx(r["max_abs_theta"], abs=1.2e-7)  # one float32 ulp at pi/2
        assert q[10] == x.shape[0]


def _assert_minima_agree(got, want, ref_scores, noise=1e-3, allowed=None):
    """Local-minima sets must be equal except at indices where the reference's score differs from a grid neighbour by
    less than `noise` (there the strict comparison of optimization.py:123-124 is decided by evaluation noise).
    Returns the symmetric difference."""
    sym = sorted(set(got) ^ set(want))
    n = len(ref_scores)
    for i in sym:
        gaps = [abs(ref_scores[j] - ref_scores[j + 1]) for j in range(max(0, i - 2), min(n - 1, i + 2))]  # a flip moves a minimum to a neighbour
        assert min(gaps) <= noise, (i, sym, [float(ref_scores[j]) for j in range(max(0, i - 2), min(n, i + 3))])
    if allowed is not None:
        assert len(sym) <= allowed, sym
    return sym


def test_small_sweeps(api):
    from vndecorrelate_b200.optimization import get_local_minima, grid_scan

    fs, viola = G.wav("viola")
    sw = G.objective()["sweeps"]
    okw = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)
    sigs = {"viola_60k": viola[40000:100000], "clip0_48k": O.coloured_clip(0, 48000), "clip1_96k": O.coloured_clip(1, 96000)}
    for name, sig in sigs.items():
        s = sw[name]
        ds = [api.VelvetNoise(sample_rate_hz=s["fs"], duration_seconds=0.03, num_impulses=30, log_distribution_strength=k,
                              normalizer=None, filtered_channels=(0,), mode="LR", seed=1) for k in np.linspace(0.0, 1.0, 32)]
        sc = grid_scan(sig, ds, **okw)
        assert sc.dtype == np.float32
        assert np.max(np.abs(sc.astype(np.float64) - np.array(s["vn_scores"]))) <= 5e-4
        assert int(np.argmin(sc)) == s["vn_argmin"]  # the selected grid point must match exactly
        # get_local_minima compares neighbours with a strict '<': where the reference's own neighbouring scores are
        # closer than the float32 evaluation noise (SURVEY.md H5) a minimum may flip; anywhere else the sets must agree
        _assert_minima_agree(get_local_minima(sc, 32), s["vn_minima"], np.array(s["vn_scores"]))
        hs = [api.HaasEffect(sample_rate_hz=s["fs"], delay_time_seconds=t, mode="LR") for t in np.linspace(0.0, 0.03, 32)]
        sh = grid_scan(sig, hs, **okw)
        assert sh.dtype == np.float64
        assert np.allclose(sh, np.array(s["haas_scores"]), rtol=1e-9, atol=1e-9)
        assert int(np.argmin(sh)) == s["haas_argmin"]
        assert get_local_minima(sh, 32) == s["haas_minima"]


def test_optimisers_short_excerpt(api):
    from vndecorrelate_b200.optimization import optimize_haas_delay, optimize_velvet_noise

    fs, viola = G.wav("viola")
    sig = viola[40000:80000]
    ref = G.objective()["optimize_haas_viola_40k"]
    tau = optimize_haas_delay(input_signal=sig, sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=ref["grid_size"])
    assert abs(tau - ref["tau"]) <= 1e-4  # Brent's xatol (optimization.py:148)
    ref = G.objective()["optimize_vn_viola_40k"]
    k = optimize_velvet_noise(input_signal=sig, sample_rate_hz=fs, duration_seconds=0.03, num_impulses=ref["num_impulses"], seed=1,
                              grid_size=ref["grid_size"])
    # the objective is piecewise constant in kappa (tap indices are rounded): the refined value is
    # only defined up to the plateau, so compare the resulting tap table and the distance
    a = api.VelvetNoise(sample_rate_hz=fs, num_impulses=ref["num_impulses"], log_distribution_strength=k, filtered_channels=(0,), mode="LR", seed=1)
    b = api.VelvetNoise(sample_rate_hz=fs, num_impulses=ref["num_impulses"], log_distribution_strength=ref["kappa"], filtered_channels=(0,), mode="LR", seed=1)
    assert abs(k - ref["kappa"]) <= 1e-4 or a.velvet_noise == b.velvet_noise  # Brent's xatol (optimization.py:148)


def test_cfg5_full_shape_one_clip(api):
    """BASELINE config 5 at its real shape for one clip: 1024 strengths x 30 s @ 48 kHz, grid stage AND refinement,
    against what the UNMODIFIED reference computed for the same clip (tests/golden/cfg5_clip0.json, generated by
    tests/golden/make_golden_r02.py): every score within 5e-4 (float32 evaluation noise at magnitude 619, SURVEY.md
    H5), the argmin identical, the refined strength within Brent's xatol, and the symmetric difference of the
    local-minima sets counted (strict '<' between neighbours closer than the evaluation noise may flip)."""
    import json
    import os

    from vndecorrelate_b200 import optimization as OPT

    ref = json.load(open(os.path.join(G.GOLDEN, "cfg5_clip0.json")))
    clip = O.coloured_clip(ref["clip_index"], ref["frames"])
    assert G.sha(clip) == ref["input_sha256"]
    kw = dict(sample_rate_hz=ref["fs"], duration_seconds=ref["duration_seconds"], num_impulses=ref["num_impulses"], seed=1, grid_size=ref["grid_size"])
    kappa, info = OPT.optimize_velvet_noise_batch(input_signals=[clip], details=True, **kw)
    scores = info["scores"][0]
    want = np.array(ref["scores"], dtype=np.float64)
    err = float(np.max(np.abs(scores.astype(np.float64) - want)))
    assert scores.dtype == np.float32 and err <= 5e-4, err
    assert info["argmin"][0] == ref["argmin"]
    # the order of the best candidates is preserved wherever the reference separates them by more than the noise
    top = np.argsort(want, kind="stable")[:16]
    for a, b in zip(top[:-1], top[1:]):
        if want[b] - want[a] > 1e-3:
            assert scores[a] < scores[b], (a, b)
    got_min, ref_min = set(info["local_minima"][0]), set(ref["local_minima"])
    _assert_minima_agree(got_min, ref_min, want, allowed=8)  # of ~312 minima; each flip is a neighbour gap below the evaluation noise
    assert abs(float(kappa[0]) - ref["kappa"]) <= 1e-4, (float(kappa[0]), ref["kappa"])
    single = OPT.optimize_velvet_noise(input_signal=clip, **kw)  # the one-clip entry point is the same computation
    assert float(single) == float(kappa[0])


def test_empty_clip_is_an_error_not_a_crash(api):
    """An empty signal has no max|theta|: the reference raises numpy's ValueError; the C ABI answers VND_EINVAL (it used to
    divide by zero while planning the launch)."""
    import ctypes as C_

    from vndecorrelate_b200 import _native as N
    from vndecorrelate_b200 import optimization as OPT
    from vndecorrelate_b200 import runtime as R
    from vndecorrelate_b200 import taps as T

    cands = [api.VelvetNoise(sample_rate_hz=48000, log_distribution_strength=k, normalizer=None, filtered_channels=(0,), mode="LR", seed=1) for k in (0.0, 1.0)]
    with pytest.raises(ValueError):
        OPT.grid_scan(np.zeros((0, 2), dtype=np.float32), cands, angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0,
                      lambda_penalty=1e3)
    prog = T.candidate_program([c.velvet_noise for c in cands], cands[0].segment_envelope, 100)
    out = np.zeros((1, 2, N.OBJ_SLOTS))
    dummy = np.zeros(4, dtype=np.float32)
    ps = prog.host_struct()
    rc = N.lib().vnd_vn_objective_batch_host(R.HostContext.get().handle, dummy.ctypes.data, 0, 1, 0, 0, C_.byref(ps), out.ctypes.data)
    assert rc == N.VND_EINVAL and b"empty" in N.lib().vnd_last_error()
    # the objective kernel reads SEGMENTED headers: the host call rejects any other order before a copy, as the _dev call does
    clip = np.zeros((1, 2, 64), dtype=np.float32)
    ps.order = N.ORDER_ASCENDING
    rc = N.lib().vnd_vn_objective_batch_host(R.HostContext.get().handle, clip.ctypes.data, 64, 1, 128, 64, C_.byref(ps), out.ctypes.data)
    assert rc == N.VND_EINVAL and b"SEGMENTED" in N.lib().vnd_last_error()


def test_host_calls_reject_what_their_dev_calls_reject(api):
    """A _host call runs the checks of its _dev twin before any copy, also where its own path would not reach them."""
    import ctypes as C_

    from vndecorrelate_b200 import _native as N
    from vndecorrelate_b200 import runtime as R

    lib, ctx = N.lib(), R.HostContext.get().handle
    # a float64 y of a wide frame-interleaved slab: the host path runs the kernel on float32 planar copies
    vn = api.VelvetNoise(sample_rate_hz=48000, num_outs=4, filtered_channels=(0, 1, 2, 3), mode="LR", normalizer=None, seed=1)
    prog = vn.tap_program(256)
    ps = prog.host_struct()
    x, y = np.zeros((256, 4), np.float32), np.zeros((256, 4), np.float64)
    xs, ys = N.SignalStruct(x.ctypes.data, 256, 4, N.VND_F32, 4, 1), N.SignalStruct(y.ctypes.data, 256, 4, N.VND_F64, 4, 1)
    assert lib.vnd_sparse_fir_host(ctx, C_.byref(xs), C_.byref(ys), C_.byref(ps)) == N.VND_EINVAL
    assert b"y must be float32" in lib.vnd_last_error()
    # an unknown clip dtype, also with nothing to score
    assert lib.vnd_haas_objective_batch_host(ctx, None, 7, 0, 0, 0, 0, None, 0, None) == N.VND_EINVAL
    assert b"unknown clip dtype" in lib.vnd_last_error()


def test_batch_optimiser_equals_clip_by_clip(api):
    """optimize_velvet_noise_batch on several clips returns, per clip, exactly what optimize_velvet_noise returns."""
    from vndecorrelate_b200 import optimization as OPT

    clips = [O.coloured_clip(i, 30000 + 0 * i) for i in range(5)]
    kw = dict(sample_rate_hz=48000, duration_seconds=0.03, num_impulses=30, seed=1, grid_size=64)
    both, info = OPT.optimize_velvet_noise_batch(input_signals=clips, details=True, **kw)
    one = [float(OPT.optimize_velvet_noise(input_signal=c, **kw)) for c in clips]
    assert [float(k) for k in both] == one
    planar = np.stack([c.T for c in clips])
    again = OPT.optimize_velvet_noise_batch(input_signals=planar, **kw)  # planar (n, 2, frames) input
    assert np.array_equal(again, both)
    ref_scores = np.stack([O.vn_grid_scores(c, np.linspace(0, 1, 64), sample_rate_hz=48000, duration_seconds=0.03, num_impulses=30, seed=1) for c in clips])
    assert np.max(np.abs(info["scores"].astype(np.float64) - ref_scores.astype(np.float64))) <= 5e-4
    assert info["argmin"] == [int(np.argmin(r)) for r in ref_scores]


def test_batched_refinement_equals_one_at_a_time(api):
    """Lock-step Brent (one launch per iteration over all local minima) returns exactly what the
    reference's loop over minima returns with the same objective (optimization.py:131-155)."""
    from vndecorrelate_b200 import optimization as OPT

    fs, viola = G.wav("viola")
    sig = viola[60000:90000]
    kw = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)

    def candidate(kappa):
        return api.VelvetNoise(sample_rate_hz=fs, duration_seconds=0.03, num_impulses=15, log_distribution_strength=kappa, normalizer=None,
                               filtered_channels=(0,), mode="LR", seed=1)

    grid = 48
    kappas = np.linspace(0.0, 1.0, grid)
    scores = OPT.grid_scan(sig, [candidate(k) for k in kappas], **kw)
    minima = OPT.get_local_minima(scores, grid)
    one_at_a_time = OPT.optimize_local_minima(minima, kappas, grid, lambda k: OPT.symmetry_aware_objective(sig, candidate(k), **kw))
    batched = OPT.optimize_velvet_noise(input_signal=sig, sample_rate_hz=fs, duration_seconds=0.03, num_impulses=15, seed=1, grid_size=grid)
    assert batched == one_at_a_time

    taus = np.linspace(0.0, 0.03, grid)
    scores = OPT.grid_scan(sig, [api.HaasEffect(sample_rate_hz=fs, delay_time_seconds=t, mode="LR") for t in taus], **kw)
    minima = OPT.get_local_minima(scores, grid)
    one_at_a_time = OPT.optimize_local_minima(
        minima, taus, grid, lambda t: OPT.symmetry_aware_objective(sig, api.HaasEffect(sample_rate_hz=fs, delay_time_seconds=t, mode="LR"), **kw))
    batched = OPT.optimize_haas_delay(input_signal=sig, sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=grid)
    assert batched == one_at_a_time


# ------------------------------------------------------------------ numpy-order sum of squares (rms_normalize, utils/dsp.py:107-109)
def _colsumsq(t):
    """vnd_colsumsq_seq_f32_dev on a (frames, channels) CUDA tensor -> float32 sums per column."""
    import ctypes as C

    import torch

    from vndecorrelate_b200 import _native as N
    from vndecorrelate_b200 import runtime as R

    sig = R.torch_signal(t)
    out = torch.empty(t.shape[1], dtype=torch.float32, device=t.device)
    rc = N.lib().vnd_colsumsq_seq_f32_dev(C.byref(sig), C.c_void_p(out.data_ptr()), C.c_void_p(R.torch_stream_ptr(t)))
    assert rc == 0, N.lib().vnd_last_error()
    torch.cuda.synchronize()
    return out.cpu().numpy()


def _seq_columns(rng, kind, frames):
    if kind == "audio":  # what rms_normalize sees
        return (rng.standard_normal((frames, 3)) * 0.2).astype(np.float32)
    if kind == "range":  # 30 decades of dynamic range: many binade changes, addends far below one ulp of the sum
        return (rng.standard_normal((frames, 3)) * 10.0 ** rng.uniform(-15, 4, (frames, 3))).astype(np.float32)
    if kind == "ties":  # squares that are small multiples of a power of two: exact ties against the running sum's ulp
        k = rng.integers(0, 64, (frames, 3)).astype(np.float32)
        x = np.sqrt(k * np.float32(2.0 ** -20)).astype(np.float32)
        x[rng.random((frames, 3)) < 0.3] = np.float32(2.0 ** -13)  # square 2^-26: half an ulp once the sum passes 2^-2
        x[0, :] = np.float32(0.5)
        return x
    if kind == "silence":  # zeros, then subnormal squares, then signal
        x = np.zeros((frames, 3), dtype=np.float32)
        x[frames // 3: frames // 2] = np.float32(1e-21) * rng.standard_normal((frames // 2 - frames // 3, 3)).astype(np.float32)
        x[frames // 2:] = (rng.standard_normal((frames - frames // 2, 3)) * 1e-3).astype(np.float32)
        return x
    if kind == "huge":  # overflow to inf on the way
        x = (rng.standard_normal((frames, 3)) * 1e17).astype(np.float32)
        x[:, 1] *= np.float32(100.0)
        return x
    if kind == "nan":
        x = (rng.standard_normal((frames, 3)) * 0.1).astype(np.float32)
        x[frames // 2, 0] = np.nan
        x[frames // 3, 1] = np.inf
        return x
    raise AssertionError(kind)


@pytest.mark.parametrize("kind", ["audio", "range", "ties", "silence", "huge", "nan"])
@pytest.mark.parametrize("frames", [4095, 4096, 8191, 8192, 8193, 100003, 407077])
def test_sequential_sum_of_squares_is_numpy_order(kind, frames):
    """The parallel evaluation (transducer scan per binade, vnd_post.cu) returns the strict left-to-right
    float32 running sum bit for bit, like the scalar chain it replaces for long signals."""
    import torch

    rng = np.random.default_rng(frames * 7 + len(kind))
    x = _seq_columns(rng, kind, frames)
    with np.errstate(over="ignore", invalid="ignore"):
        want = np.array([O.seq_sumsq_f32(x[:, c]) for c in range(x.shape[1])], dtype=np.float32)
    got = _colsumsq(torch.from_numpy(x).cuda())
    assert got.dtype == np.float32
    # NaN results compare as NaN (the payload of an arithmetic NaN is the hardware's), everything else bit for bit
    same = (lambda a, b: np.array_equal(a, b, equal_nan=True)) if kind == "nan" else G.same_bits
    assert same(got, want), (kind, frames, got, want)
    # a strided view (every second column of a wider slab) reads the same values
    wide = torch.from_numpy(np.repeat(x, 2, axis=1)).cuda()
    assert same(_colsumsq(wide[:, ::2]), want)


@pytest.mark.parametrize("kind", ["audio", "range", "ties"])
def test_sequential_sum_of_squares_many_columns(kind):
    """With many columns the scan runs on one CTA per column (the cluster of CTAs per column is for few columns,
    where SMs would idle): same bits."""
    import torch

    frames = 100003
    rng = np.random.default_rng(11 + len(kind))
    x = np.concatenate([_seq_columns(rng, kind, frames) for _ in range(14)], axis=1)  # 42 columns
    want = np.array([O.seq_sumsq_f32(x[:, c]) for c in range(x.shape[1])], dtype=np.float32)
    got = _colsumsq(torch.from_numpy(x).cuda())
    assert G.same_bits(got, want)


def test_sequential_sum_of_squares_full_length():
    """BASELINE config 3's channel length (10 min @ 48 kHz = 28.8 M frames): about 3 500 scan rounds per column on
    the cluster path, the sum crossing 20 binades; still numpy's left-to-right float32 sum bit for bit."""
    import torch

    frames = 28_800_000
    rng = np.random.default_rng(2024)
    x = (rng.standard_normal((frames, 2)) * 0.1).astype(np.float32)
    x[:, 1] *= np.float32(30.0)
    want = np.array([O.seq_sumsq_f32(x[:, c]) for c in range(2)], dtype=np.float32)
    got = _colsumsq(torch.from_numpy(x).cuda())
    assert G.same_bits(got, want), (got, want)
