"""decorrelate_batch: many clips in one call, each byte-identical to the single-clip API on that clip.

The CPU tests check argument handling, the packed layout checks and program deduplication without a device.  The GPU
tests compare every clip's dtype, shape and bytes with ``decorrelator(clip)`` - itself pinned to the reference's
fixtures and the oracle - plus the committed hashes and one direct oracle comparison.
"""

from __future__ import annotations

import ctypes as C

import numpy as np
import pytest

from tests import _golden as G
from vndecorrelate_b200 import _native as N
from vndecorrelate_b200 import decorrelation as D
from vndecorrelate_b200.utils.dsp import rms_normalize

gpu = pytest.mark.gpu
FS = 44100


def _vn(**kw):
    base = dict(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, seed=1)
    base.update(kw)
    return D.VelvetNoise(**base)


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


# ------------------------------------------------------------------ CPU: argument handling


def test_mixed_settings_raise_value_error_naming_the_setting():
    clips = _clips([100, 200])
    with pytest.raises(ValueError, match="width"):
        D.decorrelate_batch(clips, [_vn(width=None), _vn(width=0.3)])
    with pytest.raises(ValueError, match="mode"):
        D.decorrelate_batch(clips, [_vn(mode="MS"), _vn(mode="LR")])
    with pytest.raises(ValueError, match="normalizer"):
        D.decorrelate_batch(clips, [_vn(), _vn(normalizer=None)])
    with pytest.raises(ValueError, match="identity segment_envelope"):
        D.decorrelate_batch(clips, [_vn(segment_envelope=(1.0,)), _vn()])
    chain = lambda d: D.SignalChain(sample_rate_hz=FS).velvet_noise(seed=1).haas_effect(delay_time_seconds=d, mode="LR")  # noqa: E731
    with pytest.raises(ValueError, match="Haas delay"):
        D.decorrelate_batch(clips, [chain(0.02), chain(0.01)])
    with pytest.raises(ValueError, match="Haas stage"):
        D.decorrelate_batch(clips, [chain(0.02), _vn()])


def test_num_outs_other_than_two_is_rejected():
    vn = _vn(num_outs=3, mode="LR", filtered_channels=(0, 1, 2), normalizer=None)
    with pytest.raises(ValueError, match="num_outs"):
        D.decorrelate_batch(_clips([100]), vn)


def test_user_normaliser_and_unsupported_stages_are_not_implemented():
    with pytest.raises(NotImplementedError, match="normaliser"):
        D.decorrelate_batch(_clips([100]), _vn(normalizer=lambda x, y: None))
    haas_only = D.SignalChain(sample_rate_hz=FS).haas_effect(delay_time_seconds=0.02, mode="LR")
    with pytest.raises(NotImplementedError, match="HaasEffect"):
        D.decorrelate_batch(_clips([100]), haas_only)
    ms_haas = D.SignalChain(sample_rate_hz=FS).velvet_noise(seed=1).haas_effect(delay_time_seconds=0.02, mode="MS")
    with pytest.raises(NotImplementedError):
        D.decorrelate_batch(_clips([100]), ms_haas)
    with pytest.raises(NotImplementedError):
        D.decorrelate_batch(_clips([100]), D.HaasEffect(sample_rate_hz=FS))


def test_decorrelator_list_must_match_the_clips():
    with pytest.raises(ValueError, match="2 decorrelators for 3 clips"):
        D.decorrelate_batch(_clips([10, 20, 30]), [_vn(), _vn()])


def test_empty_batch_returns_empty_result():
    assert D.decorrelate_batch([], _vn()) == []
    out = D.decorrelate_batch(np.zeros((0, 50, 2), np.float32), D.SignalChain(sample_rate_hz=FS).velvet_noise(seed=1).haas_effect(mode="LR"))
    assert out.shape == (0, 50 + 882, 2) and out.dtype == np.float64


def _host_program():
    prog = _vn().tap_program(1000)
    return prog, prog.host_struct()


def test_batch_dev_rejects_bad_arguments_without_cuda():
    lib = N.lib()
    prog, ps = _host_program()
    ep = N.EpilogueStruct(1, 0, 0.0, 1, 0, 0)
    x = np.zeros((16, 2), np.float32)
    offs = np.array([0, 16], np.int64)
    pof = np.zeros(1, np.int32)
    out = np.zeros((16, 2), np.float32)

    def call(x_ptr=x.ctypes.data, x_dtype=N.VND_F32, rows=16, offs_ptr=offs.ctypes.data, n=1, pof_ptr=pof.ctypes.data, taps=C.byref(ps),
             epi=C.byref(ep), out_ptr=out.ctypes.data, out_dtype=N.VND_F32):
        return lib.vnd_vn_decorrelate_batch_dev(x_ptr, x_dtype, rows, offs_ptr, n, pof_ptr, taps, epi, out_ptr, out_dtype, None, 0, None)

    assert call(x_ptr=None) == N.VND_EINVAL
    assert call(offs_ptr=None) == N.VND_EINVAL
    assert call(pof_ptr=None) == N.VND_EINVAL
    assert call(out_ptr=None) == N.VND_EINVAL
    assert call(taps=None) == N.VND_EINVAL
    assert call(epi=None) == N.VND_EINVAL
    assert call(rows=-1) == N.VND_EINVAL
    assert call(n=-1) == N.VND_EINVAL
    assert call(x_dtype=N.VND_F64) == N.VND_EINVAL
    assert call(out_dtype=7) == N.VND_EINVAL
    bad_ep = N.EpilogueStruct(1, 0, 0.0, 1, -5, 0)
    assert call(epi=C.byref(bad_ep)) == N.VND_EINVAL
    odd = N.TapProgramStruct(ps.words, ps.offsets, ps.n_words, 1, ps.order, ps.apply_gain, ps.halo, ps.max_channel_words)
    assert call(taps=C.byref(odd)) == N.VND_EINVAL
    assert "two per filter" in lib.vnd_last_error().decode()
    assert call(n=0, rows=0) == N.VND_OK  # nothing to do, nothing launched


def test_layout_checks_reject_bad_offsets_and_program_indices():
    D._check_batch_layout(np.array([0, 3, 3, 7]), np.array([0, 1, 0], np.int32), 2, 7)
    with pytest.raises(ValueError, match="decrease"):
        D._check_batch_layout(np.array([0, 5, 3, 7]), np.array([0, 0, 0], np.int32), 1, 7)
    with pytest.raises(ValueError, match="from 0"):
        D._check_batch_layout(np.array([1, 3, 7]), np.array([0, 0], np.int32), 1, 7)
    with pytest.raises(ValueError, match="from 0"):
        D._check_batch_layout(np.array([0, 3, 6]), np.array([0, 0], np.int32), 1, 7)
    with pytest.raises(ValueError, match="program indices"):
        D._check_batch_layout(np.array([0, 3, 7]), np.array([0, 2], np.int32), 2, 7)
    with pytest.raises(ValueError, match="program indices"):
        D._check_batch_layout(np.array([0, 3, 7]), np.array([-1, 0], np.int32), 2, 7)


def test_programs_are_shared_by_clips_longer_than_the_filter():
    vn = _vn()
    table = vn.velvet_noise
    longest = int(table.index[table.filtered].max()) + 1
    lengths = [longest + 5000, 10, longest, 44100, 10, longest - 1]
    progs, prog_of = D._batch_programs([vn] * len(lengths), lengths)
    assert prog_of[0] == prog_of[2] == prog_of[3]  # every length the filter fits in: one program
    assert prog_of[1] == prog_of[4]  # the cache gives equal short lengths one program too
    assert len({int(prog_of[0]), int(prog_of[1]), int(prog_of[5])}) == 3
    assert progs[prog_of[1]].halo <= 10 and progs[prog_of[5]].halo < longest
    other = _vn(seed=2)
    progs2, prog_of2 = D._batch_programs([vn, other, vn], [44100, 44100, 50000])
    assert len(progs2) == 2 and list(prog_of2) == [0, 1, 0]
    packed = D._batch_program(progs2)
    assert packed.channels == 4 and list(packed.offsets[:3]) == list(progs2[0].offsets)
    assert np.array_equal(packed.words[packed.offsets[2]:packed.offsets[4]], progs2[1].words)


# ------------------------------------------------------------------ GPU: parity with the single-clip API


def _check(clips, dec, got):
    decs = dec if isinstance(dec, list) else [dec] * len(clips)
    assert len(got) == len(clips)
    for i, (x, d, y) in enumerate(zip(clips, decs, got)):
        want = d(x)
        assert _same(y, want), f"clip {i} (length {x.shape[0]}) differs from the single-clip call"


RAGGED = [0, 1, 127, 1023, 1024, 1025, 4095, 4096, 20479, 20480, 1_050_001, 500]


@gpu
@pytest.mark.parametrize("normalizer", [rms_normalize, None], ids=["rms", "none"])
def test_ragged_lengths_numpy(normalizer):
    clips = _clips(RAGGED, seed=1, mono=(3, 8), int16=(5,), f64=(9,))
    vn = _vn(normalizer=normalizer)
    _check(clips, vn, D.decorrelate_batch(clips, vn))


@gpu
@pytest.mark.parametrize("normalizer", [rms_normalize, None], ids=["rms", "none"])
def test_ragged_lengths_cuda_tensors(normalizer):
    import torch

    clips = [torch.from_numpy(np.ascontiguousarray(c)).cuda() for c in _clips(RAGGED, seed=2, mono=(2,), int16=(6,), f64=(7,))]
    vn = _vn(normalizer=normalizer)
    got = D.decorrelate_batch(clips, vn)
    assert all(g.is_cuda for g in got)
    _check(clips, vn, got)


@gpu
def test_equal_length_array_form():
    import torch

    x3 = (np.random.default_rng(3).standard_normal((6, 30000, 2)) * 0.3).astype(np.float32)
    chain = D.SignalChain(sample_rate_hz=FS).velvet_noise(seed=1).haas_effect(delay_time_seconds=0.02, mode="LR")
    got = D.decorrelate_batch(x3, chain)
    assert isinstance(got, np.ndarray) and got.shape == (6, 30000 + 882, 2) and got.dtype == np.float64
    for i in range(6):
        assert _same(got[i], chain(x3[i]))
    t3 = torch.from_numpy(x3).cuda()
    gt = D.decorrelate_batch(t3, chain)
    assert gt.is_cuda and gt.shape == (6, 30000 + 882, 2)
    assert _same(gt, got)


@gpu
@pytest.mark.parametrize("mode", ["MS", "LR"])
@pytest.mark.parametrize("width", [None, 0.3])
@pytest.mark.parametrize("normalizer", [rms_normalize, None], ids=["rms", "none"])
@pytest.mark.parametrize("filtered", [(0,), (0, 1)])
@pytest.mark.parametrize("envelope", [(1.0,), (0.85, 0.55, 0.35, 0.2)], ids=["identity", "decay"])
def test_every_mode(mode, width, normalizer, filtered, envelope):
    clips = _clips([7000, 1, 15000, 333, 0, 9001], seed=4, mono=(3,))
    vn = _vn(mode=mode, width=width, normalizer=normalizer, filtered_channels=filtered, segment_envelope=envelope)
    _check(clips, vn, D.decorrelate_batch(clips, vn))


def _cfg2_chain():
    return (D.SignalChain(sample_rate_hz=FS)
            .velvet_noise(duration_seconds=0.03, num_impulses=30, log_distribution_strength=1.0, seed=1)
            .haas_effect(delay_time_seconds=0.02, mode="LR"))


def _example_chain():
    return (D.SignalChain(sample_rate_hz=FS)
            .velvet_noise(duration_seconds=0.02, num_impulses=30, seed=1, log_distribution_strength=1.0, mode="MS", filtered_channels=(0, 1))
            .haas_effect(delay_time_seconds=0.02, delayed_channel=1, mode="LR"))


@gpu
@pytest.mark.parametrize("make", [_cfg2_chain, _example_chain], ids=["cfg2", "example"])
def test_chains(make):
    import torch

    clips = _clips([20000, 0, 513, 70000], seed=5, mono=(2,))
    got = D.decorrelate_batch(clips, make())
    _check(clips, make(), got)
    tclips = [torch.from_numpy(c).cuda() for c in clips]
    _check(tclips, make(), D.decorrelate_batch(tclips, make()))


@gpu
def test_committed_hashes_of_the_wav_fixtures():
    names = ["viola", "vocal", "guitar"]
    wavs = [G.wav(n) for n in names]
    assert all(fs == FS for fs, _ in wavs)
    clips = [x for _, x in wavs]
    h = G.hashes()
    for name, y in zip(names, D.decorrelate_batch(clips, _example_chain())):
        assert list(y.shape) == h["example_chain"][name]["shape"] and y.dtype == np.float64
        assert G.sha(y) == h["example_chain"][name]["sha256"], name
    y = D.decorrelate_batch(clips, _vn())[0]
    assert G.sha(y) == h["cfg1_decorrelate_viola"]
    y = D.decorrelate_batch(clips, _cfg2_chain())[2]
    assert list(y.shape) == h["cfg2_chain_guitar"]["shape"] and G.sha(y) == h["cfg2_chain_guitar"]["sha256"]


@gpu
def test_direct_oracle_comparison():
    from oracle import vnd_oracle as O

    clips = _clips([50000, 3000, 120000], seed=6)
    taps = O.class_taps(sample_rate_hz=FS, seed=1)
    for x, y in zip(clips, D.decorrelate_batch(clips, _vn())):
        assert G.same_bits(y, O.vn_decorrelate(x, taps))


@gpu
def test_per_clip_decorrelators():
    from vndecorrelate_b200.optimization import optimize_velvet_noise_batch

    clips = _clips([24000] * 3, seed=7)
    kappas = optimize_velvet_noise_batch(input_signals=clips, sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, seed=1, grid_size=12)
    decs = [_vn(log_distribution_strength=float(k)) for k in kappas]
    decs += [_vn(seed=5, num_impulses=20), _vn(seed=9, num_impulses=40, duration_seconds=0.05)]
    clips += _clips([31000, 900], seed=8)
    _check(clips, decs, D.decorrelate_batch(clips, decs))


@gpu
def test_long_filter_goes_clip_by_clip():
    import torch

    vn = _vn(duration_seconds=1.0, num_impulses=60)  # a halo of ~44 k frames: too long for the batched kernel
    assert vn.tap_program(10**6).halo > 30000
    clips = _clips([60000, 0, 20000, 90000], seed=9)
    _check(clips, vn, D.decorrelate_batch(clips, vn))
    tclips = [torch.from_numpy(c).cuda() for c in clips]
    _check(tclips, vn, D.decorrelate_batch(tclips, vn))


@gpu
def test_host_pipeline_matches_one_shot(monkeypatch):
    from vndecorrelate_b200 import runtime as R

    lengths = [int(v) for v in np.random.default_rng(10).integers(20000, 60000, size=40)]
    clips = _clips(lengths, seed=11)
    chain = _cfg2_chain()
    monkeypatch.setenv("VND_NO_PIPELINE", "1")
    one_shot = [np.array(y) for y in D.decorrelate_batch(clips, chain)]
    monkeypatch.delenv("VND_NO_PIPELINE")
    monkeypatch.setenv("VND_PIPE_CHUNK_MB", "1")
    piped = D.decorrelate_batch(clips, chain)  # pageable packed input
    for a, b in zip(piped, one_shot):
        assert G.same_bits(a, b)
    _check(clips[:3], _cfg2_chain(), piped[:3])
    pinned = R.PinnedArray((24, 50000, 2))  # page-locked input, already packed (the owner keeps the block alive)
    x3 = pinned.array
    x3[...] = (np.random.default_rng(12).standard_normal(x3.shape) * 0.3).astype(np.float32)
    vn = _vn()
    got = D.decorrelate_batch(x3, vn)
    monkeypatch.setenv("VND_NO_PIPELINE", "1")
    want = D.decorrelate_batch(x3, vn)
    assert G.same_bits(got, want)
    assert _same(got[5], vn(x3[5]))


@gpu
@pytest.mark.parametrize("normalizer,launches", [(None, 1), (rms_normalize, 3)], ids=["none", "rms"])
def test_launch_count_is_independent_of_the_clip_count(normalizer, launches):
    import torch

    vn = _vn(normalizer=normalizer)
    for n in (4, 400):
        lengths = np.random.default_rng(n).integers(0, 5000, size=n)
        clips = [torch.from_numpy(c).cuda() for c in _clips(lengths, seed=n)]
        D.decorrelate_batch(clips, vn)  # warm caches (tap programs, module loading)
        before = N.launch_count()
        D.decorrelate_batch(clips, vn)
        assert N.launch_count() - before == launches, n


@gpu
def test_batch_host_rejects_bad_layout():
    from vndecorrelate_b200 import runtime as R

    lib = N.lib()
    prog, ps = _host_program()
    ep = N.EpilogueStruct(1, 0, 0.0, 1, 0, 0)
    x = np.zeros((16, 2), np.float32)
    out = np.zeros((16, 2), np.float32)
    ctx = R.HostContext.get().handle

    def call(offs, pof):
        offs = np.asarray(offs, np.int64)
        pof = np.asarray(pof, np.int32)
        return lib.vnd_vn_decorrelate_batch_host(ctx, x.ctypes.data, N.VND_F32, 16, offs.ctypes.data, len(pof), pof.ctypes.data, C.byref(ps),
                                                 C.byref(ep), out.ctypes.data, N.VND_F32)

    assert call([0, 10, 8, 16], [0, 0, 0]) == N.VND_EINVAL
    assert call([1, 10, 16], [0, 0]) == N.VND_EINVAL
    assert call([0, 10, 15], [0, 0]) == N.VND_EINVAL
    assert call([0, 10, 16], [0, 1]) == N.VND_EINVAL
    assert call([0, 10, 16], [-1, 0]) == N.VND_EINVAL
    assert call([0, 10, 16], [0, 0]) == N.VND_OK
