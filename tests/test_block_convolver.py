"""BlockConvolver: live multichannel signals convolved block by block, one launch per step for all signals and channels,
each signal's concatenated output byte-identical to ``VelvetNoise.convolve`` on its concatenated input.

The CPU tests check the argument handling (every error before any device work, with the signal's index), the
generalised batch program and the C ABI's argument checks.  The GPU tests cut signals into blocks in many ways and
compare every signal's concatenated output with the one-shot call.
"""

from __future__ import annotations

import ctypes as C
import zlib

import numpy as np
import pytest

from tests import _golden as G
from vndecorrelate_b200 import _native as N
from vndecorrelate_b200 import decorrelation as D
from vndecorrelate_b200.taps import TapProgram

gpu = pytest.mark.gpu
FS = 48000


def _vn(**kw):
    base = dict(sample_rate_hz=FS, num_outs=4, filtered_channels=(0, 1, 2, 3), mode="LR", normalizer=None, seed=3)
    base.update(kw)
    return D.VelvetNoise(**base)


def _cfg3(num_outs, seed=1):
    return D.VelvetNoise(sample_rate_hz=FS, duration_seconds=0.03, num_impulses=30, num_outs=num_outs, filtered_channels=tuple(range(num_outs)),
                         mode="LR", normalizer=None, seed=seed)


def _cfg4(num_outs, seed=1):
    return D.VelvetNoise(sample_rate_hz=96000, duration_seconds=0.3, num_impulses=300, num_outs=num_outs,
                         filtered_channels=tuple(range(num_outs)), mode="LR", normalizer=None, seed=seed)


@pytest.fixture
def no_device(monkeypatch):
    """Call ``no_device()`` after building the objects: from then on any call into the native library fails the test."""

    def forbid():
        def forbidden(*a, **k):
            raise AssertionError("the native library was called")

        monkeypatch.setattr(N, "lib", forbidden)

    return forbid


# ------------------------------------------------------------------ CPU: construction


def test_construction_errors_name_the_signal():
    with pytest.raises(TypeError, match="takes a VelvetNoise"):
        D.BlockConvolver(object(), 2)
    with pytest.raises(TypeError, match="signal 1: BlockConvolver takes VelvetNoise filters, not HaasEffect"):
        D.BlockConvolver([_vn(), D.HaasEffect(sample_rate_hz=FS)], 2)
    with pytest.raises(ValueError, match="3 filters for 2 signals"):
        D.BlockConvolver([_vn()] * 3, 2)
    with pytest.raises(ValueError, match="n_signals must be at least 1"):
        D.BlockConvolver(_vn(), 0)
    with pytest.raises(ValueError, match="signal 2: BlockConvolver needs one num_outs for every signal, got 4 and 2"):
        D.BlockConvolver([_vn(), _vn(seed=4), _vn(num_outs=2, filtered_channels=(0, 1))], 3)
    with pytest.raises(ValueError, match="signal 1: BlockConvolver needs one identity segment_envelope"):
        D.BlockConvolver([_vn(), _vn(segment_envelope=(1.0,))], 2)


def test_mode_width_and_normalizer_are_ignored():
    b = D.BlockConvolver([_vn(), _vn(mode="MS", num_outs=4, width=0.3, normalizer=D.rms_normalize)], 2)
    assert b.num_outs == 4


def test_latency_is_the_largest_tap_index():
    vns = [_vn(seed=s, duration_seconds=0.01 * (s + 1)) for s in (1, 2, 3)]
    b = D.BlockConvolver(vns, 3)
    want = [int(v.velvet_noise.index[v.velvet_noise.filtered].max()) for v in vns]
    assert b.latency_frames.dtype == np.int64 and b.latency_frames.tolist() == want
    assert D.BlockConvolver(vns[0], 2).latency_frames.tolist() == [want[0]] * 2


def test_batch_program_is_unchanged_for_two_channels():
    """The generalised _batch_program gives the stereo callers the program of the two-channel formula, byte for byte."""
    vns = [D.VelvetNoise(sample_rate_hz=44100, normalizer=None, seed=s, filtered_channels=fc) for s, fc in ((1, (0, 1)), (2, (0,)), (3, (0, 1)))]
    progs = [v.tap_program(10**9) for v in vns] + [vns[0].tap_program(500)]
    got = D._batch_program(progs)
    words = np.concatenate([p.words for p in progs]).astype(np.int32)
    bases = np.cumsum([0] + [p.words.size for p in progs[:-1]])
    offsets = np.concatenate([[0]] + [p.offsets[1:].astype(np.int64) + b for p, b in zip(progs, bases)]).astype(np.int32)
    assert got.channels == 2 * len(progs) and got.order == N.ORDER_SEGMENTED
    assert got.words.tobytes() == words.tobytes() and got.offsets.tobytes() == offsets.tobytes()
    assert got.offsets.dtype == np.int32 and got.words.dtype == np.int32
    assert (got.apply_gain, got.halo, got.max_channel_words) == (progs[0].apply_gain, max(p.halo for p in progs),
                                                                 max(p.max_channel_words for p in progs))
    wide = D._batch_program([_vn(seed=1).tap_program(10**9), _vn(seed=2).tap_program(10**9)])
    assert wide.channels == 8 and wide.offsets.size == 9
    with pytest.raises(ValueError, match="one channel count"):
        D._batch_program([progs[0], wide])


# ------------------------------------------------------------------ CPU: rejections before device work


def test_step_rejections_name_the_signal(no_device):
    b = D.BlockConvolver(_vn(), 3)
    no_device()
    ok = np.zeros((8, 4), np.float32)
    with pytest.raises(ValueError, match="2 blocks for 3 signals"):
        b.process([ok, ok])
    with pytest.raises(IndexError, match="signal 1: too many indices for array: array is 1-dimensional"):
        b.process([ok, np.zeros(8, np.float32), ok])
    with pytest.raises(IndexError, match="signal 2: index 3 is out of bounds for axis 1 with size 3"):
        b.process([ok, None, np.zeros((8, 3), np.float32)])
    with pytest.raises(ValueError, match="signal 1: a block computed in float64 for a BlockConvolver computing in float32"):
        b.process([ok, np.zeros((8, 4), np.int32), None])
    with pytest.raises(ValueError, match="signal 1: a block computed in float32 for a BlockConvolver computing in float64"):
        b.process([np.zeros((8, 4), np.float64), np.zeros((8, 4), np.int16), None])
    assert b._received.tolist() == [0, 0, 0] and b._dtype is None


def test_a_signal_keeps_its_column_count_and_the_object_its_dtype(no_device):
    b = D.BlockConvolver(_vn(), 2)
    no_device()
    b._cols[:] = [5, -1]  # as after a 5-column block on signal 0
    b._dtype = np.dtype(np.float64)  # as after a first float64 block
    with pytest.raises(ValueError, match="signal 0: a block of 4 columns for a signal of 5"):
        b.process([np.zeros((3, 4)), None])
    with pytest.raises(ValueError, match="signal 1: a block computed in float32 for a BlockConvolver computing in float64"):
        b.process([np.zeros((3, 5)), np.zeros((0, 4), np.float32)])


def test_mixed_and_cpu_tensors_are_rejected(no_device):
    torch = pytest.importorskip("torch")
    b = D.BlockConvolver(_vn(), 2)
    no_device()
    with pytest.raises(ValueError, match="signal 1: the blocks of one step must be all numpy arrays or all CUDA tensors"):
        b.process([np.zeros((4, 4), np.float32), torch.zeros((4, 4))])
    with pytest.raises(N.VndError, match="signal 0: CPU torch tensors") as e:
        b.process([torch.zeros((4, 4)), None])
    assert e.value.status == N.VND_EUNSUPPORTED


# ------------------------------------------------------------------ CPU: the C ABI's argument checks


def _step(lib, prog: TapProgram, **over):
    ps = prog.host_struct()
    args = dict(x=None, dtype=N.VND_F32, rows=0, channels=4, offs=8, n=1, recv=8, emit=8, prog_of=8, taps=C.byref(ps), h_in=16, h_out=32,
                H=prog.halo, oo=8, out_rows=0, out=None, stream=None)
    args.update(over)
    return lib.vnd_fir_block_step_dev(*args.values())


def test_abi_rejects_illegal_arguments():
    lib = N.lib()
    prog = D.BlockConvolver(_vn(), 1)._program
    assert _step(lib, prog) == N.VND_OK  # nothing to do: no launch
    assert _step(lib, prog, rows=-1) == N.VND_EINVAL
    assert _step(lib, prog, n=-1) == N.VND_EINVAL
    assert _step(lib, prog, n=0, rows=4, x=8) == N.VND_EINVAL  # rows but no signals
    assert _step(lib, prog, rows=5, x=None) == N.VND_EINVAL
    assert _step(lib, prog, rows=5, x=2) == N.VND_EINVAL  # misaligned for float32
    assert _step(lib, prog, rows=5, x=4, dtype=N.VND_F64) == N.VND_EINVAL  # misaligned for float64
    assert _step(lib, prog, h_in=20, dtype=N.VND_F64) == N.VND_EINVAL
    assert _step(lib, prog, dtype=2) == N.VND_EINVAL
    assert _step(lib, prog, offs=None) == N.VND_EINVAL
    assert _step(lib, prog, emit=None) == N.VND_EINVAL
    assert _step(lib, prog, prog_of=None) == N.VND_EINVAL
    assert _step(lib, prog, out_rows=3, out=None) == N.VND_EINVAL
    assert _step(lib, prog, out_rows=3, out=6) == N.VND_EINVAL  # misaligned float32 out
    assert _step(lib, prog, h_out=16) == N.VND_EINVAL  # one buffer for both
    assert _step(lib, prog, h_in=None) == N.VND_EINVAL
    assert _step(lib, prog, H=prog.halo - 2) == N.VND_EINVAL  # shorter than the look-ahead
    assert _step(lib, prog, H=prog.halo - 1) == N.VND_OK
    assert _step(lib, prog, channels=3) == N.VND_EINVAL  # 4 program channels are not a multiple of 3
    assert _step(lib, prog, channels=0) == N.VND_EINVAL
    assert _step(lib, prog, channels=2) == N.VND_OK  # two 2-channel filters
    assert _step(lib, prog, taps=None) == N.VND_EINVAL
    asc = D.ascending_program(np.eye(4, dtype=np.float32), 100)
    assert _step(lib, asc, H=asc.halo) == N.VND_EINVAL  # ASCENDING order


# ------------------------------------------------------------------ GPU: byte equality with the one-shot call


def _np(a):
    return a if isinstance(a, np.ndarray) else a.cpu().numpy()


def _same(a, b) -> bool:
    return G.same_bits(_np(a), _np(b))


def _signal(L, cols, kind="f32", seed=0):
    rng = np.random.default_rng(seed)
    if kind == "int16":
        return rng.integers(-3000, 3000, size=(L, cols)).astype(np.int16)
    if kind == "int32":
        return rng.integers(-30000, 30000, size=(L, cols)).astype(np.int32)
    if kind == "f64":
        return rng.standard_normal((L, cols)) * 0.2
    return (rng.standard_normal((L, cols)) * 0.3).astype(np.float32)


def _cuts(L, A, rng):
    """Random cuts of L frames: empty, 1-frame, shorter-than-A and much-longer-than-a-tile blocks."""
    out, left = [], L
    while left > 0:
        s = int(rng.choice([0, 1, 2, max(A // 3, 1), A, A + 1, 512, 700, 5000]))
        out.append(min(s, left))
        left -= out[-1]
    return out + [0]


def _run(filters, signals, cuts, *, tensor=False, planar=False):
    """Feeds signal i the blocks cuts[i] (sizes; a None entry is an idle step), final at its last block, and returns each
    signal's concatenated output after checking the emitted counts after every non-final step."""
    torch = pytest.importorskip("torch")
    n = len(signals)
    b = D.BlockConvolver(filters, n)
    outs = [[] for _ in range(n)]
    at = [0] * n
    for s in range(max(len(c) for c in cuts)):
        blocks, fin = [], []
        for i in range(n):
            if s >= len(cuts[i]) or cuts[i][s] is None:
                blocks.append(None)
            else:
                x = signals[i][at[i]:at[i] + cuts[i][s]]
                at[i] += x.shape[0]
                if tensor:
                    x = torch.from_numpy(np.ascontiguousarray(x.T)).cuda().t() if planar else torch.from_numpy(np.ascontiguousarray(x)).cuda()
                blocks.append(x)
            fin.append(s == len(cuts[i]) - 1)
        res = b.process(blocks, final=fin)
        for i in range(n):
            if s < len(cuts[i]):
                assert isinstance(res[i], np.ndarray) != tensor
                outs[i].append(_np(res[i]))
                if not fin[i]:
                    assert sum(r.shape[0] for r in outs[i]) == max(0, at[i] - int(b.latency_frames[i]))
    return [np.concatenate(o) for o in outs]


def _check(filters, signals, cuts, **kw):
    per = filters if isinstance(filters, list) else [filters] * len(signals)
    got = _run(filters, signals, cuts, **kw)
    for i, (g, x) in enumerate(zip(got, signals)):
        want = per[i].convolve(x)
        assert _same(g, want), i


@gpu
@pytest.mark.parametrize("kind", ["f32", "f64", "int16", "int32"])
@pytest.mark.parametrize("mode", ["numpy", "tensor", "planar"])
def test_random_cuts_are_byte_identical_to_convolve(kind, mode):
    vn = _cfg3(6, seed=2)
    A = int(D.BlockConvolver(vn, 1).latency_frames[0])
    rng = np.random.default_rng(zlib.crc32(f"{kind}-{mode}".encode()))
    signals = [_signal(L, 6, kind, seed=k) for k, L in enumerate([9000, 6000, A // 2, 0, A + 1])]
    cuts = [_cuts(x.shape[0], A, rng) for x in signals]
    cuts[3] = [0]
    _check(vn, signals, cuts, tensor=mode != "numpy", planar=mode == "planar")


@gpu
def test_finals_at_different_steps_then_restart():
    vn = _vn()
    n = 5
    b = D.BlockConvolver(vn, n)
    rng = np.random.default_rng(11)
    pending = [[] for _ in range(n)]
    runs = [[] for _ in range(n)]
    checked = 0
    for s in range(40):
        blocks = [_signal(int(rng.choice([0, 1, 100, 512, 2000])), 4 + (i % 2), seed=100 * s + i) if rng.random() < 0.9 else None
                  for i in range(n)]
        fin = [bool(rng.random() < 0.15) or s == 39 for _ in range(n)]
        res = b.process(blocks, final=fin)
        for i in range(n):
            if blocks[i] is not None:
                pending[i].append(blocks[i])
            runs[i].append(res[i])
            if fin[i]:
                x = np.concatenate(pending[i]) if pending[i] else np.zeros((0, 4), np.float32)
                assert _same(np.concatenate(runs[i]), vn.convolve(x)), (i, s)
                pending[i], runs[i] = [], []
                checked += 1
    assert checked > n


@gpu
def test_extra_columns_and_a_strict_subset_of_filtered_channels():
    vn = _vn(num_outs=5, filtered_channels=(0, 1, 2), seed=8)
    signals = [_signal(7000, 7, seed=1), _signal(3000, 5, seed=2)]
    cuts = [[1000, 1, 3000, 2999], [512] * 5 + [440]]
    _check(vn, signals, cuts)
    _check(vn, signals, cuts, tensor=True)


@gpu
@pytest.mark.parametrize("channels", [37, 512])
def test_channel_counts_off_and_over_the_group_width(channels):
    vn = _cfg3(channels, seed=5)
    signals = [_signal(4000, channels, seed=1), _signal(2500, channels, "f64", seed=2)[:, :channels].astype(np.float32)]
    cuts = [[700, 1300, 2000], [1, 1499, 1000]]
    _check(vn, signals, cuts, tensor=True)


@gpu
def test_per_signal_filters_of_different_lengths():
    vns = [_vn(seed=10 + i, duration_seconds=0.005 * (i + 1), num_impulses=10 + 5 * i) for i in range(4)]
    signals = [_signal(5000 + 300 * i, 4, seed=i) for i in range(4)]
    cuts = [[512] * 12 for _ in range(4)]
    _check(vns, signals, cuts)
    _check(vns, signals, cuts, tensor=True)


@gpu
@pytest.mark.parametrize("kind", ["f32", "f64"])
def test_the_config4_filter_on_both_paths(kind):
    """float32 stages the halo in shared memory; float64 cannot and reads its taps from global memory."""
    vn = _cfg4(3, seed=1)
    A = int(D.BlockConvolver(vn, 1).latency_frames[0])
    signals = [_signal(A + 5000, 3, kind, seed=1), _signal(A // 3, 3, kind, seed=2)]
    cuts = [[1024] * ((A + 5000) // 1024) + [(A + 5000) % 1024], [1, A // 3 - 1]]
    _check(vn, signals, cuts, tensor=True)


@gpu
def test_one_launch_per_step_and_none_when_idle():
    torch = pytest.importorskip("torch")
    vn = _cfg3(16, seed=3)
    n = 8
    b = D.BlockConvolver(vn, n)
    for s in range(6):
        blocks = [torch.from_numpy(_signal(256 + 10 * i, 16, seed=s * n + i)).cuda() for i in range(n)]
        before = N.launch_count()
        b.process(blocks, final=s == 5)
        assert N.launch_count() - before == 1
    before = N.launch_count()
    assert all(r.shape == (0, 16) for r in b.process([None] * n))
    assert N.launch_count() == before


@gpu
def test_a_block_read_in_place():
    """A C-contiguous float32 tensor of exactly num_outs columns, the only non-empty block of the step, is not copied."""
    torch = pytest.importorskip("torch")
    vn = _vn()
    b = D.BlockConvolver(vn, 2)
    x = torch.from_numpy(_signal(3000, 4, seed=4)).cuda()
    keep, ptr = b._pack([x, x[:0]], np.array([0, 3000, 3000]), 3000, True, x.device, np.dtype(np.float32))
    assert ptr == x.data_ptr()
    _check(vn, [_signal(3000, 4, seed=4), _signal(0, 4)], [[3000], [0]], tensor=True)
