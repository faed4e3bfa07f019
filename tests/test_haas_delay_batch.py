"""optimize_haas_delay_batch: the Haas-delay optimiser over many clips of any lengths, each clip's delay equal to the
single-clip ``optimize_haas_delay``; and the pair-list form of the Haas objective kernel it runs on.

The CPU tests check the vectorised scoring bit for bit against the one-row chain, argument handling, the C ABI's
argument checks, and - with an oracle-backed clip bank over gloo - the partition, the collectives and the lock-step
refinement against the reference's procedure clip by clip.  The GPU tests check the pair kernel bit for bit against the
grid kernel, per-clip equality with the single-clip optimiser, the committed known answer, the launch count and the
two-GPU run.
"""

from __future__ import annotations

import os
import socket

import numpy as np
import pytest

from oracle import vnd_oracle as O
from tests import _golden as G
from vndecorrelate_b200 import _native as N
from vndecorrelate_b200 import optimization as OPT
from vndecorrelate_b200.utils.dsp import EPSILON

gpu = pytest.mark.gpu
KW = dict(angle_limit=np.pi / 4, lambda_mean=5.0, lambda_skew=2.0, lambda_correlation=15.0, lambda_penalty=1e3)


# ------------------------------------------------------------------ CPU: vectorised scoring


def _score_rows():
    rng = np.random.default_rng(11)
    n = 4000
    p = np.empty((n, N.HAAS_SLOTS))
    p[:, 0] = rng.uniform(0.0, 5e4, n)                       # sum r
    p[:, 1] = rng.normal(0.0, 1.0, n) * p[:, 0] * 0.3          # sum r th
    p[:, 2] = rng.uniform(0.0, 0.8, n) * p[:, 0]               # sum r th^2
    p[:, 3] = rng.normal(0.0, 0.2, n) * p[:, 0]                # sum r th^3
    p[:, 4] = rng.uniform(0.0, np.pi / 2, n)                   # max |th|
    p[:, 6] = rng.uniform(0.0, 3e3, n)                         # sum L L
    p[:, 5] = rng.uniform(-1.0, 1.0, n) * p[:, 6]              # sum L R
    p[:, 7] = rng.integers(1, 2_000_000, n)
    a = np.pi / 4
    edge = [
        np.zeros(8),                                           # all-zero sums
        [10.0, 1.0, 2.0, 0.3, a - 1e-12, 4.0, 9.0, 100.0],     # max|th| just below the limit
        [10.0, 1.0, 2.0, 0.3, a, 4.0, 9.0, 100.0],             # at it
        [10.0, 1.0, 2.0, 0.3, a + 1e-12, 4.0, 9.0, 100.0],     # just above
        [10.0, 1.0, 2.0, 0.3, 1.5, 4.0, 9.0, 100.0],           # well above
        [10.0, 0.5, 1e-13, 1e-14, 0.2, 4.0, 9.0, 100.0],       # spread below EPSILON
        [10.0, 0.5, 10.0 * EPSILON, 1e-14, 0.2, 4.0, 9.0, 1.0],  # spread about EPSILON
        [10.0, 0.5, 0.0, -1e-12, 0.2, 4.0, 9.0, 100.0],        # zero spread, negative third moment
        [10.0, 1.0, 2.0, 0.3, 0.2, 0.0, 0.0, 100.0],           # sum L*L == 0 (and L*R)
        [10.0, 1.0, 2.0, 0.3, 0.2, 3.0, 0.0, 100.0],           # sum L*L == 0, L*R not
        [1e300, 3e299, 5e299, -1e299, 0.7, 1e300, 2e300, 1e9],  # very large magnitudes
        [1e150, -2e149, 4e149, 1e148, 0.9, -1e150, 1e150, 1e9],
        [1e-300, 1e-301, 1e-301, 1e-302, 0.1, 1e-300, 1e-300, 1.0],  # tiny magnitudes
    ]
    return np.vstack([p, np.asarray(edge, dtype=np.float64)])


def test_haas_scores_rows_equal_the_one_row_chain_bit_for_bit():
    p = _score_rows()
    got = OPT._haas_scores_rows(p, **KW)
    want = np.array([OPT._haas_score(row, **KW) for row in p], dtype=np.float64)
    assert got.dtype == np.float64 and got.shape == (len(p),)
    assert G.same_bits(got, want)
    other = dict(angle_limit=0.3, lambda_mean=1.5, lambda_skew=0.25, lambda_correlation=40.0, lambda_penalty=7.0)
    assert G.same_bits(OPT._haas_scores_rows(p, **other), np.array([OPT._haas_score(row, **other) for row in p]))
    # and haas_scores_from_partials, the public entry point, goes through it with its shapes
    p3 = p[:4000].reshape(40, 100, N.HAAS_SLOTS)
    assert G.same_bits(OPT.haas_scores_from_partials(p3, **KW), want[:4000].reshape(40, 100))
    assert OPT.haas_scores_from_partials(np.zeros((0, 5, 8)), **KW).shape == (0, 5)


# ------------------------------------------------------------------ CPU: argument handling

_FS, _MAXD, _GRID = 48000, 0.03, 24


class _NoBank:
    def __init__(self, *a, **k):
        raise AssertionError("device work started before the arguments were checked")


def _call(signals, **kw):
    return OPT.optimize_haas_delay_batch(input_signals=signals, sample_rate_hz=_FS, max_delay_seconds=_MAXD, grid_size=_GRID,
                                         _bank_factory=_NoBank, **kw)


def test_empty_clip_raises_with_its_index_before_any_device_work():
    clips = [O.coloured_clip(0, 500), O.coloured_clip(1, 700), np.zeros((0, 2), np.float32), O.coloured_clip(2, 300)]
    with pytest.raises(ValueError, match="clip 2 is empty"):
        _call(clips)
    with pytest.raises(ValueError, match="clip 1 is empty"):
        _call([np.ones(10, np.float32), np.zeros(0, np.int16)])


def test_bad_shapes_raise():
    with pytest.raises(ValueError, match=r"\(n_clips, frames, 2\)"):
        _call(np.zeros((3, 100, 3), np.float32))
    with pytest.raises(ValueError, match=r"\(n_clips, frames, 2\)"):
        _call(np.zeros((3, 100), np.float32))
    with pytest.raises(ValueError, match="clip 1"):
        _call([np.zeros((100, 2), np.float32), np.zeros((2, 100, 2), np.float32)])
    with pytest.raises(ValueError, match="clip 0"):
        _call([np.zeros((100, 1), np.float32)])


def test_mixed_numpy_and_torch_clips_raise():
    torch = pytest.importorskip("torch")
    with pytest.raises(ValueError, match="not a mix"):
        _call([np.zeros((100, 2), np.float32), torch.zeros((100, 2))])
    with pytest.raises(ValueError, match="CUDA"):
        _call([torch.zeros((100, 2)), torch.zeros((50, 2))])


def test_local_signals_need_total_clips_and_the_right_block():
    clips = [O.coloured_clip(i, 200) for i in range(3)]
    with pytest.raises(ValueError, match="total_clips"):
        OPT.optimize_haas_delay_batch(local_signals=clips, sample_rate_hz=_FS, max_delay_seconds=_MAXD, _bank_factory=_NoBank)
    with pytest.raises(ValueError, match="owns clips"):
        OPT.optimize_haas_delay_batch(local_signals=clips, total_clips=4, sample_rate_hz=_FS, max_delay_seconds=_MAXD, _bank_factory=_NoBank)
    with pytest.raises(ValueError, match="input_signals"):
        OPT.optimize_haas_delay_batch(sample_rate_hz=_FS, max_delay_seconds=_MAXD, _bank_factory=_NoBank)


def test_pairs_dev_rejects_bad_arguments_without_cuda():
    lib = N.lib()
    x = np.zeros((2, 16), np.float32)
    offs = np.array([0, 16], np.int64)
    pc = np.zeros(3, np.int32)
    pd = np.array([0, 1, 2], np.int32)
    out = np.zeros((3, 8), np.float64)

    def call(x_ptr=x.ctypes.data, rows=16, stride=16, offs_ptr=offs.ctypes.data, n=1, pc_ptr=pc.ctypes.data, pd_ptr=pd.ctypes.data, n_pairs=3,
             out_ptr=out.ctypes.data):
        return lib.vnd_haas_objective_pairs_dev(x_ptr, rows, stride, offs_ptr, n, pc_ptr, pd_ptr, n_pairs, out_ptr, None)

    assert call(x_ptr=None) == N.VND_EINVAL
    assert call(offs_ptr=None) == N.VND_EINVAL
    assert call(pc_ptr=None) == N.VND_EINVAL
    assert call(pd_ptr=None) == N.VND_EINVAL
    assert call(out_ptr=None) == N.VND_EINVAL
    assert call(rows=-1) == N.VND_EINVAL
    assert call(n=-1) == N.VND_EINVAL
    assert call(n_pairs=-1) == N.VND_EINVAL
    assert call(stride=15) == N.VND_EINVAL
    assert "chan_stride" in lib.vnd_last_error().decode()
    assert call(n=0) == N.VND_EINVAL  # pairs but no clips
    assert call(n_pairs=0) == N.VND_OK  # nothing to do, nothing launched
    assert call(n_pairs=0, x_ptr=None, offs_ptr=None, pc_ptr=None, pd_ptr=None, out_ptr=None) == N.VND_OK


# ------------------------------------------------------------------ CPU: two ranks over gloo, oracle-backed bank


class _OracleHaasBank:
    """The clip bank's interface, scoring every (clip, delay) pair with the oracle (the reference's procedure in numpy)."""

    lanes = 1

    def __init__(self, clips, kw):
        self.clips = [np.asarray(c) for c in clips]
        self.kw = kw
        self.n, self.device = len(self.clips), None
        self.evaluations = self.launches = 0

    def grid_scores(self, delays):
        return self.submit(np.repeat(np.arange(self.n), len(delays)), np.tile(delays, self.n)).reshape(self.n, len(delays))

    def submit(self, clip_ids, delays):
        self.launches += 1
        self.evaluations += len(clip_ids)
        # sample_rate_hz=1 makes the oracle's round(t * fs) the delay in frames itself
        return np.array([O.objective(O.haas(self.clips[c], sample_rate_hz=1, delay_time_seconds=int(d)), **self.kw)
                         for c, d in zip(clip_ids, delays)], dtype=np.float64)

    def collect(self, handle):
        return handle


_LENGTHS = (3000, 4500, 1200, 5200, 3700)


def _ragged_clips():
    return [O.coloured_clip(i, n) for i, n in enumerate(_LENGTHS)]


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gloo_worker(rank, world, port, result_dir):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        taus, info = OPT.optimize_haas_delay_batch(input_signals=_ragged_clips(), sample_rate_hz=_FS, max_delay_seconds=_MAXD, grid_size=_GRID,
                                                  details=True, _bank_factory=_OracleHaasBank)
        np.save(os.path.join(result_dir, f"tau_{rank}.npy"), taus)
        np.save(os.path.join(result_dir, f"scores_{rank}.npy"), info["scores"])
    finally:
        dist.destroy_process_group()


def test_optimize_haas_delay_batch_world2_gloo(tmp_path):
    import torch.multiprocessing as mp

    world = 2
    mp.spawn(_gloo_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    clips = _ragged_clips()
    one, info = OPT.optimize_haas_delay_batch(input_signals=clips, sample_rate_hz=_FS, max_delay_seconds=_MAXD, grid_size=_GRID, details=True,
                                              _bank_factory=_OracleHaasBank)
    assert info["launches_local"] == 1 + info["rounds_local"]  # one evaluation call for the grid, one per Brent round
    assert info["scores"].shape == (len(clips), _GRID) and info["scores"].dtype == np.float64
    # the reference's procedure, clip by clip, one scipy minimiser at a time
    taus = np.linspace(0.0, _MAXD, _GRID)
    want, want_scores = [], []
    for c in clips:
        row = O.haas_grid_scores(c, taus, sample_rate_hz=_FS)
        want_scores.append(row)
        fn = lambda t, c=c: O.objective(O.haas(c, sample_rate_hz=_FS, delay_time_seconds=t))  # noqa: E731
        want.append(O.refine(OPT.get_local_minima(row, _GRID), taus, fn))
    want = np.asarray(want, dtype=np.float64)
    assert np.array_equal(info["scores"], np.asarray(want_scores))
    assert one.dtype == np.float64 and np.array_equal(one, want)
    for r in range(world):
        assert np.array_equal(np.load(os.path.join(str(tmp_path), f"tau_{r}.npy")), want)              # every rank: all clips, same bits
        assert np.array_equal(np.load(os.path.join(str(tmp_path), f"scores_{r}.npy")), info["scores"])  # and the full score matrix


# ------------------------------------------------------------------ GPU: the pair kernel against the grid kernel


def _pack(clips):
    """Channel-planar float32 (2, rows) and the int64 offsets of (frames, 2) float32 clips."""
    offs = np.concatenate([[0], np.cumsum([len(c) for c in clips])]).astype(np.int64)
    x = np.empty((2, int(offs[-1])), np.float32)
    for c, a, b in zip(clips, offs[:-1], offs[1:]):
        x[:, a:b] = c.T
    return x, offs


def _pair_case():
    rng = np.random.default_rng(5)
    fs, viola = G.wav("viola")
    _, vocal = G.wav("vocal")
    clips = [
        viola[40000:52000],
        (rng.standard_normal((1, 2)) * 0.3).astype(np.float32),     # one frame
        vocal[90000:90700],                                         # shorter than the largest delay
        (rng.standard_normal((7001, 2)) * 0.2).astype(np.float32),
        O.coloured_clip(3, 2500),
        viola[100000:100001 + 4096],
    ]
    delays = [0, 1, 5, 255, 256, 257, 699, 700, 701, 1000, 1323]
    pairs = np.array([(i, d) for i in range(len(clips)) for d in delays], dtype=np.int32)
    pairs = pairs[rng.permutation(len(pairs))]  # any order
    return clips, pairs


@gpu
def test_pair_partials_equal_the_grid_kernel_bit_for_bit():
    import torch

    clips, pairs = _pair_case()
    x, offs = _pack(clips)
    want = np.stack([OPT.haas_objective_partials(clips[c], [d])[0, 0] for c, d in pairs])
    host = OPT.haas_objective_pair_partials(x, offs, pairs[:, 0], pairs[:, 1])
    assert G.same_bits(host, want)
    xt = torch.from_numpy(x).cuda()
    dev = OPT.haas_objective_pair_partials(xt, torch.from_numpy(offs).cuda(), torch.from_numpy(pairs[:, 0].copy()).cuda(),
                                           torch.from_numpy(pairs[:, 1].copy()).cuda())
    assert G.same_bits(dev.cpu().numpy(), want)
    # a wider stride between the two channels changes nothing
    wide = np.zeros((2, x.shape[1] + 37), np.float32)
    wide[:, : x.shape[1]] = x
    assert G.same_bits(OPT.haas_objective_pair_partials(wide, offs, pairs[:, 0], pairs[:, 1]), want)


@gpu
def test_pairs_host_checks_offsets_and_pairs_before_any_copy():
    clips, pairs = _pair_case()
    x, offs = _pack(clips)
    with pytest.raises(N.VndError, match="decrease"):
        OPT.haas_objective_pair_partials(x, np.array([0, 9000, 100] + list(offs[3:])), pairs[:, 0], pairs[:, 1])
    with pytest.raises(N.VndError, match="not 0"):
        OPT.haas_objective_pair_partials(x, np.concatenate([[1], offs[1:]]), pairs[:, 0], pairs[:, 1])
    with pytest.raises(N.VndError, match="pair_clip"):
        OPT.haas_objective_pair_partials(x, offs, np.array([0, len(clips)]), np.array([1, 1]))
    with pytest.raises(N.VndError, match="negative"):
        OPT.haas_objective_pair_partials(x, offs, np.array([0, 1]), np.array([1, -1]))
    with pytest.raises(N.VndError, match="empty"):
        OPT.haas_objective_pair_partials(x, np.array(list(offs) + [offs[-1]]), np.array([len(clips)]), np.array([0]))
    # an empty clip with a positive delay has an objective (d frames of silence)
    got = OPT.haas_objective_pair_partials(x, np.array(list(offs) + [offs[-1]]), np.array([len(clips)]), np.array([3]))
    assert got[0, 7] == 3.0 and not np.any(got[0, :7])


# ------------------------------------------------------------------ GPU: per-clip equality with optimize_haas_delay


def _mixed_clips():
    rng = np.random.default_rng(9)
    fs, viola = G.wav("viola")
    _, vocal = G.wav("vocal")
    _, guitar = G.wav("guitar")
    clips = [
        viola[40000:80000],
        vocal[20000:51000],
        guitar[100000:157000],
        (rng.standard_normal(23000) * 0.3).astype(np.float32),                   # mono
        (rng.standard_normal((18000, 2)) * 3000).astype(np.int16),               # int16, not rescaled
        rng.standard_normal((26000, 2)) * 0.2,                                   # float64
        np.column_stack([viola[120000:150000], vocal[60000:90000, :1]]),         # (frames, 3)
        O.coloured_clip(7, 900),                                                 # shorter than the largest delay
        (rng.standard_normal((2, 2)) * 0.3).astype(np.float32),                  # two frames
    ]
    return fs, clips


def _single(clip, fs, grid):
    return OPT.optimize_haas_delay(input_signal=clip, sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=grid)


@gpu
def test_batch_equals_the_single_clip_optimiser_numpy_list():
    fs, clips = _mixed_clips()
    got = OPT.optimize_haas_delay_batch(input_signals=clips, sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=48)
    assert got.dtype == np.float64 and got.shape == (len(clips),)
    for i, c in enumerate(clips):
        assert got[i] == _single(c, fs, 48), f"clip {i}"
    three = [clips[0], clips[3], clips[5]]
    got = OPT.optimize_haas_delay_batch(input_signals=three, sample_rate_hz=fs, max_delay_seconds=0.03)  # the default grid of 400
    for i, c in enumerate(three):
        assert got[i] == _single(c, fs, 400), f"clip {i} at grid 400"


@gpu
def test_batch_equals_the_single_clip_optimiser_cuda_tensors_and_3d_array():
    import torch

    fs, clips = _mixed_clips()
    tensors = [torch.from_numpy(np.ascontiguousarray(c)).cuda() for c in clips]
    got = OPT.optimize_haas_delay_batch(input_signals=tensors, sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=48)
    for i, t in enumerate(tensors):
        assert got[i] == _single(t.cpu().numpy(), fs, 48), f"clip {i}"
    _, viola = G.wav("viola")
    stack = np.stack([viola[a: a + 30000] for a in (10000, 70000, 130000, 190000)])
    got = OPT.optimize_haas_delay_batch(input_signals=stack, sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=48)
    for i in range(len(stack)):
        assert got[i] == _single(stack[i], fs, 48), f"row {i}"
    got_t = OPT.optimize_haas_delay_batch(input_signals=torch.from_numpy(stack).cuda(), sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=48)
    assert np.array_equal(got_t, got)


@gpu
def test_known_answer_viola_40k():
    fs, viola = G.wav("viola")
    ref = G.objective()["optimize_haas_viola_40k"]
    got = OPT.optimize_haas_delay_batch(input_signals=[viola[40000:80000]], sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=ref["grid_size"])
    assert abs(got[0] - ref["tau"]) <= 1e-4  # Brent's xatol (optimization.py:148)


@gpu
def test_launches_are_one_plus_the_brent_rounds_whatever_the_clip_count():
    fs, viola = G.wav("viola")
    rng = np.random.default_rng(3)
    starts = rng.integers(0, len(viola) - 40000, 16)
    clips = [viola[s: s + int(rng.integers(5000, 40000))] for s in starts]
    counts = {}
    for n in (2, 16):
        before = N.launch_count()
        _, info = OPT.optimize_haas_delay_batch(input_signals=clips[:n], sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=64, details=True)
        launches = N.launch_count() - before
        assert launches == info["launches_local"] == 1 + info["rounds_local"], (n, launches, info["rounds_local"])
        counts[n] = (launches, info["evaluations_local"])
    # the per-clip loop would launch once per clip for the grid and once per clip and round: the batch does not grow with
    # the clip count beyond the longest minimiser (500 evaluations at most)
    assert counts[16][1] > counts[2][1] and counts[16][0] <= 1 + 500


# ------------------------------------------------------------------ GPU: two ranks over NCCL


def _nccl_worker(rank, world, port, result_dir):
    import torch
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ["VND_DEVICE"] = str(rank)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world)
    try:
        fs, clips = _mixed_clips()
        taus = OPT.optimize_haas_delay_batch(input_signals=clips, sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=48)
        np.save(os.path.join(result_dir, f"tau_{rank}.npy"), taus)
    finally:
        dist.destroy_process_group()


@gpu
def test_world2_nccl_equals_world1(tmp_path):
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world = 2
    mp.spawn(_nccl_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    fs, clips = _mixed_clips()
    one = OPT.optimize_haas_delay_batch(input_signals=clips, sample_rate_hz=fs, max_delay_seconds=0.03, grid_size=48)
    for r in range(world):
        assert np.array_equal(np.load(os.path.join(str(tmp_path), f"tau_{r}.npy")), one)
