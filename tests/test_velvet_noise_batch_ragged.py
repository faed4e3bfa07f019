"""optimize_velvet_noise_batch over clips of any lengths, dtypes and channel counts, each clip's strength equal to the
single-clip ``optimize_velvet_noise``; and the run-list form of the velvet-noise objective kernel it runs on.

The CPU tests check argument handling, the C ABI's argument checks, the length-class tap programs against the
single-clip packing, and - with an oracle-backed ragged clip bank over gloo - the partition, the collectives and the
lock-step refinement against the reference's procedure clip by clip.  The GPU tests check the run kernel bit for bit
against the single-clip kernel on clips packed between loud neighbours, per-clip equality with the single-clip optimiser,
the launch counts, the pipeline into ``decorrelate_batch`` and the two-GPU run.
"""

from __future__ import annotations

import ctypes as C
import os
import re
import socket

import numpy as np
import pytest

from oracle import vnd_oracle as O
from tests import _golden as G
from vndecorrelate_b200 import _native as N
from vndecorrelate_b200 import optimization as OPT
from vndecorrelate_b200 import taps as T

gpu = pytest.mark.gpu
_FS, _DUR, _NIMP, _GRID = 48000, 0.03, 30, 24
_SETTINGS = dict(sample_rate_hz=_FS, duration_seconds=_DUR, num_impulses=_NIMP, seed=1)


def _family():
    return OPT._vn_family(**_SETTINGS)


# ------------------------------------------------------------------ CPU: argument handling


class _NoBank:
    def __init__(self, *a, **k):
        raise AssertionError("device work started before the arguments were checked")


def _call(signals, **kw):
    return OPT.optimize_velvet_noise_batch(input_signals=signals, grid_size=_GRID, _bank_factory=_NoBank, **_SETTINGS, **kw)


def test_empty_clip_raises_with_its_index_before_any_device_work():
    clips = [O.coloured_clip(0, 500), O.coloured_clip(1, 700), np.zeros((0, 2), np.float32), O.coloured_clip(2, 300)]
    with pytest.raises(ValueError, match="clip 2 is empty"):
        _call(clips)
    with pytest.raises(ValueError, match="clip 1 is empty"):
        _call([np.ones(10, np.float32), np.zeros(0, np.int16)])
    with pytest.raises(ValueError, match="clip 0 is empty"):
        _call(np.zeros((3, 2, 0), np.float32))


def test_bad_shapes_raise():
    with pytest.raises(ValueError, match=r"\(n_clips, 2, frames\)"):
        _call(np.zeros((3, 100, 2), np.float32))  # the Haas batch's layout, not this one's
    with pytest.raises(ValueError, match=r"\(n_clips, 2, frames\)"):
        _call(np.zeros((100, 2), np.float32))
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
    with pytest.raises(ValueError, match="CUDA"):
        _call(torch.zeros((2, 2, 50)))


def test_local_signals_need_total_clips_and_the_right_block():
    clips = [O.coloured_clip(i, 200 + 50 * i) for i in range(3)]
    with pytest.raises(ValueError, match="total_clips"):
        OPT.optimize_velvet_noise_batch(local_signals=clips, _bank_factory=_NoBank, **_SETTINGS)
    with pytest.raises(ValueError, match="owns clips"):
        OPT.optimize_velvet_noise_batch(local_signals=clips, total_clips=4, _bank_factory=_NoBank, **_SETTINGS)


def _runs_case():
    lib = N.lib()
    x = np.zeros((2, 16), np.float32)
    offs = np.array([0, 10, 10, 16], np.int64)  # clip 1 is empty
    prog = _family()([0.0, 0.5, 1.0], 16)
    out = np.zeros((4, N.OBJ_SLOTS), np.float64)

    def call(offs=offs, rows=16, stride=16, runs=((0, 2), (0, 1), (3, 2), (0, 2)), n_rows=4, n_clips=3):
        r = [np.ascontiguousarray(v, dtype=np.int32) for v in runs]
        ps = prog.host_struct()
        return lib.vnd_vn_objective_runs_dev(x.ctypes.data, rows, stride, offs.ctypes.data, n_clips, C.byref(ps), r[0].ctypes.data, r[1].ctypes.data,
                                             r[2].ctypes.data, r[3].ctypes.data, len(r[0]), out.ctypes.data, n_rows, None, 0, None)

    return lib, call


def test_runs_dev_rejects_bad_arguments_without_cuda():
    lib, call = _runs_case()

    def bad(match, **kw):
        assert call(**kw) == N.VND_EINVAL
        assert match in lib.vnd_last_error().decode(), lib.vnd_last_error()

    bad("not 0", offs=np.array([1, 10, 10, 16], np.int64))
    bad("decrease", offs=np.array([0, 10, 9, 16], np.int64))
    bad("not at rows", offs=np.array([0, 10, 10, 15], np.int64))
    bad("overlap", stride=15)
    bad("outside [0, 3)", runs=((0, 3), (0, 1), (3, 2), (0, 2)))
    bad("outside [0, 3)", runs=((-1,), (0,), (1,), (0,)))
    bad("empty signal", runs=((1,), (0,), (1,), (0,)))
    bad("outside the program", runs=((0, 2), (0, 2), (3, 2), (0, 2)))
    bad("outside the program", runs=((0,), (-1,), (1,), (0,)))
    bad("outside the 4 partial rows", runs=((0, 2), (0, 1), (3, 2), (0, 3)))
    bad("outside the 4 partial rows", runs=((0,), (0,), (1,), (-1,)), n_rows=4)
    bad("negative", runs=((0,), (0,), (-1,), (0,)))
    # n_runs == 0 launches nothing (and needs no device), and so does a run of no candidates, even on an empty clip
    assert call(runs=((), (), (), ()), n_rows=0) == N.VND_OK
    assert call(runs=((1,), (0,), (0,), (0,))) == N.VND_OK


def test_length_class_programs_are_the_single_clip_programs():
    """The one program of a call holds, for every run, the channels ``family(kappas, frames)`` builds for that clip alone:
    clips longer than the family's largest tap share the full program, each shorter length gets its own class,
    including clips shorter than the filter (where the vectorised packing gives way to table-by-table packing)."""
    family = _family()
    lengths = np.array([1, 900, 1439, 1440, 1441, 4000, 7000, 900])
    grid = np.linspace(0.0, 1.0, 9).tolist()
    assert T.kappa_family_program(grid, envelope=OPT.VelvetNoise(sample_rate_hz=_FS, seed=1).segment_envelope, frames=900,
                                  **{k: v for k, v in _SETTINGS.items()}) is None  # shorter than the filter: table by table
    last_tap = family(grid, OPT._NO_FRAME_LIMIT).halo - 1
    assert 1300 < last_tap < 1440  # read from the tables: jittered positions are rounded, below fir_length_samples

    def check(groups, base):
        prog, runs = OPT._run_program(family, lengths, groups, base)
        assert runs.shape == (4, len(groups))
        for (clip, ks, _, out), (c, cand, count, o) in zip(groups, runs.T):
            assert (c, count, o) == (clip, len(ks), out)
            want = family(ks, int(lengths[clip]))
            got = prog.slice_channels(int(cand), int(cand + count))
            assert np.array_equal(got.words, want.words) and np.array_equal(got.offsets, want.offsets), (clip, lengths[clip])
            assert prog.apply_gain == want.apply_gain
        return prog, runs

    # grid shaped: every clip on all grid strengths; clips of one length share their class
    prog, runs = check([(i, grid, 0, i * len(grid)) for i in range(len(lengths))], grid)
    assert runs[1][1] == runs[1][7] and runs[1][5] == runs[1][6] == 0
    n_classes = len({int(f) for f in lengths if f <= last_tap})
    assert prog.channels == len(grid) * (1 + n_classes)
    # Brent shaped: clip-major pairs, a few strengths per clip
    rng = np.random.default_rng(5)
    ks = rng.uniform(0.0, 1.0, 20).tolist()
    cuts = [0, 3, 4, 6, 9, 12, 15, 17, 20]
    groups = [(i, ks[a:b], a, a) for i, (a, b) in enumerate(zip(cuts[:-1], cuts[1:]))]
    prog, runs = check(groups, ks)
    long = [i for i in range(len(lengths)) if lengths[i] > last_tap]
    assert all(runs[1][i] == runs[3][i] for i in long)  # long clips: the run's channels are its pairs


# ------------------------------------------------------------------ CPU: world-2 gloo with an oracle-backed ragged bank

_LENGTHS = [1, 900, 1440, 4000, 7000]


class _OracleRaggedBank:
    """The clip bank's interface over ragged clips, scoring with the oracle."""

    lanes = 1

    def __init__(self, clips, family, kw):
        self.clips = [np.ascontiguousarray(np.asarray(c)) for c in clips]
        self.n, self.device = len(self.clips), None
        self.evaluations = self.launches = 0

    def _scores(self, c, ks):
        self.evaluations += len(ks)
        return np.asarray(O.vn_grid_scores(self.clips[c], list(ks), **_SETTINGS), dtype=np.float32)

    def grid_scores(self, kappas):
        self.launches += 1
        return np.stack([self._scores(c, kappas) for c in range(self.n)])

    def submit(self, clip_ids, kappas):
        self.launches += 1
        kappas = np.asarray(kappas)
        return np.concatenate([self._scores(c, kappas[clip_ids == c]) for c in np.unique(clip_ids)])

    def collect(self, handle):
        return handle


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
        ks, info = OPT.optimize_velvet_noise_batch(input_signals=_ragged_clips(), grid_size=_GRID, details=True, _bank_factory=_OracleRaggedBank,
                                                   **_SETTINGS)
        np.save(os.path.join(result_dir, f"kappa_{rank}.npy"), ks)
        np.save(os.path.join(result_dir, f"scores_{rank}.npy"), info["scores"])
    finally:
        dist.destroy_process_group()


def test_optimize_velvet_noise_batch_ragged_world2_gloo(tmp_path):
    import torch.multiprocessing as mp

    world = 2
    mp.spawn(_gloo_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    clips = _ragged_clips()
    one, info = OPT.optimize_velvet_noise_batch(input_signals=clips, grid_size=_GRID, details=True, _bank_factory=_OracleRaggedBank, **_SETTINGS)
    kappas = np.linspace(0.0, 1.0, _GRID)
    want = []
    for c in clips:  # the reference's procedure, clip by clip, one scipy minimiser at a time (oracle/vnd_oracle.py::refine)
        row = np.asarray(O.vn_grid_scores(c, kappas, **_SETTINGS), dtype=np.float32)
        minima = OPT.get_local_minima(row, _GRID)
        fn = lambda k, c=c: O.vn_grid_scores(c, [k], **_SETTINGS)[0]  # noqa: E731
        want.append(O.refine(minima, kappas, fn))
    want = np.asarray(want, dtype=np.float64)
    assert one.dtype == np.float64 and np.array_equal(one, want)
    assert info["launches_local"] == 1 + info["rounds_local"]
    for r in range(world):
        assert np.array_equal(np.load(os.path.join(str(tmp_path), f"kappa_{r}.npy")), want)
        assert np.array_equal(np.load(os.path.join(str(tmp_path), f"scores_{r}.npy")), info["scores"])


# ------------------------------------------------------------------ GPU: the run kernel against the single-clip kernel


_BIT_LENGTHS = [1, 7, 1439, 1440, 1441, 4095, 4096, 4097, 3 * 4096 + 5, 50000, 1_440_000]


def _clip_set():
    clips = [O.coloured_clip(i, n) for i, n in enumerate(_BIT_LENGTHS)]
    for name, a, n in (("viola", 10000, 30000), ("guitar", 5000, 8193), ("vocal", 20000, 1000)):
        clips.append(np.ascontiguousarray(G.wav(name)[1][a: a + n, :2], dtype=np.float32))
    return clips


def _pack_between_loud_neighbours(clips):
    """Channel-planar packing with a loud block (amplitude 1e3) before, between and after the clips: a read past a
    clip's end would pick it up."""
    rng = np.random.default_rng(9)
    parts, offs, at = [], [], 0
    for c in clips:
        loud = (rng.standard_normal((2, 4099)) * 1e3).astype(np.float32)
        parts += [loud, np.ascontiguousarray(c.T)]
        offs.append(at + loud.shape[1])
        at += loud.shape[1] + c.shape[0]
    parts.append((rng.standard_normal((2, 4099)) * 1e3).astype(np.float32))
    x = np.ascontiguousarray(np.concatenate(parts, axis=1))
    return x, np.asarray(offs, np.int64)


@gpu
def test_run_partials_equal_the_single_clip_kernel_bit_for_bit():
    import torch

    family = _family()
    clips = _clip_set()
    lengths = np.array([c.shape[0] for c in clips])
    x, starts = _pack_between_loud_neighbours(clips)
    # the loud blocks are clips of their own that no run names: offsets over the whole packing
    bounds = np.concatenate([[0], np.ravel(np.column_stack((starts, starts + lengths))), [x.shape[1]]])
    clip_of = 2 * np.arange(len(clips)) + 1
    grid = np.linspace(0.0, 1.0, 16).tolist()
    rng = np.random.default_rng(4)
    ks = rng.uniform(0.0, 1.0, 40).tolist()
    cuts = np.sort(rng.choice(np.arange(1, 40), len(clips) - 1, replace=False))
    cuts = [0, *cuts.tolist(), 40]
    cases = {
        "grid": ([(i, grid, 0, i * len(grid)) for i in range(len(clips))], grid),
        "brent": ([(i, ks[a:b], a, a) for i, (a, b) in enumerate(zip(cuts[:-1], cuts[1:]))], ks),
    }
    xt = torch.from_numpy(x).cuda()
    for name, (groups, base) in cases.items():
        prog, runs = OPT._run_program(family, lengths, groups, base)
        order = rng.permutation(runs.shape[1])  # runs in any order
        runs = runs[:, order]
        groups = [groups[i] for i in order]
        twice = runs[:, :1].copy()  # a clip in two runs: again into rows behind the others
        twice[3] = int((runs[3] + runs[2]).max())
        runs = np.concatenate([runs, twice], axis=1)
        groups = groups + [groups[0]]
        table = runs.copy()
        table[0] = clip_of[runs[0]]
        got = OPT.vn_objective_run_partials(xt, bounds, prog, table).cpu().numpy()
        host = OPT.vn_objective_run_partials(x, bounds, prog, table)
        assert np.array_equal(got, host), name
        for (clip, kk, _, _), (_, _, count, out) in zip(groups, runs.T):
            want = OPT.vn_objective_partials(clips[clip][None].transpose(0, 2, 1).copy(), family(kk, int(lengths[clip])))[0]
            assert np.array_equal(got[out: out + count], want), (name, clip, int(lengths[clip]))


@gpu
def test_run_partials_reject_bad_tables_before_any_launch():
    import torch

    family = _family()
    x = np.ones((2, 300), np.float32)
    prog = family([0.0, 1.0], 300)
    before = N.launch_count()
    for xx in (x, torch.from_numpy(x).cuda()):
        for offs, runs, match in (([0, 100, 300], [[2], [0], [2], [0]], "outside [0, 2)"),
                                  ([0, 200, 100], [[0], [0], [2], [0]], "decrease"),
                                  ([0, 0, 300], [[0], [0], [2], [0]], "empty signal"),
                                  ([0, 100, 300], [[1], [1], [2], [0]], "outside the program")):
            with pytest.raises(N.VndError, match=re.escape(match)) as e:
                OPT.vn_objective_run_partials(xx, offs, prog, runs)
            assert e.value.status == N.VND_EINVAL
    assert N.launch_count() == before


# ------------------------------------------------------------------ GPU: the optimiser against the single-clip optimiser


def _single(clip, grid):
    return float(OPT.optimize_velvet_noise(input_signal=clip, grid_size=grid, **_SETTINGS))


def _mixed_clips():
    rng = np.random.default_rng(12)
    clips = [O.coloured_clip(0, 30000), O.coloured_clip(1, 700)[:, 0].copy(), O.coloured_clip(2, 1440),
             (O.coloured_clip(3, 9000) * 20000).astype(np.int16), O.coloured_clip(4, 5000).astype(np.float64),
             np.column_stack((O.coloured_clip(5, 12000), rng.standard_normal(12000).astype(np.float32))), O.coloured_clip(6, 1)]
    return clips


@gpu
def test_ragged_numpy_list_equals_the_single_clip_optimiser():
    clips = _mixed_clips()
    got, info = OPT.optimize_velvet_noise_batch(input_signals=clips, grid_size=32, details=True, **_SETTINGS)
    assert got.dtype == np.float64 and got.shape == (len(clips),)
    assert set(info) >= {"scores", "local_minima", "argmin", "evaluations_local", "launches_local", "rounds_local", "clips_local"}
    for i, c in enumerate(clips):
        assert float(got[i]) == _single(c, 32), f"clip {i}"


@gpu
def test_ragged_cuda_list_equals_the_single_clip_optimiser():
    import torch

    clips = _mixed_clips()
    tensors = [torch.from_numpy(np.ascontiguousarray(c)).cuda() for c in clips]
    got = OPT.optimize_velvet_noise_batch(input_signals=tensors, grid_size=32, **_SETTINGS)
    for i, t in enumerate(tensors):
        assert float(got[i]) == _single(t.cpu().numpy(), 32), f"clip {i}"


@gpu
def test_equal_lengths_list_planar_array_and_planar_tensor_agree():
    import torch

    clips = [O.coloured_clip(i, 24000) for i in range(4)]
    got = OPT.optimize_velvet_noise_batch(input_signals=clips, grid_size=32, **_SETTINGS)
    for i, c in enumerate(clips):
        assert float(got[i]) == _single(c, 32), f"clip {i}"
    planar = np.stack([c.T for c in clips])
    assert np.array_equal(OPT.optimize_velvet_noise_batch(input_signals=planar, grid_size=32, **_SETTINGS), got)
    block = torch.from_numpy(planar).cuda()
    assert np.array_equal(OPT.optimize_velvet_noise_batch(input_signals=block, grid_size=32, **_SETTINGS), got)
    assert np.array_equal(OPT.optimize_velvet_noise_batch(local_signals=block, total_clips=4, grid_size=32, **_SETTINGS), got)


class _CountingBank(OPT._ClipBank):
    submits = 0

    def submit(self, clip_ids, kappas):
        type(self).submits += 1
        return super().submit(clip_ids, kappas)


@gpu
def test_one_call_and_two_kernels_per_stage_whatever_the_clip_count():
    rng = np.random.default_rng(8)
    for n in (3, 300):
        clips = [O.coloured_clip(i, int(rng.integers(500, 6000))) for i in range(n)]
        _CountingBank.submits = 0
        before = N.launch_count()
        _, info = OPT.optimize_velvet_noise_batch(input_signals=clips, grid_size=16, details=True, _bank_factory=_CountingBank, **_SETTINGS)
        launches = N.launch_count() - before
        assert info["launches_local"] == 1 + _CountingBank.submits, n
        assert launches == 2 * info["launches_local"], (n, launches, info["launches_local"])


@gpu
def test_optimised_strengths_feed_decorrelate_batch():
    from vndecorrelate_b200.decorrelation import VelvetNoise, decorrelate_batch

    clips = [O.coloured_clip(i, n) for i, n in enumerate([24000, 900, 31000, 5000, 1441])]
    kappas = OPT.optimize_velvet_noise_batch(input_signals=clips, grid_size=16, **_SETTINGS)
    decs = [VelvetNoise(sample_rate_hz=_FS, duration_seconds=_DUR, num_impulses=_NIMP, seed=1, log_distribution_strength=float(k)) for k in kappas]
    ys = decorrelate_batch(clips, decs)
    for c, y in zip(clips, ys):
        k = OPT.optimize_velvet_noise(input_signal=c, grid_size=16, **_SETTINGS)
        want = VelvetNoise(sample_rate_hz=_FS, duration_seconds=_DUR, num_impulses=_NIMP, seed=1, log_distribution_strength=k).decorrelate(c)
        assert G.same_bits(np.asarray(y), np.asarray(want))


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
        ks = OPT.optimize_velvet_noise_batch(input_signals=_mixed_clips(), grid_size=32, **_SETTINGS)
        np.save(os.path.join(result_dir, f"kappa_{rank}.npy"), ks)
    finally:
        dist.destroy_process_group()


@gpu
def test_world2_nccl_equals_world1(tmp_path):
    import torch
    import torch.multiprocessing as mp

    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    mp.spawn(_nccl_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    one = OPT.optimize_velvet_noise_batch(input_signals=_mixed_clips(), grid_size=32, **_SETTINGS)
    for r in range(2):
        assert np.array_equal(np.load(os.path.join(str(tmp_path), f"kappa_{r}.npy")), one)
