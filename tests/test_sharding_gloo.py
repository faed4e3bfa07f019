"""world_size-2 tests of the multi-GPU partitioning on CPU (gloo).  The scoring function is the
oracle (tests may use it); what is under test is the partition, the tap-table slicing and the
all-gather, which are the same code the NCCL path runs."""

from __future__ import annotations

import os
import socket

import numpy as np
import pytest

from oracle import vnd_oracle as O
from vndecorrelate_b200 import sharding as S
from vndecorrelate_b200 import taps as T


def test_block_range_covers_everything():
    for total in (0, 1, 7, 64, 4096):
        for world in (1, 2, 3, 8):
            spans = [S.block_range(total, r, world) for r in range(world)]
            assert spans[0][0] == 0 and spans[-1][1] == total
            assert all(a[1] == b[0] for a, b in zip(spans, spans[1:]))
            sizes = [b - a for a, b in spans]
            assert max(sizes) - min(sizes) <= 1
    with pytest.raises(ValueError):
        S.block_range(4, 2, 2)


def test_shard_program_slices_one_table():
    table = T.generate_tap_table(sample_rate_hz=48000, duration_seconds=0.03, num_impulses=30, num_outs=16, num_segments=4,
                                 log_distribution_strength=1.0, filtered_channels=tuple(range(16)), seed=1)
    prog = T.segmented_program(table, O.DEFAULT_ENVELOPE, 100000)
    parts = [S.shard_program(prog, r, 4) for r in range(4)]
    assert [(a, b) for _, a, b in parts] == [(0, 4), (4, 8), (8, 12), (12, 16)]
    assert np.array_equal(np.concatenate([p.words for p, _, _ in parts]), prog.words)
    for p, a, b in parts:
        assert p.channels == 4 and p.offsets[0] == 0 and p.offsets[-1] == p.words.size and p.halo == prog.halo


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _candidate_program(kappas, frames):
    tables = [T.generate_tap_table(sample_rate_hz=48000, duration_seconds=0.03, num_impulses=30, num_outs=2, num_segments=4,
                                   log_distribution_strength=k, filtered_channels=(0,), seed=1) for k in kappas]
    return T.candidate_program(tables, O.DEFAULT_ENVELOPE, frames)


def _oracle_score_fn(kappas_all):
    """Scores a (clips subset, program subset) pair with the oracle; the candidate subset is
    recognised by its position in the full program (tests only)."""
    full = _candidate_program(kappas_all, 6000)

    def fn(clips, prog):
        # locate the slice of candidates this sub-program holds
        start = 0
        for start in range(full.channels - prog.channels + 1):
            lo, hi = full.offsets[start], full.offsets[start + prog.channels]
            if hi - lo == prog.words.size and np.array_equal(full.words[lo:hi], prog.words):
                break
        ks = kappas_all[start : start + prog.channels]
        out = np.zeros((clips.shape[0], len(ks)), dtype=np.float32)
        for i, c in enumerate(clips):
            x = np.ascontiguousarray(c.T)
            out[i] = O.vn_grid_scores(x, ks, sample_rate_hz=48000, duration_seconds=0.03, num_impulses=30, seed=1)
        return out

    return fn


def _worker(rank, world, port, by, result_dir):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        kappas = np.linspace(0.0, 1.0, 6)
        clips = np.stack([O.coloured_clip(i, 6000).T for i in range(3)])  # identical on every rank
        prog = _candidate_program(kappas, 6000)
        scores = S.sweep_scores_sharded(clips, prog, _oracle_score_fn(kappas), by=by)
        np.save(os.path.join(result_dir, f"scores_{by}_{rank}.npy"), scores)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("by", ["clips", "candidates"])
def test_sweep_sharded_world2_gloo(tmp_path, by):
    import torch.multiprocessing as mp

    world = 2
    port = _free_port()
    mp.spawn(_worker, args=(world, port, by, str(tmp_path)), nprocs=world, join=True)
    kappas = np.linspace(0.0, 1.0, 6)
    clips = np.stack([O.coloured_clip(i, 6000).T for i in range(3)])
    want = _oracle_score_fn(kappas)(clips, _candidate_program(kappas, 6000))
    for r in range(world):
        got = np.load(os.path.join(str(tmp_path), f"scores_{by}_{r}.npy"))
        assert got.shape == (3, 6) and got.dtype == np.float32
        assert np.array_equal(got, want)  # every rank holds the full matrix
    argmins, minima = S.select_from_scores(want)
    assert len(argmins) == 3 and all(0 <= a < 6 for a in argmins) and all(len(m) >= 1 for m in minima)


# --------------------------------------------------------------------------------------------------------------
# optimize_velvet_noise_batch (BASELINE config 5): clips sharded, one all-gather of the score matrix, lock-step
# refinement per rank.  On CPU the clip bank is replaced by one that scores with the oracle; partition, collective,
# minima selection and the Brent bookkeeping are the code the NCCL path runs.
# --------------------------------------------------------------------------------------------------------------
_FS, _DUR, _NIMP, _GRID, _FRAMES = 48000, 0.03, 30, 24, 4000


class _OracleBank:
    """The clip bank's interface (one batch in flight), scoring with the oracle."""

    lanes = 1

    def __init__(self, clips, family, kw):
        self.clips = [np.ascontiguousarray(np.asarray(c)) for c in clips]
        self.n, self.frames, self.device = len(self.clips), self.clips[0].shape[0], None
        self.evaluations = self.launches = 0

    def _scores(self, c, ks):
        self.evaluations += len(ks)
        return np.asarray(O.vn_grid_scores(self.clips[c], list(ks), sample_rate_hz=_FS, duration_seconds=_DUR, num_impulses=_NIMP, seed=1),
                          dtype=np.float32)

    def grid_scores(self, kappas):
        return np.stack([self._scores(c, kappas) for c in range(self.n)])

    def submit(self, clip_ids, kappas):
        kappas = np.asarray(kappas)
        return np.concatenate([self._scores(c, kappas[clip_ids == c]) for c in np.unique(clip_ids)])

    def collect(self, handle):
        return handle


def _batch_clips():
    return [O.coloured_clip(i, _FRAMES) for i in range(5)]


def _batch_worker(rank, world, port, result_dir):
    import torch.distributed as dist

    from vndecorrelate_b200 import optimization as OPT

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        ks, info = OPT.optimize_velvet_noise_batch(input_signals=_batch_clips(), sample_rate_hz=_FS, duration_seconds=_DUR, num_impulses=_NIMP,
                                                   seed=1, grid_size=_GRID, details=True, _bank_factory=_OracleBank)
        np.save(os.path.join(result_dir, f"kappa_{rank}.npy"), ks)
        np.save(os.path.join(result_dir, f"scores_{rank}.npy"), info["scores"])
    finally:
        dist.destroy_process_group()


def test_optimize_velvet_noise_batch_world2_gloo(tmp_path):
    import torch.multiprocessing as mp

    from vndecorrelate_b200 import optimization as OPT

    world = 2
    mp.spawn(_batch_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    clips = _batch_clips()
    # single process, same code
    one, info = OPT.optimize_velvet_noise_batch(input_signals=clips, sample_rate_hz=_FS, duration_seconds=_DUR, num_impulses=_NIMP, seed=1,
                                                grid_size=_GRID, details=True, _bank_factory=_OracleBank)
    # the reference's procedure, clip by clip, one scipy minimiser at a time (oracle/vnd_oracle.py::refine)
    kappas = np.linspace(0.0, 1.0, _GRID)
    want = []
    for c in clips:
        row = np.asarray(O.vn_grid_scores(c, kappas, sample_rate_hz=_FS, duration_seconds=_DUR, num_impulses=_NIMP, seed=1), dtype=np.float32)
        minima = OPT.get_local_minima(row, _GRID)
        fn = lambda k, c=c: O.vn_grid_scores(c, [k], sample_rate_hz=_FS, duration_seconds=_DUR, num_impulses=_NIMP, seed=1)[0]  # noqa: E731
        want.append(O.refine(minima, kappas, fn))
    want = np.asarray(want, dtype=np.float64)
    assert one.dtype == np.float64 and np.array_equal(one, want)
    for r in range(world):
        assert np.array_equal(np.load(os.path.join(str(tmp_path), f"kappa_{r}.npy")), want)          # every rank: all clips, same bits
        assert np.array_equal(np.load(os.path.join(str(tmp_path), f"scores_{r}.npy")), info["scores"])  # and the full score matrix


class _OracleBankAsync(_OracleBank):
    """The same oracle-backed bank with two lanes, as the CUDA bank has, so that the refinement keeps two batches in
    flight on CPU."""

    lanes = 2


def test_refinement_with_two_batches_in_flight_equals_the_single_batch():
    """The refinement splits the rank's clips into two half-batches that are evaluated alternately (the host work of one
    runs under the kernels of the other on a GPU); a minimiser only sees its own values, so the result must not change."""
    from vndecorrelate_b200 import optimization as OPT

    clips = _batch_clips()
    kw = dict(input_signals=clips, sample_rate_hz=_FS, duration_seconds=_DUR, num_impulses=_NIMP, seed=1, grid_size=_GRID, details=True)
    one, info1 = OPT.optimize_velvet_noise_batch(_bank_factory=_OracleBank, **kw)
    two, info2 = OPT.optimize_velvet_noise_batch(_bank_factory=_OracleBankAsync, **kw)
    assert np.array_equal(one, two) and np.array_equal(info1["scores"], info2["scores"])
    assert info1["evaluations_local"] == info2["evaluations_local"]
