"""Stereo-image objective and parameter sweeps with the reference's API
(``src/vndecorrelate/optimization.py``), evaluated by batched CUDA kernels.

``grid_scan`` recognises the two candidate families the reference's optimisers build —
``VelvetNoise(filtered_channels=(0,), mode='LR', normalizer=None, log_distribution_strength=k)``
(optimization.py:260-272) and ``HaasEffect(delay_time_seconds=t, mode='LR')`` (:183-190) — and
scores ALL candidates of a family in one kernel launch: the clip is read once per tile and every
candidate is evaluated from shared memory.  Two wider families also score in one launch each, every score
equal to that candidate's own decorrelate-then-score result: velvet-noise candidates with two outputs and no
normaliser (any filtered channels, LR or MS, any width; ``vn_stereo_objective_partials``) and any ``HaasEffect``
(``haas_effect_objective_partials``); a mixed list is split into its families.  Any other decorrelator is run and
its output scored by the same kernels (one candidate).  The kernels return the sums the objective is made of; the scalar
combination below follows the reference's dtype chain (float32 for velvet-noise candidates, float64
for Haas candidates; SURVEY.md Appendix A.5).

Refinement is the bounded Brent minimiser scipy runs for the reference (``minimize_scalar(method="bounded")``),
restated in array form (``_BrentBatch``) so that every local minimum - of every clip - advances in lock-step
(``_refine_minima``): one kernel launch per Brent iteration over all live minimisers instead of one per evaluation.

``optimize_velvet_noise_batch`` runs the whole optimisation for MANY clips of any lengths (BASELINE config 5): clips
are partitioned over the ranks of ``torch.distributed`` (one process per GPU), the grid scores are all-gathered as one
float32 matrix (the only collective on the data path), and each rank refines the local minima of its own clips, with
one call of the run-list objective (``vn_objective_run_partials``) for the grid and one per batch of Brent steps.
``optimize_haas_delay_batch`` does the same for ``optimize_haas_delay`` on clips of any lengths: one launch of the Haas
objective over a flat (clip, delay) list for the whole grid, and one per Brent round over every live minimiser of every
clip of the rank.  Both run the same driver (``_optimize_batch``) over a clip bank of their objective.
"""

from __future__ import annotations

import ctypes as C
from typing import Any, Callable, Sequence

import numpy as np

from . import _native as N
from . import runtime as R
from .decorrelation import Decorrelator, HaasEffect, VelvetNoise, _batch_program, _is_mode
from .taps import IDENTITY_ENVELOPE, TapProgram, candidate_program, kappa_family_program
from .utils.dsp import EPSILON, LayoutMode, rms_normalize, to_float32

__all__ = [
    "symmetry_aware_objective", "grid_scan", "get_local_minima", "optimize_local_minima", "optimize_haas_delay",
    "optimize_velvet_noise", "optimize_velvet_noise_batch", "optimize_haas_delay_batch", "vn_objective_partials", "haas_objective_partials",
    "haas_objective_pair_partials", "vn_objective_run_partials", "vn_scores_from_partials", "haas_scores_from_partials",
    "vn_stereo_objective_partials", "vn_stereo_rms_objective_partials", "haas_effect_objective_partials",
]

_F32_HALF_PI = np.float32(np.pi / 2)
_F32_PI = np.float32(np.pi)


# ------------------------------------------------------------------------------------------------
# kernel calls
# ------------------------------------------------------------------------------------------------


def _planar_clips(clips, dtype=np.float32):
    """``(n_clips, 2, frames)`` contiguous array from a ``(frames, 2)`` signal, a list of such, or an
    already planar 3-D array."""
    if isinstance(clips, np.ndarray) and clips.ndim == 3:
        return np.ascontiguousarray(clips, dtype=dtype)
    if isinstance(clips, np.ndarray) and clips.ndim == 2:
        clips = [clips]
    if isinstance(clips, np.ndarray) and clips.ndim == 1:
        clips = [np.column_stack((clips, clips))]
    frames = clips[0].shape[0]
    out = np.empty((len(clips), 2, frames), dtype=dtype)
    for i, c in enumerate(clips):
        c = np.asarray(c)
        if c.ndim == 1:
            c = np.column_stack((c, c))
        if c.shape != (frames, 2):
            raise ValueError(f"all clips must be (frames, 2) with the same length, got {c.shape}")
        out[i] = c.T
    return out


def vn_objective_partials(clips, program: TapProgram):
    """Per (clip, candidate) partial sums of the objective for velvet-noise candidates.

    ``clips``: float32 ``(n_clips, 2, frames)`` numpy array or CUDA tensor (planar stereo).
    Returns float64 ``(n_clips, n_candidates, 12)`` (layout in ``include/vnd_b200.h``)."""
    lib = N.lib()
    if R.is_torch_tensor(clips):
        import torch

        if not clips.is_cuda or clips.dtype != torch.float32 or clips.dim() != 3 or clips.shape[1] != 2:
            raise ValueError("clips must be a CUDA float32 tensor of shape (n_clips, 2, frames)")
        clips = clips.contiguous()
        n_clips, _, frames = clips.shape
        out = torch.empty((n_clips, program.channels, N.OBJ_SLOTS), dtype=torch.float64, device=clips.device)
        nbytes = C.c_size_t()
        with torch.cuda.device(clips.device):
            N.check(lib.vnd_objective_workspace(frames, n_clips, program.channels, C.byref(nbytes)), "vnd_objective_workspace")
            work = torch.empty(nbytes.value, dtype=torch.uint8, device=clips.device)
            ps = R.device_program(program, clips.device)
            N.check(lib.vnd_vn_objective_batch_dev(clips.data_ptr(), frames, n_clips, 2 * frames, frames, C.byref(ps), out.data_ptr(),
                                                   work.data_ptr(), nbytes.value, R.torch_stream_ptr(clips)), "vnd_vn_objective_batch_dev")
        return out
    clips = _planar_clips(clips)
    n_clips, _, frames = clips.shape
    out = np.empty((n_clips, program.channels, N.OBJ_SLOTS), dtype=np.float64)
    ps = program.host_struct()
    N.check(lib.vnd_vn_objective_batch_host(R.HostContext.get().handle, clips.ctypes.data, frames, n_clips, 2 * frames, frames, C.byref(ps),
                                            out.ctypes.data), "vnd_vn_objective_batch_host")
    return out


def haas_objective_partials(clips, delays: Sequence[int]):
    """Per (clip, delay) partial sums for LR Haas candidates delaying channel 0 (float64
    arithmetic).  ``clips``: float32 or float64 ``(n_clips, 2, frames)``.  Returns float64
    ``(n_clips, n_delays, 8)``."""
    lib = N.lib()
    delays = np.ascontiguousarray(delays, dtype=np.int32)
    if R.is_torch_tensor(clips):
        import torch

        if not clips.is_cuda or clips.dtype not in (torch.float32, torch.float64) or clips.dim() != 3 or clips.shape[1] != 2:
            raise ValueError("clips must be a CUDA float32/float64 tensor of shape (n_clips, 2, frames)")
        clips = clips.contiguous()
        n_clips, _, frames = clips.shape
        out = torch.empty((n_clips, len(delays), N.HAAS_SLOTS), dtype=torch.float64, device=clips.device)
        with torch.cuda.device(clips.device):
            d = torch.from_numpy(delays).to(clips.device)
            N.check(lib.vnd_haas_objective_batch_dev(clips.data_ptr(), N.VND_F64 if clips.dtype == torch.float64 else N.VND_F32, frames, n_clips,
                                                     2 * frames, frames, d.data_ptr(), len(delays), out.data_ptr(), None, 0,
                                                     R.torch_stream_ptr(clips)), "vnd_haas_objective_batch_dev")
        return out
    dt = np.float64 if (isinstance(clips, np.ndarray) and clips.dtype == np.float64) else np.float32
    clips = _planar_clips(clips, dt)
    n_clips, _, frames = clips.shape
    out = np.empty((n_clips, len(delays), N.HAAS_SLOTS), dtype=np.float64)
    N.check(lib.vnd_haas_objective_batch_host(R.HostContext.get().handle, clips.ctypes.data, N.VND_F64 if dt == np.float64 else N.VND_F32, frames,
                                              n_clips, 2 * frames, frames, delays.ctypes.data, len(delays), out.ctypes.data),
            "vnd_haas_objective_batch_host")
    return out


def haas_objective_pair_partials(x, frame_offsets, pair_clip, pair_delay):
    """Partial sums of the Haas objective for a flat list of (clip, delay) pairs over ragged clips, in one launch.

    ``x``: float32 ``(2, chan_stride)`` channel-planar clips (numpy array or CUDA tensor); clip ``i`` is columns
    ``frame_offsets[i]:frame_offsets[i + 1]``.  Pair ``p`` delays channel 0 of clip ``pair_clip[p]`` by ``pair_delay[p]``
    frames.  Returns float64 ``(n_pairs, 8)``, row ``p`` bit-equal to ``haas_objective_partials(clip, [d])[0, 0]`` of
    that clip cast to float32.  With a CUDA tensor the offsets and pairs may be numpy or CUDA tensors and the result is
    a CUDA tensor enqueued on torch's current stream (nothing is checked that would need the device's copy of the
    offsets); with numpy everything is checked on the host first."""
    lib = N.lib()
    if R.is_torch_tensor(x):
        import torch

        if not x.is_cuda or x.dtype != torch.float32 or x.dim() != 2 or x.shape[0] != 2 or x.stride(1) != 1:
            raise ValueError("x must be a CUDA float32 tensor of shape (2, chan_stride) with contiguous rows")
        dev = x.device
        # rows only bounds the stride check: taken from host offsets, else from x itself (reading a device tensor would wait)
        rows = x.shape[1] if R.is_torch_tensor(frame_offsets) else int(np.asarray(frame_offsets)[-1])
        offs = torch.as_tensor(frame_offsets, dtype=torch.int64, device=dev).contiguous()
        pc = torch.as_tensor(pair_clip, dtype=torch.int32, device=dev).contiguous()
        pd = torch.as_tensor(pair_delay, dtype=torch.int32, device=dev).contiguous()
        if pc.shape != pd.shape or pc.dim() != 1 or offs.dim() != 1 or offs.numel() == 0:
            raise ValueError("frame_offsets must be 1-D with n_clips + 1 entries; pair_clip and pair_delay 1-D and of one length")
        out = torch.empty((pc.shape[0], N.HAAS_SLOTS), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            N.check(lib.vnd_haas_objective_pairs_dev(x.data_ptr(), rows, x.stride(0), offs.data_ptr(), offs.shape[0] - 1, pc.data_ptr(), pd.data_ptr(),
                                                     pc.shape[0], out.data_ptr(), R.torch_stream_ptr(x)), "vnd_haas_objective_pairs_dev")
        return out
    x = np.asarray(x)
    if x.dtype != np.float32 or x.ndim != 2 or x.shape[0] != 2:
        raise ValueError("x must be a float32 array of shape (2, chan_stride)")
    x = np.ascontiguousarray(x)
    offs = np.ascontiguousarray(frame_offsets, dtype=np.int64)
    pc = np.ascontiguousarray(pair_clip, dtype=np.int32)
    pd = np.ascontiguousarray(pair_delay, dtype=np.int32)
    if pc.shape != pd.shape or pc.ndim != 1 or offs.ndim != 1 or offs.size == 0:
        raise ValueError("frame_offsets must be 1-D with n_clips + 1 entries; pair_clip and pair_delay 1-D and of one length")
    out = np.empty((pc.size, N.HAAS_SLOTS), dtype=np.float64)
    N.check(lib.vnd_haas_objective_pairs_host(R.HostContext.get().handle, x.ctypes.data, int(offs[-1]), x.shape[1], offs.ctypes.data, offs.size - 1,
                                              pc.ctypes.data, pd.ctypes.data, pc.size, out.ctypes.data), "vnd_haas_objective_pairs_host")
    return out


def vn_objective_run_partials(x, frame_offsets, program: TapProgram, runs):
    """Partial sums of the velvet-noise objective for a list of runs over ragged clips: one objective launch and one
    combine launch.

    ``x``: float32 ``(2, chan_stride)`` channel-planar clips (numpy array or CUDA tensor with contiguous rows); clip ``i``
    is columns ``frame_offsets[i]:frame_offsets[i + 1]``.  ``runs``: a ``(4, n_runs)`` integer array (or four sequences)
    of ``(clip, first channel, count, first output row)``: run ``r`` scores clip ``runs[0][r]`` on the ``runs[2][r]``
    consecutive channels of ``program`` that start at ``runs[1][r]``, into rows ``runs[3][r]`` on.  The channels a run
    uses must be packed for its clip's length.  Returns float64 ``(n_rows, 12)``, ``n_rows`` the end of the last output
    row; rows no run names are zero.  Each row is bit-equal to ``vn_objective_partials`` on that clip alone with that
    channel.  The offsets and runs are read on the host (they size the launch); with a CUDA tensor the result is a CUDA
    tensor enqueued on torch's current stream, with numpy everything is uploaded and downloaded inside the call."""
    lib = N.lib()
    offs = np.ascontiguousarray(frame_offsets.cpu().numpy() if R.is_torch_tensor(frame_offsets) else frame_offsets, dtype=np.int64)
    table = np.asarray(runs, dtype=np.int64)
    if table.size == 0:
        table = table.reshape(4, 0)
    if table.ndim != 2 or table.shape[0] != 4 or offs.ndim != 1 or offs.size == 0:
        raise ValueError("frame_offsets must be 1-D with n_clips + 1 entries and runs a (4, n_runs) integer array")
    if table.size and (table.min() < -2**31 or table.max() >= 2**31):
        raise ValueError("run entries must fit in int32")
    run_clip, run_cand, run_count, run_out = (np.ascontiguousarray(r, dtype=np.int32) for r in table)
    n_runs = table.shape[1]
    n_rows = max(0, int((table[3] + table[2]).max())) if n_runs else 0
    tables = (run_clip.ctypes.data, run_cand.ctypes.data, run_count.ctypes.data, run_out.ctypes.data, n_runs)
    if R.is_torch_tensor(x):
        import torch

        if not x.is_cuda or x.dtype != torch.float32 or x.dim() != 2 or x.shape[0] != 2 or x.stride(1) != 1:
            raise ValueError("x must be a CUDA float32 tensor of shape (2, chan_stride) with contiguous rows")
        dev = x.device
        out = torch.zeros((n_rows, N.OBJ_SLOTS), dtype=torch.float64, device=dev)
        nbytes = C.c_size_t()
        N.check(lib.vnd_vn_objective_runs_workspace(offs.ctypes.data, offs.size - 1, run_clip.ctypes.data, run_count.ctypes.data, n_runs,
                                                    C.byref(nbytes)), "vnd_vn_objective_runs_workspace")
        with torch.cuda.device(dev):
            work = torch.empty(max(nbytes.value, 1), dtype=torch.uint8, device=dev)
            ps = R.device_program(program, dev)
            N.check(lib.vnd_vn_objective_runs_dev(x.data_ptr(), int(offs[-1]), x.stride(0), offs.ctypes.data, offs.size - 1, C.byref(ps), *tables,
                                                  out.data_ptr(), n_rows, work.data_ptr(), nbytes.value, R.torch_stream_ptr(x)),
                    "vnd_vn_objective_runs_dev")
        return out
    x = np.asarray(x)
    if x.dtype != np.float32 or x.ndim != 2 or x.shape[0] != 2:
        raise ValueError("x must be a float32 array of shape (2, chan_stride)")
    x = np.ascontiguousarray(x)
    out = np.zeros((n_rows, N.OBJ_SLOTS), dtype=np.float64)
    ps = program.host_struct()
    N.check(lib.vnd_vn_objective_runs_host(R.HostContext.get().handle, x.ctypes.data, int(offs[-1]), x.shape[1], offs.ctypes.data, offs.size - 1,
                                           C.byref(ps), *tables, out.ctypes.data, n_rows), "vnd_vn_objective_runs_host")
    return out


def _planar_input(x):
    """A cast and checked input (``to_float32``: numpy array or CUDA tensor) as a float32 channel-planar ``(2, frames)``
    clip on the same side: a mono signal in both channels, a wider one cut to its first two."""
    if R.is_torch_tensor(x):
        import torch

        if not x.is_cuda:
            raise N.VndError(N.VND_EUNSUPPORTED, "objective", "CPU torch tensors are not supported (no CPU fallback); pass a CUDA tensor or a numpy array")
        return (torch.stack((x, x)) if x.dim() == 1 else x[:, :2].t()).contiguous()
    return np.ascontiguousarray(np.stack((x, x)) if x.ndim == 1 else x[:, :2].T)


def _cast_input(input_signal):
    """The input as ``decorrelate`` casts it."""
    return to_float32(input_signal if R.is_torch_tensor(input_signal) else np.asarray(input_signal))


def _vn_stereo_records(frames: int, decorrelators):
    """The program (candidate j: channels 2 j, 2 j + 1) and the settings records of a velvet-noise stereo call."""
    progs = [d.tap_program(frames) for d in decorrelators]
    if len({p.apply_gain for p in progs}) > 1:
        raise ValueError("the candidates of one call must agree on whether the segment envelope is the identity (1.0,)")
    cands = np.zeros(len(decorrelators), dtype=N.VN_STEREO_CAND_DTYPE)
    widths = [float(d.width) if d.width is not None else 0.0 for d in decorrelators]
    cands["ms_encode"] = [_is_mode(d.mode, LayoutMode.MS) for d in decorrelators]
    cands["use_width"] = [d.width is not None for d in decorrelators]
    cands["w_mid"] = [np.float32(1.0 - w) for w in widths]  # the float32 roundings of vnd_vn_decorrelate_dev
    cands["w_side"] = [np.float32(w) for w in widths]
    return _batch_program(progs), cands


def _vn_stereo_partials(x, xp, decorrelators):
    """``vn_stereo_objective_partials`` on an input already cast and checked, ``xp`` its ``_planar_input``."""
    lib = N.lib()
    frames = x.shape[0]
    prog, cands = _vn_stereo_records(frames, decorrelators)
    n = len(decorrelators)
    if R.is_torch_tensor(xp):
        import torch

        dev = xp.device
        out = torch.empty((n, N.OBJ_SLOTS), dtype=torch.float64, device=dev)
        nbytes = C.c_size_t()
        N.check(lib.vnd_vn_stereo_objective_workspace(frames, n, C.byref(nbytes)), "vnd_vn_stereo_objective_workspace")
        with torch.cuda.device(dev):
            work = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
            dc = torch.from_numpy(cands.view(np.uint8)).to(dev)
            ps = R.device_program(prog, dev)
            N.check(lib.vnd_vn_stereo_objective_dev(xp.data_ptr(), frames, xp.stride(0), C.byref(ps), dc.data_ptr(), n, out.data_ptr(), work.data_ptr(),
                                                    nbytes.value, R.torch_stream_ptr(xp)), "vnd_vn_stereo_objective_dev")
        return out
    out = np.empty((n, N.OBJ_SLOTS), dtype=np.float64)
    ps = prog.host_struct()
    N.check(lib.vnd_vn_stereo_objective_host(R.HostContext.get().handle, xp.ctypes.data, frames, xp.shape[1], C.byref(ps), cands.ctypes.data, n,
                                             out.ctypes.data), "vnd_vn_stereo_objective_host")
    return out


def _vn_stereo_rms_partials(x, xp, decorrelators):
    """``vn_stereo_rms_objective_partials`` on an input already cast and checked, ``xp`` its ``_planar_input``."""
    frames = x.shape[0]
    prog, cands = _vn_stereo_records(frames, decorrelators)
    lib = N.lib()
    n = len(decorrelators)
    if R.is_torch_tensor(xp):
        import torch

        dev = xp.device
        out = torch.empty((n, N.OBJ_SLOTS), dtype=torch.float64, device=dev)
        gains = torch.empty((n, 2), dtype=torch.float32, device=dev)
        nbytes = C.c_size_t()
        N.check(lib.vnd_vn_stereo_rms_objective_workspace(frames, n, C.byref(nbytes)), "vnd_vn_stereo_rms_objective_workspace")
        with torch.cuda.device(dev):
            work = torch.empty(nbytes.value, dtype=torch.uint8, device=dev)
            dc = torch.from_numpy(cands.view(np.uint8)).to(dev)
            ps = R.device_program(prog, dev)
            N.check(lib.vnd_vn_stereo_rms_objective_dev(xp.data_ptr(), frames, xp.stride(0), C.byref(ps), dc.data_ptr(), n, gains.data_ptr(),
                                                        out.data_ptr(), work.data_ptr(), nbytes.value, R.torch_stream_ptr(xp)),
                    "vnd_vn_stereo_rms_objective_dev")
        return out, gains
    out = np.empty((n, N.OBJ_SLOTS), dtype=np.float64)
    gains = np.empty((n, 2), dtype=np.float32)
    ps = prog.host_struct()
    N.check(lib.vnd_vn_stereo_rms_objective_host(R.HostContext.get().handle, xp.ctypes.data, frames, xp.shape[1], C.byref(ps), cands.ctypes.data, n,
                                                 gains.ctypes.data, out.ctypes.data), "vnd_vn_stereo_rms_objective_host")
    return out, gains


def _sums_follow_frames(x) -> bool:
    """Whether ``decorrelate`` sums the squares of the cast input ``x`` frame by frame, as numpy's axis-0 reduction of a
    C-order array does and as the rms family's kernel does.  A channel-planar 2-D input of more than one frame (a
    Fortran-order array, a transposed tensor) is summed column by column in numpy's pairwise order instead; any other
    numpy layout is copied to C order first."""
    if x.ndim != 2 or x.shape[0] <= 1:
        return True
    if R.is_torch_tensor(x):
        return not (x.stride(0) == 1 and x.stride(1) >= x.shape[0])
    return bool(x.flags.c_contiguous) or not x.T.flags.c_contiguous


def _haas_effect_partials(x, xp, haas_effects):
    """``haas_effect_objective_partials`` on an input already cast and checked, ``xp`` its ``_planar_input``."""
    lib = N.lib()
    n = len(haas_effects)
    frames = x.shape[0]
    table = np.zeros(n, dtype=N.HAAS_CLIP_DTYPE)
    table["delay"] = [h.delay_len_samples for h in haas_effects]
    table["delayed_channel"] = [h.delayed_channel % 2 for h in haas_effects]
    table["mode_ms"] = [_is_mode(h.mode, LayoutMode.MS) for h in haas_effects]
    table["mono"] = x.ndim == 1
    table["use_width"] = [h.width is not None for h in haas_effects]
    table["width"] = [float(h.width) if h.width is not None else 0.0 for h in haas_effects]
    if R.is_torch_tensor(xp):
        import torch

        dev = xp.device
        out = torch.empty((n, N.HAAS_SLOTS), dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            dc = torch.from_numpy(table.view(np.uint8)).to(dev)
            N.check(lib.vnd_haas_effect_objective_dev(xp.data_ptr(), frames, xp.stride(0), dc.data_ptr(), n, out.data_ptr(), R.torch_stream_ptr(xp)),
                    "vnd_haas_effect_objective_dev")
        return out
    out = np.empty((n, N.HAAS_SLOTS), dtype=np.float64)
    N.check(lib.vnd_haas_effect_objective_host(R.HostContext.get().handle, xp.ctypes.data, frames, xp.shape[1], table.ctypes.data, n, out.ctypes.data),
            "vnd_haas_effect_objective_host")
    return out


def vn_stereo_objective_partials(clip, decorrelators: Sequence[VelvetNoise]):
    """Partial sums of the objective of ``VelvetNoise`` candidates with two outputs and ``normalizer=None`` - any
    ``filtered_channels``, mode LR or MS, any ``width`` - on one clip: one objective launch and one combine launch for
    all of them, with each candidate's output computed in registers and never stored.

    ``clip``: the input signal as ``decorrelate`` takes it (numpy array or CUDA tensor, mono or ``(frames, >= 2)``, any
    dtype; cast with ``to_float32``).  The candidates may differ in taps, mode, filtered channels and width; they must
    agree on whether the segment envelope is the identity ``(1.0,)``.  Each candidate's input checks run first and raise
    what its ``decorrelate`` raises.  Returns float64 ``(n_candidates, 12)`` (the layout of ``vn_objective_partials``):
    numpy for numpy input, a CUDA tensor enqueued on torch's current stream for a CUDA tensor (nothing is downloaded).

    Bit contract: row ``j`` equals, bit for bit, the partials the objective computes from
    ``decorrelators[j].decorrelate(clip)`` (``vn_objective_partials`` of that output with the one-tap identity program),
    so ``vn_scores_from_partials`` gives the scores ``symmetry_aware_objective`` returns for each candidate alone.
    A filter whose halo does not fit the kernel's shared memory raises ``VndError`` with ``VND_EUNSUPPORTED``."""
    decorrelators = list(decorrelators)
    for d in decorrelators:
        if not _is_vn_stereo_candidate(d):
            raise ValueError("candidates must be VelvetNoise with num_outs=2, normalizer=None, mode LR or MS and filtered_channels in (0, 1)")
    x = _cast_input(clip)
    for d in decorrelators:
        d._check_input(x)
    return _vn_stereo_partials(x, _planar_input(x), decorrelators)


def vn_stereo_rms_objective_partials(clip, decorrelators: Sequence[VelvetNoise]):
    """Partial sums of the objective, and the gains, of ``VelvetNoise`` candidates with two outputs and the default
    normaliser ``rms_normalize`` - any ``filtered_channels``, mode LR or MS, any ``width`` - on one clip, in three
    launches for all of them: the exact sums of squares of every candidate's output and its two gains, the objective
    of the scaled outputs, and the combine.  No candidate's output is stored.

    ``clip``: the input signal as ``decorrelate`` takes it (numpy array or CUDA tensor, mono or ``(frames, 2)``, any
    dtype; cast with ``to_float32``), in a layout that ``decorrelate`` sums frame by frame: not channel-planar (a
    Fortran-order array or a transposed tensor of more than one frame), whose sums numpy takes in pairwise order.  The
    candidates must agree on whether the segment envelope is the identity ``(1.0,)``.  Each candidate's input checks run
    first and raise what its ``decorrelate`` raises.  Returns ``(partials, gains)``: float64 ``(n_candidates, 12)`` (the
    layout of ``vn_objective_partials``) and float32 ``(n_candidates, 2)``; numpy for numpy input, CUDA tensors enqueued
    on torch's current stream for a CUDA tensor (nothing is downloaded).

    Bit contract: ``gains[j]`` are the per-channel gains ``rms_normalize`` applies in ``decorrelators[j].decorrelate(clip)``
    and row ``j`` of ``partials`` equals, bit for bit, the partials of that output (``vn_objective_partials`` with the
    one-tap identity program), so ``vn_scores_from_partials`` gives the scores ``symmetry_aware_objective`` returns for
    each candidate alone.  A filter whose halo does not fit the kernels' shared memory raises ``VndError`` with
    ``VND_EUNSUPPORTED``."""
    decorrelators = list(decorrelators)
    for d in decorrelators:
        if not _is_vn_rms_candidate(d):
            raise ValueError("candidates must be VelvetNoise with num_outs=2, normalizer=rms_normalize, mode LR or MS and filtered_channels in (0, 1)")
    x = _cast_input(clip)
    for d in decorrelators:
        d._check_input(x)
    if not _sums_follow_frames(x):
        raise ValueError("a channel-planar input is summed in numpy's pairwise order, which this call does not reproduce; pass it in C order")
    return _vn_stereo_rms_partials(x, _planar_input(x), decorrelators)


def haas_effect_objective_partials(clip, haas_effects: Sequence[HaasEffect]):
    """Partial sums of the objective of ``HaasEffect`` candidates - delayed channel 0, 1, -1 or -2, mode LR or MS, any
    ``width`` - on one clip: one launch, one CTA per candidate, the clip read in place and no candidate's output stored.

    ``clip``: the input signal as ``HaasEffect.decorrelate`` takes it (numpy array or CUDA tensor, mono or
    ``(frames, 2)``, any dtype; cast with ``to_float32``).  Each candidate's input checks run first and raise what its
    ``decorrelate`` raises.  Returns float64 ``(n_candidates, 8)`` (the layout of ``haas_objective_partials``): numpy for
    numpy input, a CUDA tensor enqueued on torch's current stream for a CUDA tensor.

    Bit contract: row ``j`` equals, bit for bit, ``haas_objective_partials(z, [0])[0, 0]`` for the float64 output ``z`` of
    ``haas_effects[j].decorrelate(clip)``, so ``haas_scores_from_partials`` gives the scores ``symmetry_aware_objective``
    returns for each candidate alone."""
    haas_effects = list(haas_effects)
    for h in haas_effects:
        if not _is_haas_effect_candidate(h):
            raise ValueError("candidates must be HaasEffect with a delay in [0, 2**31)")
    x = _cast_input(clip)
    for h in haas_effects:
        h._check(x)
    return _haas_effect_partials(x, _planar_input(x), haas_effects)


# ------------------------------------------------------------------------------------------------
# scalar combination (optimization.py:71-105 and the helpers :11-43)
# ------------------------------------------------------------------------------------------------


def _max_abs_theta_f32(p: np.ndarray) -> np.float32:
    """max|theta| exactly as the reference's float32 pipeline rounds it, from the two tracked
    frames: a correctly rounded float32 arctan2 (via float64), then the fold of
    utils/dsp.py:405-410 in float32."""
    d_pos, s_pos, d_neg, s_neg = p[6], p[7], p[8], p[9]
    a = np.float32(np.arctan2(np.float64(d_pos), np.float64(s_pos)))
    best = a
    if d_neg > 0.0 or s_neg != 1.0:  # a frame with s < 0 was seen (the tracker starts at 0 / 1)
        t = np.float32(np.arctan2(np.float64(d_neg), -np.float64(s_neg)))
        if t > _F32_HALF_PI:
            t = np.float32(t - _F32_PI)
        best = max(best, np.float32(abs(t)))
    return np.float32(best)


def _max_abs_theta_rows(p: np.ndarray) -> np.ndarray:
    """``_max_abs_theta_f32`` for many rows (the array ``arctan2`` runs the same numpy loop as the scalar call; the
    CPU tests compare the two bit for bit)."""
    d_pos, s_pos, d_neg, s_neg = p[:, 6], p[:, 7], p[:, 8], p[:, 9]
    best = np.arctan2(d_pos, s_pos).astype(np.float32)
    seen = (d_neg > 0.0) | (s_neg != 1.0)  # a frame with s < 0 was seen (the tracker starts at 0 / 1)
    t = np.arctan2(d_neg, -s_neg).astype(np.float32)
    t = np.where(t > _F32_HALF_PI, (t - _F32_PI).astype(np.float32), t)
    cand = np.abs(t)
    return np.where(seen & (cand > best), cand, best).astype(np.float32)  # Python's max(best, cand): cand only if greater


def _vn_score(p: np.ndarray, angle_limit, lambda_mean, lambda_skew, lambda_correlation, lambda_penalty) -> np.float32:
    denom = np.float32(np.float32(p[0]) + np.float32(EPSILON))  # radii.sum() + EPSILON, float32 (utils/dsp.py:418)
    spread = float(np.float32(p[2] / np.float64(denom)))  # optimization.py:19-21
    cen = float(np.float32(p[1] / np.float64(denom)))  # :24-26
    m3 = float(np.float32(p[3] / np.float64(denom)))
    skew = m3 / (max(spread, EPSILON) ** 1.5)  # :29-38
    nl = np.float32(np.float32(np.sqrt(p[5])) + np.float32(EPSILON))  # :11-16, both channels over ||L||
    corr = np.float32(p[4] / (np.float64(nl) * np.float64(nl)))
    exceed = max(0.0, float(np.float32(_max_abs_theta_f32(p) - np.float32(angle_limit))))  # :41-43
    mean_theta_penalty = lambda_mean * cen**2
    skewness_penalty = lambda_skew * skew**2
    lr_correlation_penalty = lambda_correlation * corr**2  # np.float32
    constraint_penalty = lambda_penalty * exceed**2
    objective = spread - mean_theta_penalty - skewness_penalty - lr_correlation_penalty - constraint_penalty
    return -objective  # np.float32, like the reference for float32 decorrelator output


def _haas_score(p: np.ndarray, angle_limit, lambda_mean, lambda_skew, lambda_correlation, lambda_penalty) -> np.float64:
    denom = p[0] + EPSILON
    spread = float(p[2] / denom)
    cen = float(p[1] / denom)
    skew = float(p[3] / denom) / (max(spread, EPSILON) ** 1.5)
    nl = np.sqrt(p[6]) + EPSILON
    corr = np.float64(p[5] / (nl * nl))
    exceed = max(0.0, float(p[4] - angle_limit))
    objective = spread - lambda_mean * cen**2 - lambda_skew * skew**2 - lambda_correlation * corr**2 - lambda_penalty * exceed**2
    return np.float64(-objective)


def _vn_scores_rows(flat: np.ndarray, angle_limit, lambda_mean, lambda_skew, lambda_correlation, lambda_penalty) -> np.ndarray:
    """``_vn_score`` for many rows at once: the same operations in the same dtypes, element by element (IEEE basic
    operations give the same bits in an array as on scalars); every ``**`` stays the scalar call it is in the one-row
    chain, so that no vector math library can round them
    differently from the one-row chain.  ``tests/test_host_logic.py`` asserts bit equality with ``_vn_score``."""
    p = np.asarray(flat, dtype=np.float64)
    eps32 = np.float32(EPSILON)
    denom = (p[:, 0].astype(np.float32) + eps32).astype(np.float64)          # float32 sum, widened for the divisions
    spread = (p[:, 2] / denom).astype(np.float32).astype(np.float64)         # float(np.float32(...)) per row
    cen = (p[:, 1] / denom).astype(np.float32).astype(np.float64)
    m3 = (p[:, 3] / denom).astype(np.float32).astype(np.float64)
    skew = m3 / np.array([m ** 1.5 for m in np.maximum(spread, EPSILON).tolist()], dtype=np.float64)
    nl = (np.sqrt(p[:, 5]).astype(np.float32) + eps32).astype(np.float64)
    corr = (p[:, 4] / (nl * nl)).astype(np.float32)
    max_theta = _max_abs_theta_rows(p)
    exceed = np.maximum(0.0, (max_theta - np.float32(angle_limit)).astype(np.float64))
    # every power stays the scalar call of the one-row chain (float ** 2 is C pow, np.float32 ** 2 is powf: neither is
    # guaranteed to round like x * x, which is what an array power would compute)
    sq = lambda v: np.array([t ** 2 for t in v.tolist()], dtype=np.float64)  # noqa: E731  (Python floats)
    partial = spread - lambda_mean * sq(cen) - lambda_skew * sq(skew)       # Python-float arithmetic in the one-row chain
    corr2 = np.array([c ** 2 for c in corr], dtype=np.float32)               # np.float32 scalars
    lr_pen = (np.float32(lambda_correlation) * corr2).astype(np.float32)    # weak Python scalar times float32
    objective = partial.astype(np.float32) - lr_pen                          # float minus np.float32 -> np.float32
    objective = objective - (lambda_penalty * sq(exceed)).astype(np.float32)
    return -objective


def _haas_scores_rows(flat: np.ndarray, angle_limit, lambda_mean, lambda_skew, lambda_correlation, lambda_penalty) -> np.ndarray:
    """``_haas_score`` for many rows at once, as ``_vn_scores_rows`` does it for ``_vn_score``: the basic operations and
    ``np.sqrt`` element by element in float64, every ``**`` the scalar call of the one-row chain (Python-float ``** 1.5``
    and ``** 2``, ``np.float64 ** 2`` for the correlation), and Python's ``max`` as the selection it is.
    ``tests/test_haas_delay_batch.py`` asserts bit equality with ``_haas_score``."""
    p = np.asarray(flat, dtype=np.float64)
    denom = p[:, 0] + EPSILON
    spread = p[:, 2] / denom
    cen = p[:, 1] / denom
    m3 = p[:, 3] / denom
    floor = np.where(EPSILON > spread, EPSILON, spread)  # max(spread, EPSILON): spread unless EPSILON is greater
    skew = m3 / np.array([v ** 1.5 for v in floor.tolist()], dtype=np.float64)
    nl = np.sqrt(p[:, 6]) + EPSILON
    corr = p[:, 5] / (nl * nl)
    over = p[:, 4] - angle_limit
    exceed = np.where(over > 0.0, over, 0.0)  # max(0.0, over): over only if greater
    sq = lambda v: np.array([t ** 2 for t in v.tolist()], dtype=np.float64)  # noqa: E731  (Python floats)
    objective = spread - lambda_mean * sq(cen) - lambda_skew * sq(skew)
    objective = objective - lambda_correlation * np.array([c ** 2 for c in corr], dtype=np.float64)  # np.float64 scalars
    objective = objective - lambda_penalty * sq(exceed)
    return -objective


def vn_scores_from_partials(partials, **kw) -> np.ndarray:
    p = partials.cpu().numpy() if R.is_torch_tensor(partials) else np.asarray(partials)
    flat = p.reshape(-1, N.OBJ_SLOTS)
    if len(flat) == 0:
        return np.zeros(p.shape[:-1], dtype=np.float32)
    return _vn_scores_rows(flat, **kw).astype(np.float32).reshape(p.shape[:-1])


def haas_scores_from_partials(partials, **kw) -> np.ndarray:
    p = partials.cpu().numpy() if R.is_torch_tensor(partials) else np.asarray(partials)
    flat = p.reshape(-1, N.HAAS_SLOTS)
    if len(flat) == 0:
        return np.zeros(p.shape[:-1], dtype=np.float64)
    return _haas_scores_rows(flat, **kw).reshape(p.shape[:-1])


# ------------------------------------------------------------------------------------------------
# candidate recognition
# ------------------------------------------------------------------------------------------------


def _is_vn_candidate(d) -> bool:
    return (
        isinstance(d, VelvetNoise) and d.num_outs == 2 and d.width is None and d.normalizer is None
        and tuple(d.filtered_channels) == (0,) and _is_mode(d.mode, LayoutMode.LR)
    )


def _is_haas_candidate(d) -> bool:
    return isinstance(d, HaasEffect) and d.width is None and _is_mode(d.mode, LayoutMode.LR) and d.delayed_channel == 0


def _is_vn_stereo_candidate(d) -> bool:
    """A candidate ``vn_stereo_objective_partials`` scores (the reference's velvet-noise family is one of them)."""
    return (
        isinstance(d, VelvetNoise) and d.num_outs == 2 and d.normalizer is None and (_is_mode(d.mode, LayoutMode.LR) or _is_mode(d.mode, LayoutMode.MS))
        and set(d.filtered_channels) <= {0, 1} and len(set(d.filtered_channels)) == len(tuple(d.filtered_channels))
    )


def _is_vn_rms_candidate(d) -> bool:
    """A candidate ``vn_stereo_rms_objective_partials`` scores: a ``_is_vn_stereo_candidate`` but with the default
    normaliser (the identity check ``VelvetNoise._decorrelate`` makes)."""
    return (
        isinstance(d, VelvetNoise) and d.num_outs == 2 and d.normalizer is rms_normalize
        and (_is_mode(d.mode, LayoutMode.LR) or _is_mode(d.mode, LayoutMode.MS))
        and set(d.filtered_channels) <= {0, 1} and len(set(d.filtered_channels)) == len(tuple(d.filtered_channels))
    )


def _is_haas_effect_candidate(d) -> bool:
    """A candidate ``haas_effect_objective_partials`` scores: any HaasEffect whose delay a settings record holds (the
    per-candidate path reports any other delay itself)."""
    return isinstance(d, HaasEffect) and 0 <= d.delay_len_samples < 2**31


def _as_stereo_f32(input_signal):
    x = np.asarray(input_signal).astype(np.float32, copy=False)
    if x.ndim == 1:
        x = np.column_stack((x, x))
    if x.ndim != 2 or x.shape[1] < 2:
        raise ValueError(f"Input shape invalid: Expected shape (num samples, 2), but got shape {x.shape}.")
    return x[:, :2]


def _vn_family_program(decorrelators: Sequence[VelvetNoise], frames: int) -> TapProgram | None:
    env = decorrelators[0].segment_envelope
    if any(d.segment_envelope != env for d in decorrelators):
        return None
    return candidate_program([d.velvet_noise for d in decorrelators], env, frames)


_IDENTITY_PROGRAM_WORDS = np.array([1, 0, 1, np.float32(1.0).view(np.int32), 0], dtype=np.int32)  # one +1 tap at index 0


def _score_signal(y, kw) -> Any:
    """Objective of an already decorrelated stereo signal (generic decorrelators)."""
    y = y.detach().cpu().numpy() if R.is_torch_tensor(y) else np.asarray(y)
    if y.dtype == np.float32:
        prog = TapProgram(_IDENTITY_PROGRAM_WORDS, np.array([0, 5], dtype=np.int32), 1, N.ORDER_SEGMENTED, 0, 1, 5)
        return vn_scores_from_partials(vn_objective_partials(y[:, :2], prog), **kw)[0, 0]
    return haas_scores_from_partials(haas_objective_partials(y[:, :2].astype(np.float64, copy=False), [0]), **kw)[0, 0]


# ------------------------------------------------------------------------------------------------
# public API (optimization.py:46-310)
# ------------------------------------------------------------------------------------------------


def symmetry_aware_objective(input_signal, decorrelator: Decorrelator, *, angle_limit: float, lambda_mean: float, lambda_skew: float,
                             lambda_correlation: float, lambda_penalty: float):
    """Value to minimise: ``-(E_w[th^2] - l1*E_w[th]^2 - l2*skew^2 - l3*r^2 - lp*exceed^2)``
    for ``decorrelator`` applied to ``input_signal`` (optimization.py:46-105)."""
    kw = dict(angle_limit=angle_limit, lambda_mean=lambda_mean, lambda_skew=lambda_skew, lambda_correlation=lambda_correlation,
              lambda_penalty=lambda_penalty)
    return _scan(input_signal, [decorrelator], kw)[0]


def _scan(input_signal, decorrelators, kw) -> np.ndarray:
    if len(decorrelators) == 0:
        return np.array([])
    if len(input_signal) == 0:  # the reference takes max(|theta|) of the frames (optimization.py:41-43): numpy's own error
        raise ValueError("zero-size array to reduction operation maximum which has no identity")
    if all(_is_vn_candidate(d) for d in decorrelators):
        x = _as_stereo_f32(input_signal)
        prog = _vn_family_program(decorrelators, x.shape[0])
        if prog is not None:
            return vn_scores_from_partials(vn_objective_partials(x, prog), **kw)[0]
    if all(_is_haas_candidate(d) for d in decorrelators):
        x = _as_stereo_f32(input_signal)
        delays = [d.delay_len_samples for d in decorrelators]
        return haas_scores_from_partials(haas_objective_partials(x, delays), **kw)[0]
    return _scan_families(input_signal, decorrelators, kw)


# Fewest rms-normalised velvet-noise candidates of one envelope kind that take the family route.  Below it the loop is
# faster: the family's sums pass walks the whole clip once at about 13.5 ns a frame whatever the number of candidates
# (measured; not profiled further), while the loop costs 2.7 ns a frame and candidate on a CUDA
# tensor of 30 s, the cheapest case measured: about five candidates' worth (B200 at 1000 W; tools/bench_objective_rms.py,
# profiles/r11_objective_rms.json).  Both scale with the clip's length, so the threshold is a candidate count.
_RMS_FAMILY_MIN = 6


def _scan_families(input_signal, decorrelators, kw) -> np.ndarray:
    """Scores of any candidate list: the velvet-noise stereo candidates in one launch per envelope kind
    (``_vn_stereo_partials``), groups of at least ``_RMS_FAMILY_MIN`` rms-normalised ones in three launches per envelope
    kind (``_vn_stereo_rms_partials``), the Haas effects in one launch (``_haas_effect_partials``), every other candidate
    run and scored on its own (``_score_signal``); each score is the one that candidate alone gets, in list order.  Every
    grouped candidate's input check runs before any device work, so the first exception is the one the
    candidate-by-candidate loop raises."""
    vn = [i for i, d in enumerate(decorrelators) if _is_vn_stereo_candidate(d)]
    rms = [i for i, d in enumerate(decorrelators) if _is_vn_rms_candidate(d)]
    haas = [i for i, d in enumerate(decorrelators) if _is_haas_effect_candidate(d)]
    cpu_tensor = R.is_torch_tensor(input_signal) and not input_signal.is_cuda  # decorrelate raises its own error for it
    loop = lambda: np.array([_score_signal(d.decorrelate(input_signal), kw) for d in decorrelators])  # noqa: E731
    if (not vn and not haas and len(rms) < _RMS_FAMILY_MIN) or cpu_tensor:
        return loop()
    x = _cast_input(input_signal)
    rms_groups: dict = {}
    if len(rms) >= _RMS_FAMILY_MIN and _sums_follow_frames(x):
        for i in rms:
            rms_groups.setdefault(decorrelators[i].tap_program(x.shape[0]).apply_gain, []).append(i)
        rms_groups = {g: idx for g, idx in rms_groups.items() if len(idx) >= _RMS_FAMILY_MIN}
    if not vn and not haas and not rms_groups:
        return loop()
    grouped = set(vn) | set(haas) | {i for idx in rms_groups.values() for i in idx}
    others = [i for i in range(len(decorrelators)) if i not in grouped]
    for i, d in enumerate(decorrelators):
        if i not in grouped:
            continue
        try:
            d._check_input(x) if isinstance(d, VelvetNoise) else d._check(x)
        except Exception:
            for j in others:  # the loop would have run these first: any exception of theirs comes first
                if j < i:
                    decorrelators[j].decorrelate(input_signal)
            raise
    xp = _planar_input(x)
    scores: list = [None] * len(decorrelators)
    by_gain: dict = {}
    for i in vn:
        by_gain.setdefault(decorrelators[i].tap_program(x.shape[0]).apply_gain, []).append(i)
    families = [(idx, lambda c: _vn_stereo_partials(x, xp, c)) for idx in by_gain.values()]
    families += [(idx, lambda c: _vn_stereo_rms_partials(x, xp, c)[0]) for idx in rms_groups.values()]
    for idx, partials in families:
        try:
            s = vn_scores_from_partials(partials([decorrelators[i] for i in idx]), **kw)
        except N.VndError as e:
            if e.status != N.VND_EUNSUPPORTED:
                raise
            others.extend(idx)  # a halo beyond the kernels' shared memory: candidate by candidate
            continue
        for i, v in zip(idx, s):
            scores[i] = v
    if haas:
        for i, v in zip(haas, haas_scores_from_partials(_haas_effect_partials(x, xp, [decorrelators[i] for i in haas]), **kw)):
            scores[i] = v
    for i in sorted(others):
        scores[i] = _score_signal(decorrelators[i].decorrelate(input_signal), kw)
    return np.array(scores)


def grid_scan(input_signal, decorrelators: list[Decorrelator], **kwargs) -> np.ndarray:
    """Scores of all ``decorrelators`` on ``input_signal`` (optimization.py:108-117), one launch per
    candidate family."""
    print("Starting Grid Scan")
    return _scan(input_signal, list(decorrelators), kwargs)


def get_local_minima(scores, grid_size: int) -> list[int]:
    """Strict interior local minima, or ``[argmin]`` if there are none (optimization.py:120-128)."""
    local_minima = [i for i in range(1, grid_size - 1) if scores[i] < scores[i - 1] and scores[i] < scores[i + 1]]
    if not local_minima:
        return [int(np.argmin(scores))]
    return local_minima


def optimize_local_minima(local_minima: list[int], scalars, grid_size: int, scalar_objective: Callable[[float], float]):
    """Bounded Brent (``xatol=1e-4``) between the grid neighbours of each local minimum; the first
    strictly best result wins (optimization.py:131-155)."""
    from scipy.optimize import minimize_scalar

    best_scalar, best_score = 0.0, np.inf
    print("Starting Local Minima optimization")
    for i in local_minima:
        low = scalars[max(0, i - 1)]
        high = scalars[min(grid_size - 1, i + 1)]
        result = minimize_scalar(fun=scalar_objective, bounds=(low, high), method="bounded", options={"xatol": 1e-4})
        if result.fun < best_score:
            best_score = result.fun
            best_scalar = result.x
    return best_scalar


# ------------------------------------------------------------------------------------------------
# ``_BrentBatch`` below restates ``scipy.optimize._optimize._minimize_scalar_bounded`` statement for statement, in array
# form, which SURVEY.md section 8(f).1 asks for so that every comparison of the refinement comes out as in the reference.
# That routine is part of SciPy:
#
#   Copyright (c) 2001-2002 Enthought, Inc. 2003, SciPy Developers.  All rights reserved.
#
#   Redistribution and use in source and binary forms, with or without modification, are permitted provided that the
#   following conditions are met:
#   1. Redistributions of source code must retain the above copyright notice, this list of conditions and the following
#      disclaimer.
#   2. Redistributions in binary form must reproduce the above copyright notice, this list of conditions and the
#      following disclaimer in the documentation and/or other materials provided with the distribution.
#   3. Neither the name of the copyright holder nor the names of its contributors may be used to endorse or promote
#      products derived from this software without specific prior written permission.
#
#   THIS SOFTWARE IS PROVIDED BY THE COPYRIGHT HOLDERS AND CONTRIBUTORS "AS IS" AND ANY EXPRESS OR IMPLIED WARRANTIES,
#   INCLUDING, BUT NOT LIMITED TO, THE IMPLIED WARRANTIES OF MERCHANTABILITY AND FITNESS FOR A PARTICULAR PURPOSE ARE
#   DISCLAIMED. IN NO EVENT SHALL THE COPYRIGHT OWNER OR CONTRIBUTORS BE LIABLE FOR ANY DIRECT, INDIRECT, INCIDENTAL,
#   SPECIAL, EXEMPLARY, OR CONSEQUENTIAL DAMAGES (INCLUDING, BUT NOT LIMITED TO, PROCUREMENT OF SUBSTITUTE GOODS OR
#   SERVICES; LOSS OF USE, DATA, OR PROFITS; OR BUSINESS INTERRUPTION) HOWEVER CAUSED AND ON ANY THEORY OF LIABILITY,
#   WHETHER IN CONTRACT, STRICT LIABILITY, OR TORT (INCLUDING NEGLIGENCE OR OTHERWISE) ARISING IN ANY WAY OUT OF THE USE
#   OF THIS SOFTWARE, EVEN IF ADVISED OF THE POSSIBILITY OF SUCH DAMAGE.
#
# (BSD 3-Clause; the algorithm is Forsythe, Malcolm and Moler's ``fmin``.)
# ------------------------------------------------------------------------------------------------
class _BrentBatch:
    """Brent's bounded scalar minimiser - ``scipy.optimize.minimize_scalar(method="bounded")``, the reference's
    refinement step (optimization.py:144-149) - for MANY intervals at once, as array arithmetic: one state vector per
    variable of ``_minimize_scalar_bounded`` of the pinned scipy (1.16 in the reference's lock file, 1.18 here), every
    statement of its loop applied under a mask to the minimisers that take it.  ``pending`` hands out the abscissa each
    live minimiser wants evaluated and ``feed`` takes the values, so that all minimisers advance in lock-step.

    The element-wise operations (+, -, *, /, abs, sign, comparisons, maximum) are IEEE basic operations, identical in
    an array and on scalars, and the dtypes are the scalar code's: abscissae and step sizes float64, function values
    the objective's own dtype (float32 for velvet-noise candidates), so that ``(xf - nfc) * (fx - ffulc)`` is a float64
    product of a float64 and an exactly widened float32 difference, as under numpy's scalar promotion.  Every minimiser
    therefore sees the abscissae, takes the branches and returns the values of scipy's; ``tests/test_host_logic.py``
    compares them abscissa by abscissa on thousands of float32 and float64 objectives.  A Brent round over 20 000
    minimisers costs about a millisecond here."""

    def __init__(self, lows, highs, xatol: float, maxiter: int = 500):
        from math import sqrt

        a = np.asarray(lows, dtype=np.float64).copy()
        b = np.asarray(highs, dtype=np.float64).copy()
        if not (np.all(np.isfinite(a)) and np.all(np.isfinite(b))):
            raise ValueError("Optimization bounds must be finite scalars.")
        if np.any(a > b):
            raise ValueError("The lower bound exceeds the upper bound.")
        self.n = len(a)
        self.xatol, self.maxiter = xatol, maxiter
        self.sqrt_eps = sqrt(2.2e-16)
        self.golden_mean = 0.5 * (3.0 - sqrt(5.0))
        self.a, self.b = a, b
        self.fulc = a + self.golden_mean * (b - a)
        self.nfc = self.fulc.copy()
        self.xf = self.fulc.copy()
        self.rat = np.zeros(self.n)
        self.e = np.zeros(self.n)
        self.x = self.xf.copy()
        self.num = np.zeros(self.n, dtype=np.int64)
        self.flag = np.zeros(self.n, dtype=np.int64)
        self.live = np.ones(self.n, dtype=bool)
        self.started = False
        self.fx = self.ffulc = self.fnfc = self.fu = np.zeros(0)  # set by the first feed (an empty batch is never fed)

    def pending(self):
        """Indices of the live minimisers and the abscissa each wants evaluated."""
        idx = np.nonzero(self.live)[0]
        return idx, self.x[idx]

    def _propose(self, m):
        """The body of scipy's ``while`` loop up to the evaluation, for the minimisers in mask ``m`` (all of which
        passed the loop condition)."""
        a, b, xf, nfc, fulc, fx, ffulc, fnfc, xm, tol1, tol2 = (self.a, self.b, self.xf, self.nfc, self.fulc, self.fx, self.ffulc, self.fnfc, self.xm,
                                                                self.tol1, self.tol2)
        golden = m.copy()
        para = m & (np.abs(self.e) > tol1)
        if para.any():
            i = np.nonzero(para)[0]
            r = (xf[i] - nfc[i]) * (fx[i] - ffulc[i])
            q = (xf[i] - fulc[i]) * (fx[i] - fnfc[i])
            p = (xf[i] - fulc[i]) * q - (xf[i] - nfc[i]) * r
            q = 2.0 * (q - r)
            p = np.where(q > 0.0, -p, p)
            q = np.abs(q)
            r = self.e[i]
            self.e[i] = self.rat[i]
            ok = (np.abs(p) < np.abs(0.5 * q * r)) & (p > q * (a[i] - xf[i])) & (p < q * (b[i] - xf[i]))
            golden[i] = ~ok
            if ok.any():
                j = i[ok]
                with np.errstate(divide="ignore", invalid="ignore"):
                    rat = (p[ok] + 0.0) / q[ok]
                x = xf[j] + rat
                near = ((x - a[j]) < tol2[j]) | ((b[j] - x) < tol2[j])
                d = xm[j] - xf[j]
                si = np.sign(d) + (d == 0)
                self.rat[j] = np.where(near, tol1[j] * si, rat)
        if golden.any():
            i = np.nonzero(golden)[0]
            self.e[i] = np.where(xf[i] >= xm[i], a[i] - xf[i], b[i] - xf[i])
            self.rat[i] = self.golden_mean * self.e[i]
        i = np.nonzero(m)[0]
        si = np.sign(self.rat[i]) + (self.rat[i] == 0)
        self.x[i] = xf[i] + si * np.maximum(np.abs(self.rat[i]), tol1[i])

    def _close_or_propose(self, m):
        """Loop condition for the minimisers in ``m``: the converged ones finish, the others get their next abscissa."""
        go = m & (np.abs(self.xf - self.xm) > (self.tol2 - 0.5 * (self.b - self.a)))
        self.live[m & ~go] = False
        if go.any():
            self._propose(go)

    def feed(self, idx, values):
        """Function values (array in the objective's dtype) for the abscissae handed out by ``pending``."""
        values = np.asarray(values)
        if not self.started:  # the first evaluation of every minimiser (scipy evaluates before its loop)
            assert len(idx) == self.n
            self.started = True
            self.fx = values.copy()
            self.ffulc = values.copy()
            self.fnfc = values.copy()
            self.fu = np.full(self.n, np.inf, dtype=values.dtype)
            self.num[:] = 1
            self.xm = 0.5 * (self.a + self.b)
            self.tol1 = self.sqrt_eps * np.abs(self.xf) + self.xatol / 3.0
            self.tol2 = 2.0 * self.tol1
            self._close_or_propose(self.live.copy())
            return
        a, b, x, xf = self.a, self.b, self.x, self.xf
        fu = values
        self.fu[idx] = fu
        self.num[idx] += 1
        better = fu <= self.fx[idx]
        ib, iw = idx[better], idx[~better]
        if len(ib):  # fu <= fx
            right = x[ib] >= xf[ib]
            a[ib[right]] = xf[ib[right]]
            b[ib[~right]] = xf[ib[~right]]
            self.fulc[ib], self.ffulc[ib] = self.nfc[ib], self.fnfc[ib]
            self.nfc[ib], self.fnfc[ib] = xf[ib], self.fx[ib]
            self.xf[ib], self.fx[ib] = x[ib], fu[better]
        if len(iw):
            fw = fu[~better]
            left = x[iw] < xf[iw]
            a[iw[left]] = x[iw[left]]
            b[iw[~left]] = x[iw[~left]]
            c1 = (fw <= self.fnfc[iw]) | (self.nfc[iw] == xf[iw])
            c2 = ~c1 & ((fw <= self.ffulc[iw]) | (self.fulc[iw] == xf[iw]) | (self.fulc[iw] == self.nfc[iw]))
            i1, i2 = iw[c1], iw[c2]
            self.fulc[i1], self.ffulc[i1] = self.nfc[i1], self.fnfc[i1]
            self.nfc[i1], self.fnfc[i1] = x[i1], fw[c1]
            self.fulc[i2], self.ffulc[i2] = x[i2], fw[c2]
        self.xm[idx] = 0.5 * (a[idx] + b[idx])
        self.tol1[idx] = self.sqrt_eps * np.abs(self.xf[idx]) + self.xatol / 3.0
        self.tol2[idx] = 2.0 * self.tol1[idx]
        m = np.zeros(self.n, dtype=bool)
        m[idx] = True
        over = m & (self.num >= self.maxiter)
        self.flag[over] = 1
        self.live[over] = False
        self._close_or_propose(m & ~over)

    def results(self):
        """(x, fun, nfev, status) arrays, the fields of scipy's ``OptimizeResult``: ``fun`` in the objective's dtype,
        ``status`` 0 (converged), 1 (``maxiter`` evaluations) or 2 (a NaN)."""
        status = np.where(np.isnan(self.xf) | np.isnan(self.fx) | np.isnan(self.fu), 2, self.flag)
        return self.xf.copy(), self.fx.copy(), self.num.copy(), status


def _refine_minima(minima: Sequence[Sequence[int]], grid, submit: Callable[[np.ndarray, np.ndarray], Any],
                   collect: Callable[[Any], Any] = lambda handle: handle, lanes: int = 1) -> tuple[np.ndarray, int]:
    """``optimize_local_minima`` for many clips, every minimiser in lock-step: bounded Brent (``xatol=1e-4``) between
    the grid neighbours of each local minimum (``minima[c]``: the grid indices of clip ``c``'s minima), and per clip
    the first strictly best result (optimization.py:131-155).  Returns the float64 array of each clip's abscissa and the
    number of Brent rounds.

    ``submit(clip_ids, abscissae)`` starts the evaluation of a clip-major list of pairs and returns a handle;
    ``collect(handle)`` returns their values in the objective's dtype.  The clips run in ``lanes`` contiguous blocks,
    each with its own minimisers and one evaluation in flight, so that the host can advance one lane while the device
    evaluates another.  A minimiser only ever sees its own values, so the result does not depend on the lanes."""
    print("Starting Local Minima optimization")
    grid = np.asarray(grid, dtype=np.float64)
    n = len(minima)
    at = np.array([i for m in minima for i in m], dtype=np.int64)
    owner = np.repeat(np.arange(n), [len(m) for m in minima])
    lows, highs = grid[np.maximum(at - 1, 0)], grid[np.minimum(at + 1, len(grid) - 1)]
    cuts = np.searchsorted(owner, [h * n // lanes for h in range(lanes + 1)])  # lane h: clips [h n / lanes, (h + 1) n / lanes)
    members = [np.arange(a, b) for a, b in zip(cuts[:-1], cuts[1:])]
    engines = [_BrentBatch(lows[m], highs[m], 1e-4) for m in members]
    rounds = [0] * lanes

    def launch(h):
        idx, xs = engines[h].pending()
        if len(idx) == 0:
            return None
        rounds[h] += 1
        return idx, submit(owner[members[h][idx]], xs)

    handles = [launch(h) for h in range(lanes)]
    while any(handle is not None for handle in handles):
        for h in range(lanes):
            if handles[h] is not None:
                idx, handle = handles[h]
                engines[h].feed(idx, collect(handle))
                handles[h] = launch(h)
    best, best_score = np.zeros(n), [np.inf] * n
    for eng, m in zip(engines, members):
        xs, funs = eng.results()[:2]
        for x, fun, c in zip(xs, funs, owner[m]):  # first strictly best minimum of each clip (optimization.py:150-153)
            if fun < best_score[c]:
                best_score[c], best[c] = fun, x
    return best, max(rounds)


def _device_clip(x: np.ndarray):
    """The clip as a resident planar CUDA tensor (uploaded once per optimisation) when torch is there;
    otherwise the numpy array itself (the host entry points then upload it on every call)."""
    try:
        import torch

        if torch.cuda.is_available():
            return torch.from_numpy(np.ascontiguousarray(x.T)[None]).to(f"cuda:{R.default_device()}")
    except ImportError:
        pass
    return x


def optimize_haas_delay(*, input_signal, sample_rate_hz: int, max_delay_seconds: int, grid_size: int = 400, angle_limit: float = np.pi / 4,
                        lambda_mean: float = 5.0, lambda_skew: float = 2.0, lambda_correlation: float = 15.0, lambda_penalty: float = 1e3) -> float:
    """Optimised ``delay_time_seconds`` in ``[0, max_delay_seconds]`` (optimization.py:158-227)."""
    kw = dict(angle_limit=angle_limit, lambda_mean=lambda_mean, lambda_skew=lambda_skew, lambda_correlation=lambda_correlation,
              lambda_penalty=lambda_penalty)
    taus = np.linspace(0.0, max_delay_seconds, grid_size)
    candidates = [HaasEffect(sample_rate_hz=sample_rate_hz, delay_time_seconds=tau, mode="LR") for tau in taus]
    scores = grid_scan(input_signal, candidates, **kw)
    local_minima = get_local_minima(scores, grid_size)
    clip = _device_clip(_as_stereo_f32(input_signal))

    def batch(ts):
        delays = [HaasEffect(sample_rate_hz=sample_rate_hz, delay_time_seconds=t, mode="LR").delay_len_samples for t in ts]
        p = haas_objective_partials(clip, delays)
        p = p.cpu().numpy() if R.is_torch_tensor(p) else p
        return list(haas_scores_from_partials(p, **kw)[0])

    best, _ = _refine_minima([local_minima], taus, lambda _, ts: batch(ts.tolist()))
    return best[0]


def optimize_velvet_noise(*, input_signal, sample_rate_hz: int, duration_seconds: float, num_impulses: int, seed: int = 1, grid_size: int = 400,
                          angle_limit: float = np.pi / 4, lambda_mean: float = 5.0, lambda_skew: float = 2.0, lambda_correlation: float = 15.0,
                          lambda_penalty: float = 1e3) -> float:
    """Optimised ``log_distribution_strength`` in ``[0, 1]`` (optimization.py:230-310)."""
    kw = dict(angle_limit=angle_limit, lambda_mean=lambda_mean, lambda_skew=lambda_skew, lambda_correlation=lambda_correlation,
              lambda_penalty=lambda_penalty)

    def candidate(kappa):
        return VelvetNoise(sample_rate_hz=sample_rate_hz, duration_seconds=duration_seconds, num_impulses=num_impulses,
                           log_distribution_strength=kappa, normalizer=None, filtered_channels=(0,), mode="LR", seed=seed)

    kappas = np.linspace(0.0, 1.0, grid_size)
    x = _as_stereo_f32(input_signal)
    clip = _device_clip(x)
    envelope = candidate(0.0).segment_envelope

    def family_program(ks):
        """The candidates of the sweep differ only in the strength and share their random draws: their tap
        programs are packed in one vectorised pass (taps.kappa_family_program), table by table only when
        that shortcut does not apply."""
        prog = kappa_family_program(ks, sample_rate_hz=sample_rate_hz, duration_seconds=duration_seconds, num_impulses=num_impulses,
                                    envelope=envelope, seed=seed, frames=x.shape[0]) if seed is not None else None
        return prog if prog is not None else _vn_family_program([candidate(k) for k in ks], x.shape[0])

    def batch(ks):
        p = vn_objective_partials(clip, family_program(ks))
        p = p.cpu().numpy() if R.is_torch_tensor(p) else p
        return list(vn_scores_from_partials(p, **kw)[0])

    print("Starting Grid Scan")  # grid_scan's message (optimization.py:112)
    scores = np.asarray(batch(kappas))
    local_minima = get_local_minima(scores, grid_size)

    best, _ = _refine_minima([local_minima], kappas, lambda _, ks: batch(ks.tolist()))
    return best[0]


# ------------------------------------------------------------------------------------------------
# many clips at once (BASELINE config 5): clips sharded over ranks, one all-gather of the scores
# ------------------------------------------------------------------------------------------------


_NO_FRAME_LIMIT = 2**31 - 1  # a clip length no tap reaches: family(kappas, _NO_FRAME_LIMIT) keeps every tap


def _concat_programs(progs: Sequence[TapProgram]) -> TapProgram:
    """The channels of several SEGMENTED programs of one envelope, in order, as one program."""
    if len(progs) == 1:
        return progs[0]
    base = np.cumsum([0] + [p.words.size for p in progs])
    offsets = np.concatenate([p.offsets[:-1].astype(np.int64) + b for p, b in zip(progs, base[:-1])] + [base[-1:]])
    if offsets[-1] >= 2**31:
        raise ValueError("tap program too large")
    return TapProgram(np.ascontiguousarray(np.concatenate([p.words for p in progs]), dtype=np.int32), offsets.astype(np.int32),
                      sum(p.channels for p in progs), N.ORDER_SEGMENTED, progs[0].apply_gain, max(p.halo for p in progs),
                      max(p.max_channel_words for p in progs))


def _run_program(family: Callable[[Sequence[float], int], TapProgram], lengths, groups, base: list) -> tuple[TapProgram, np.ndarray]:
    """One tap program and the ``(4, n_runs)`` run table of ``vn_objective_run_partials`` for ``groups``: run ``r`` is
    ``(clip, kappas, position of kappas[0] in base, first output row)``.

    A program drops the taps at or beyond the clip's length, so a channel is valid for every clip longer than its
    largest tap.  Channels ``[0, len(base))`` are ``family(base, ...)`` with every tap kept: the runs of clips longer
    than the largest tap of ``base`` point into it.  Each shorter length is a class of its own, packed exactly as
    ``family(kappas, frames)`` packs it for one clip of that length, and appended; runs of one class that share a kappa
    list (the grid) share its channels."""
    full = family(base, _NO_FRAME_LIMIT)
    last_tap = full.halo - 1
    classes: dict[int, tuple[list, dict]] = {}
    where = []
    for clip, ks, pos, _ in groups:
        f = int(lengths[clip])
        if f > last_tap:
            where.append((None, pos))
            continue
        kappas, seen = classes.setdefault(f, ([], {}))
        if id(ks) not in seen:
            seen[id(ks)] = len(kappas)
            kappas.extend(ks)
        where.append((f, seen[id(ks)]))
    progs, first = [full], {}
    at = full.channels
    for f, (kappas, _) in classes.items():
        progs.append(family(kappas, f))
        first[f] = at
        at += progs[-1].channels
    runs = np.array([[g[0] for g in groups], [pos if f is None else first[f] + pos for f, pos in where], [len(g[1]) for g in groups],
                     [g[3] for g in groups]], dtype=np.int64).reshape(4, len(groups))
    return _concat_programs(progs), runs


def _pack_clips(clips):
    """The clips as one channel-planar float32 ``(2, rows)`` tensor on their GPU (clip ``i`` is columns
    ``offs[i]:offs[i + 1]``, cast and sliced as ``_as_stereo_f32`` does), the int64 offsets and the device.  ``clips``:
    a list of numpy arrays or of CUDA tensors, or a planar ``(n, 2, frames)`` array or CUDA tensor (one copy)."""
    import torch

    planar = R.is_torch_tensor(clips) or isinstance(clips, np.ndarray)
    lengths = [int(clips.shape[2])] * int(clips.shape[0]) if planar else [int(c.shape[0]) for c in clips]
    offs = np.zeros(len(lengths) + 1, dtype=np.int64)
    np.cumsum(lengths, out=offs[1:])
    rows = int(offs[-1])
    if planar:
        if R.is_torch_tensor(clips):
            return clips.to(torch.float32).permute(1, 0, 2).contiguous().reshape(2, rows), offs, clips.device  # one copy, whatever the strides
        device = torch.device("cuda", R.default_device())
        host = np.ascontiguousarray(np.asarray(clips).astype(np.float32, copy=False).transpose(1, 0, 2)).reshape(2, rows)
        return torch.from_numpy(host).to(device), offs, device
    if clips and R.is_torch_tensor(clips[0]):
        device = clips[0].device
        x = torch.empty((2, rows), dtype=torch.float32, device=device)
        for c, a, b in zip(clips, offs[:-1], offs[1:]):
            t = c.to(torch.float32)  # rounds like numpy's astype
            x[:, a:b] = (t[:, None].expand(-1, 2) if t.dim() == 1 else t[:, :2]).T
        return x, offs, device
    device = torch.device("cuda", R.default_device())
    host = np.empty((2, rows), dtype=np.float32)
    for c, a, b in zip(clips, offs[:-1], offs[1:]):
        host[:, a:b] = _as_stereo_f32(c).T
    return torch.from_numpy(host).to(device), offs, device


class _ClipBank:
    """The rank's clips resident on its GPU, packed once into one channel-planar float32 ``(2, rows)`` tensor
    (``_pack_clips``), and the velvet-noise objective on them: the grid and every flat (clip, strength) list are ONE
    ``vn_objective_run_partials`` call each (one run per clip, one tap program per call with a class of channels per
    clip length that drops taps, ``_run_program``), then one asynchronous download of the partial sums and one
    vectorised scoring pass.  ``lanes = 2`` from two clips on: the refinement keeps two half-batches of clips in flight,
    so that scoring and the Brent step of one run under the kernels of the other."""

    def __init__(self, clips, family: Callable[[Sequence[float], int], TapProgram], kw: dict):
        self.x, self.offs, self.device = _pack_clips(clips)
        self.lengths = np.diff(self.offs)
        self.n = len(self.lengths)
        self.lanes = 2 if self.n >= 2 else 1
        self.family = family
        self.kw = kw
        self.evaluations = 0
        self.launches = 0

    def _partials(self, groups, base):
        prog, runs = _run_program(self.family, self.lengths, groups, base)
        import torch

        with torch.cuda.device(self.device):
            out = vn_objective_run_partials(self.x, self.offs, prog, runs)
        self.launches += 1
        return out

    def grid_scores(self, kappas: Sequence[float]) -> np.ndarray:
        """float32 ``(n, len(kappas))`` scores of every clip at every strength: ONE call."""
        k = len(kappas)
        partials = self._partials([(i, kappas, 0, i * k) for i in range(self.n)], kappas)
        self.evaluations += self.n * k
        return vn_scores_from_partials(partials.cpu().numpy().reshape(self.n, k, N.OBJ_SLOTS), **self.kw)

    def submit(self, clip_ids: np.ndarray, kappas: Sequence[float]):
        """Enqueue the evaluation of the clip-major pairs (``clip_ids[p]``, ``kappas[p]``) - ONE call, one run per
        clip - and the download of their partial sums into page-locked memory; returns a handle for ``collect``."""
        import torch

        starts = np.flatnonzero(np.r_[True, clip_ids[1:] != clip_ids[:-1]])  # one run of pairs per clip
        ends = np.r_[starts[1:], len(clip_ids)]
        out = self._partials([(int(clip_ids[a]), kappas[a:b], a, a) for a, b in zip(starts.tolist(), ends.tolist())], kappas)
        self.evaluations += len(kappas)
        host = torch.empty(out.shape, dtype=out.dtype, pin_memory=True)
        host.copy_(out, non_blocking=True)
        done = torch.cuda.Event()
        done.record(torch.cuda.current_stream(self.device))
        return host, done, out  # out is kept alive until the copy has run

    def collect(self, handle) -> np.ndarray:
        """Scores (flat float32 array, pair order) of a submitted batch."""
        host, done, _ = handle
        done.synchronize()
        return vn_scores_from_partials(host.numpy(), **self.kw)


def _optimize_batch(*, input_signals, local_signals, total_clips, group, details: bool, split: Callable[[Any, int], Sequence],
                    make_bank: Callable[[Sequence], Any], grid: np.ndarray, convert: Callable[[np.ndarray], Any], dtype):
    """The multi-clip optimiser behind ``optimize_velvet_noise_batch`` and ``optimize_haas_delay_batch``: resolve the
    rank's block of clips, score it on the grid, all-gather the score matrix, refine the local minima of the rank's
    clips in lock-step and all-gather the results.

    ``split(signals, first)`` checks the clips and returns them as a sequence (``first``: the index of the first clip,
    for the messages).  ``make_bank(clips)`` holds the rank's clips and scores them: ``grid_scores(args)`` returns the
    ``(n_local, len(grid))`` score matrix in one launch; ``submit(clip_ids, args)`` and ``collect(handle)`` score flat
    clip-major pairs; ``lanes``, ``device``, ``evaluations`` and ``launches`` are read.  ``convert`` turns an array of
    grid values or abscissae into the bank's arguments; ``dtype`` is the objective's."""
    from . import sharding as S

    rank, world = S._world(group)
    if local_signals is not None:
        if total_clips is None:
            raise ValueError("local_signals needs total_clips (the number of clips over all ranks)")
        n_clips = int(total_clips)
        lo, hi = S.block_range(n_clips, rank, world)
        local = split(local_signals, lo)
        if len(local) != hi - lo:
            raise ValueError(f"rank {rank} of {world} owns clips [{lo}, {hi}) but local_signals holds {len(local)}")
    else:
        if input_signals is None:
            raise ValueError("pass input_signals (all clips) or local_signals (this rank's block)")
        every = split(input_signals, 0)  # every rank checks every clip, so that all ranks raise alike
        n_clips = len(every)
        lo, hi = S.block_range(n_clips, rank, world)
        local = every[lo:hi]

    bank = None
    local_scores = np.zeros((0, len(grid)), dtype=dtype)
    if hi > lo:
        bank = make_bank(local)
        print("Starting Grid Scan")
        local_scores = np.ascontiguousarray(bank.grid_scores(convert(grid)), dtype=dtype)
    counts = [b - a for a, b in (S.block_range(n_clips, r, world) for r in range(world))]
    device = bank.device if (bank is not None and bank.device is not None) else S.collective_device(group)
    scores = S.all_gather_rows(local_scores, counts, device=device, group=group)  # every rank: (n_clips, grid)

    minima = [get_local_minima(row, len(grid)) for row in scores]
    best, rounds = np.zeros(hi - lo), 0
    if hi > lo:
        best, rounds = _refine_minima(minima[lo:hi], grid, lambda clip_ids, xs: bank.submit(clip_ids, convert(xs)), bank.collect, bank.lanes)
    refined = S.all_gather_rows(best.reshape(-1, 1), counts, device=device, group=group).reshape(-1)
    if details:
        info = {"scores": scores, "local_minima": minima, "argmin": [int(np.argmin(r)) for r in scores],
                "evaluations_local": bank.evaluations if bank is not None else 0, "launches_local": bank.launches if bank is not None else 0,
                "rounds_local": rounds, "clips_local": (lo, hi)}
        return refined, info
    return refined


def _vn_family(*, sample_rate_hz: int, duration_seconds: float, num_impulses: int, seed) -> Callable[[Sequence[float], int], TapProgram]:
    """``family(kappas, frames)``: the tap program of the candidates ``optimize_velvet_noise`` scores for a clip of
    ``frames`` samples, packed as it packs them (``kappa_family_program``, table by table when that does not apply)."""

    def candidate(kappa):
        return VelvetNoise(sample_rate_hz=sample_rate_hz, duration_seconds=duration_seconds, num_impulses=num_impulses,
                           log_distribution_strength=kappa, normalizer=None, filtered_channels=(0,), mode="LR", seed=seed)

    envelope = candidate(0.0).segment_envelope

    def family(ks, frames):
        prog = kappa_family_program(ks, sample_rate_hz=sample_rate_hz, duration_seconds=duration_seconds, num_impulses=num_impulses,
                                    envelope=envelope, seed=seed, frames=frames) if seed is not None else None
        return prog if prog is not None else _vn_family_program([candidate(k) for k in ks], frames)

    return family


def optimize_velvet_noise_batch(*, input_signals=None, sample_rate_hz: int, duration_seconds: float, num_impulses: int, seed: int = 1,
                                grid_size: int = 400, angle_limit: float = np.pi / 4, lambda_mean: float = 5.0, lambda_skew: float = 2.0,
                                lambda_correlation: float = 15.0, lambda_penalty: float = 1e3, group=None, details: bool = False,
                                local_signals=None, total_clips: int | None = None, _bank_factory=None):
    """``optimize_velvet_noise`` (optimization.py:230-310) for MANY clips of any lengths: returns the float64 array of
    optimised ``log_distribution_strength`` values, element ``i`` equal to what ``optimize_velvet_noise(input_signal=
    input_signals[i], ...)`` returns (for a CUDA tensor clip: on ``clip.cpu().numpy()``).  All clips share the
    optimiser's settings.

    ``input_signals``: a list of clips - numpy arrays or CUDA tensors (not a mix, one device), mono ``(frames,)``,
    stereo ``(frames, 2)`` or wider ``(frames, k)`` (the first two channels are used), any dtype, cast to float32 as the
    single-clip call does - or one PLANAR ``(n_clips, 2, frames)`` array or CUDA tensor (unlike
    ``optimize_haas_delay_batch``, whose batch array is ``(n_clips, frames, 2)``).  An empty clip raises ``ValueError``
    naming its index before any device work, and so do bad shapes and mixed numpy and CUDA clips.  With
    ``torch.distributed`` initialised (one process per GPU) the clips are partitioned in contiguous blocks over the ranks
    of ``group`` (``sharding.block_range``); every rank passes the SAME ``input_signals`` (only its block is read and
    uploaded) - or, when the clips already live on the ranks, its own block as ``local_signals`` (e.g. a resident CUDA
    tensor) together with ``total_clips``.

    Data path per rank: its clips are packed once into one resident channel-planar float32 tensor; the grid scores are
    ONE run-list objective call over every clip (``vn_objective_run_partials``) -> ONE all-gather of the float32 score
    matrix so that every rank holds all rows (``get_local_minima`` needs both neighbours of every grid point,
    optimization.py:120-128) -> lock-step Brent refinement of the local minima of its own clips, ONE call per batch of
    live minimisers -> one all-gather of the refined strengths.  ``details=True`` also returns the score matrix, the
    local-minima sets, the per-clip argmin, and this rank's evaluation, launch (objective calls) and Brent-round counts
    and clip range."""
    kw = dict(angle_limit=angle_limit, lambda_mean=lambda_mean, lambda_skew=lambda_skew, lambda_correlation=lambda_correlation,
              lambda_penalty=lambda_penalty)
    family = _vn_family(sample_rate_hz=sample_rate_hz, duration_seconds=duration_seconds, num_impulses=num_impulses, seed=seed)
    return _optimize_batch(input_signals=input_signals, local_signals=local_signals, total_clips=total_clips, group=group, details=details,
                           split=_vn_batch_clips, make_bank=lambda clips: (_bank_factory or _ClipBank)(clips, family, kw),
                           grid=np.linspace(0.0, 1.0, grid_size), convert=np.ndarray.tolist, dtype=np.float32)


# ------------------------------------------------------------------------------------------------
# optimize_haas_delay for many clips of any lengths: one launch for the grid, one per Brent round
# ------------------------------------------------------------------------------------------------


def _check_clip_list(clips, first: int) -> list:
    """The per-clip checks both multi-clip optimisers make before any device work: all numpy arrays or all CUDA tensors
    on one device, each mono ``(frames,)`` or ``(frames, k >= 2)`` (the shapes ``_as_stereo_f32`` accepts) and not
    empty.  ``first`` is the index of the first clip in the whole batch (for the messages)."""
    clips = [c if R.is_torch_tensor(c) else np.asarray(c) for c in clips]
    kinds = {R.is_torch_tensor(c) for c in clips}
    if len(kinds) > 1:
        raise ValueError("clips must be all numpy arrays or all CUDA tensors, not a mix")
    if kinds == {True}:
        if not all(c.is_cuda for c in clips):
            raise ValueError("torch clips must be CUDA tensors")
        if len({c.device for c in clips}) > 1:
            raise ValueError(f"CUDA clips must be on one device, got {sorted({str(c.device) for c in clips})}")
    for i, c in enumerate(clips):
        shape = tuple(c.shape)
        if len(shape) not in (1, 2) or (len(shape) == 2 and shape[1] < 2):
            raise ValueError(f"clip {first + i}: Input shape invalid: Expected shape (num samples, 2), but got shape {shape}.")
        if shape[0] == 0:
            raise ValueError(f"clip {first + i} is empty: zero-size array to reduction operation maximum which has no identity")
    return clips


def _haas_batch_clips(signals, first: int = 0) -> list:
    """The clips of ``signals`` (a list of numpy arrays or CUDA tensors, or one ``(n_clips, frames, 2)`` array or
    tensor) as a list, after ``_check_clip_list``."""
    if R.is_torch_tensor(signals) or isinstance(signals, np.ndarray):
        if signals.ndim != 3 or signals.shape[2] != 2:
            raise ValueError(f"a batch array must have shape (n_clips, frames, 2), got {tuple(signals.shape)}")
        return _check_clip_list([signals[i] for i in range(signals.shape[0])], first)
    return _check_clip_list(signals, first)


def _vn_batch_clips(signals, first: int = 0):
    """The clips of ``signals`` for ``optimize_velvet_noise_batch``: a list after ``_check_clip_list``, or a planar
    ``(n_clips, 2, frames)`` numpy array or CUDA tensor, kept whole (it packs with one copy)."""
    if R.is_torch_tensor(signals) or isinstance(signals, np.ndarray):
        if signals.ndim != 3 or signals.shape[1] != 2:
            raise ValueError(f"a batch array must be planar with shape (n_clips, 2, frames), got {tuple(signals.shape)}")
        if R.is_torch_tensor(signals) and not signals.is_cuda:
            raise ValueError("torch clips must be CUDA tensors")
        if signals.shape[0] and signals.shape[2] == 0:
            raise ValueError(f"clip {first} is empty: zero-size array to reduction operation maximum which has no identity")
        return signals
    return _check_clip_list(signals, first)


class _HaasClipBank:
    """The rank's clips resident on its GPU, packed once into one channel-planar float32 ``(2, rows)`` tensor (clip ``i``
    is columns ``offs[i]:offs[i + 1]``, cast and sliced as ``_as_stereo_f32`` does), and the evaluation of flat
    (clip, delay) lists on them: one launch, one synchronous download of the partial sums, one vectorised scoring pass.
    ``lanes = 1``: one batch in flight, so that the launches are one for the grid and one per Brent round."""

    def __init__(self, clips, kw: dict):
        import torch

        self.x, self.offs, self.device = _pack_clips(clips)
        self.n = len(clips)
        self.kw = kw
        self.offs_dev = torch.from_numpy(self.offs).to(self.device)
        self.lanes = 1
        self.evaluations = 0
        self.launches = 0

    def grid_scores(self, delays) -> np.ndarray:
        """float64 ``(n, len(delays))`` scores of every clip at every delay: ONE launch."""
        return self.collect(self.submit(np.repeat(np.arange(self.n), len(delays)), np.tile(delays, self.n))).reshape(self.n, len(delays))

    def submit(self, clip_ids, delays) -> np.ndarray:
        """float64 scores of the pairs (``clip_ids[p]``, ``delays[p]``), in pair order: ONE kernel launch; the scores
        are the handle."""
        import torch

        pc = np.ascontiguousarray(clip_ids, dtype=np.int32)
        pairs = torch.from_numpy(np.stack((pc, np.ascontiguousarray(delays, dtype=np.int32)))).to(self.device)
        with torch.cuda.device(self.device):
            p = haas_objective_pair_partials(self.x, self.offs_dev, pairs[0], pairs[1])
        self.launches += 1
        self.evaluations += pc.size
        return haas_scores_from_partials(p.cpu().numpy(), **self.kw)

    def collect(self, handle) -> np.ndarray:
        return handle


def optimize_haas_delay_batch(*, input_signals=None, sample_rate_hz: int, max_delay_seconds: float, grid_size: int = 400,
                              angle_limit: float = np.pi / 4, lambda_mean: float = 5.0, lambda_skew: float = 2.0, lambda_correlation: float = 15.0,
                              lambda_penalty: float = 1e3, group=None, details: bool = False, local_signals=None, total_clips: int | None = None,
                              _bank_factory=None):
    """``optimize_haas_delay`` (optimization.py:158-227) for MANY clips of any lengths: returns the float64 array of
    optimised ``delay_time_seconds`` values, element ``i`` equal to what ``optimize_haas_delay(input_signal=
    input_signals[i], ...)`` returns (for a CUDA tensor clip: on ``clip.cpu().numpy()``).

    ``input_signals``: a list of clips - numpy arrays or CUDA tensors (not a mix, one device), mono ``(frames,)``,
    stereo ``(frames, 2)`` or wider ``(frames, k)`` (the first two channels are used), any dtype, cast to float32 as the
    single-clip call does - or one ``(n_clips, frames, 2)`` array or tensor.  An empty clip raises ``ValueError`` naming
    its index before any device work.  With ``torch.distributed`` initialised the clips are partitioned in contiguous
    blocks over the ranks of ``group`` (``sharding.block_range``), exactly as in ``optimize_velvet_noise_batch``: every
    rank passes the same ``input_signals``, or its own block as ``local_signals`` with ``total_clips``.

    Per rank: its clips are packed once into one resident channel-planar float32 tensor; the grid stage is ONE launch
    over every (clip, grid delay) pair; the float64 ``(n_clips, grid_size)`` score matrix is all-gathered once; the
    local minima of every clip of the rank are refined in lock-step with ONE launch per Brent round over all live
    minimisers; the refined delays are all-gathered once.  Delays in frames are ``round(t * sample_rate_hz)``, as
    ``HaasEffect.delay_len_samples`` computes them.  ``details=True`` also returns the score matrix, the local-minima
    sets, the per-clip argmin, and this rank's evaluation, launch and Brent-round counts and clip range."""
    kw = dict(angle_limit=angle_limit, lambda_mean=lambda_mean, lambda_skew=lambda_skew, lambda_correlation=lambda_correlation,
              lambda_penalty=lambda_penalty)

    def delays(ts):  # HaasEffect.delay_len_samples
        return np.array([round(t * sample_rate_hz) for t in ts.tolist()], dtype=np.int64)

    return _optimize_batch(input_signals=input_signals, local_signals=local_signals, total_clips=total_clips, group=group, details=details,
                           split=_haas_batch_clips, make_bank=lambda clips: (_bank_factory or _HaasClipBank)(clips, kw),
                           grid=np.linspace(0.0, max_delay_seconds, grid_size), convert=delays, dtype=np.float64)
