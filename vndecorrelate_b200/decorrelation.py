"""Decorrelators with the reference's API (``src/vndecorrelate/decorrelation.py``) running on the
sm_100a kernels of ``libvnd_b200.so``.

Same names, keyword arguments, defaults, return dtypes/shapes and exceptions as the reference for
the hot path: ``VelvetNoise`` (``decorrelate`` / ``convolve`` / ``FIR`` / ``velvet_noise``),
``HaasEffect``, ``SignalChain`` (``velvet_noise`` / ``haas_effect`` / ``stateless``),
``generate_velvet_noise`` and ``convolve_velvet_noise``.  Inputs may be numpy arrays (numpy comes
back, copies inside the call) or CUDA ``torch.Tensor``s (tensors come back, no host round trip).
A ``[VelvetNoise, HaasEffect(LR)]`` pair in a ``SignalChain`` runs as ONE fused launch sequence.

``WhiteNoise`` (a dense Gaussian FIR, decorrelation.py:670-716) is outside the sparse hot path and
is not provided; ``SignalChain.white_noise`` raises ``NotImplementedError``.
"""

from __future__ import annotations

import ctypes as C
import os
from functools import partial
from typing import Any, Callable, Sequence

import numpy as np

from . import _native as N
from . import runtime as R
from .taps import (
    IDENTITY_ENVELOPE,
    TapProgram,
    TapTable,
    ascending_program,
    generate_dense_fir,
    generate_tap_table,
    segmented_program,
)
from .utils.dsp import LayoutMode, apply_stereo_width, check_equal_length, rms_normalize, to_float32

__all__ = ["Decorrelator", "SignalChain", "HaasEffect", "VelvetNoise", "BlockDecorrelator", "BlockConvolver", "decorrelate_batch", "haas_effect_batch", "generate_velvet_noise",
           "convolve_velvet_noise"]


class Decorrelator:
    """Base of the decorrelators: ``num_outs``, ``width``, ``decorrelate`` and ``__call__``
    (decorrelation.py:40-54)."""

    sample_rate_hz: int
    num_outs: int = 2
    width: float | None = None

    def decorrelate(self, input_signal):  # pragma: no cover - abstract
        raise NotImplementedError

    def __call__(self, input_signal):
        return self.decorrelate(input_signal)


# ------------------------------------------------------------------------------------------------
# low-level runners shared by the classes
# ------------------------------------------------------------------------------------------------


def _is_mode(mode, which: LayoutMode) -> bool:
    return mode == which  # StrEnum compares equal to plain 'LR' / 'MS' strings (decorrelation.py:217,433)


def _fir_compute_dtype(dtype) -> np.dtype:
    """The dtype numpy would effectively feed ``f32_buffer -= x[i:]`` with: float32 stays float32,
    float64 stays float64, small integers behave like float32 and 32/64-bit integers like float64
    (numpy type promotion with a float32 accumulator)."""
    dtype = np.dtype(dtype)
    if dtype in (np.float32, np.float64):
        return dtype
    if dtype == np.float16 or (dtype.kind in "iub" and dtype.itemsize <= 2):
        return np.dtype(np.float32)
    if dtype.kind in "iuf":
        return np.dtype(np.float64)
    raise TypeError(f"unsupported input dtype {dtype}")


def _fir_compute_array(x: np.ndarray) -> np.ndarray:
    """``x`` in ``_fir_compute_dtype``: the array itself when it already has that dtype."""
    dt = _fir_compute_dtype(x.dtype)
    return x if x.dtype == dt else x.astype(dt)


def _fir_tensor_dtype(x):
    """The torch dtype ``_sparse_fir`` computes a tensor in: float32 and float64 as they are, half precision and
    integers of up to 2 bytes in float32, anything wider in float64."""
    import torch

    if x.dtype in (torch.float32, torch.float64):
        return x.dtype
    return torch.float32 if (x.dtype == torch.float16 or x.element_size() <= 2) else torch.float64


def _sparse_fir(x, program: TapProgram, num_outs: int):
    """``(frames, >= num_outs)`` signal -> float32 ``(frames, num_outs)``."""
    lib = N.lib()
    if R.is_torch_tensor(x):
        import torch

        if not x.is_cuda:
            raise N.VndError(N.VND_EUNSUPPORTED, "sparse FIR", "CPU torch tensors are not supported (no CPU fallback); pass a CUDA tensor or a numpy array")
        x = x.to(_fir_tensor_dtype(x))
        frames = x.shape[0]
        # planar inputs (a transposed (C, n) tensor) get a planar output, so loads and stores coalesce
        planar = x.dim() == 2 and x.shape[1] > 1 and x.stride(0) == 1
        y = torch.empty((num_outs, frames), dtype=torch.float32, device=x.device).t() if planar else torch.empty((frames, num_outs), dtype=torch.float32, device=x.device)
        sx, sy = R.torch_signal(x), R.torch_signal(y)
        with torch.cuda.device(x.device):
            ps = R.device_program(program, x.device)
            N.check(lib.vnd_sparse_fir_dev(C.byref(sx), C.byref(sy), C.byref(ps), R.torch_stream_ptr(x)), "vnd_sparse_fir_dev")
        return y
    xa = R.dense(_fir_compute_array(np.asarray(x)))
    frames = xa.shape[0]
    planar = xa.ndim == 2 and xa.shape[1] > 1 and not xa.flags.c_contiguous
    y = R.pinned_empty((num_outs, frames), np.float32).T if planar else R.pinned_empty((frames, num_outs), np.float32)
    sx, sy = R.host_signal(xa), R.host_signal(y)
    ps = program.host_struct()
    N.check(lib.vnd_sparse_fir_host(R.HostContext.get().handle, C.byref(sx), C.byref(sy), C.byref(ps)), "vnd_sparse_fir_host")
    return y


def _vn_decorrelate(x32, program: TapProgram, *, num_outs: int, ms_encode: bool, width, rms: bool, haas_delay: int = 0,
                    haas_channel: int = 0, out_f64: bool = False):
    """Fused decorrelate on a float32 signal (1-D mono or ``(frames, >= num_outs)``)."""
    lib = N.lib()
    ep = N.EpilogueStruct(int(ms_encode), int(width is not None), float(width) if width is not None else 0.0, int(rms), int(haas_delay), int(haas_channel))
    mono = x32.ndim == 1
    frames = x32.shape[0]
    if R.is_torch_tensor(x32):
        import torch

        if not x32.is_cuda:
            raise N.VndError(N.VND_EUNSUPPORTED, "decorrelate", "CPU torch tensors are not supported (no CPU fallback); pass a CUDA tensor or a numpy array")
        out = torch.empty((frames + haas_delay, num_outs), dtype=torch.float64 if out_f64 else torch.float32, device=x32.device)
        sx = R.torch_signal(x32, mono_as_stereo=mono)
        so = R.torch_signal(out)
        nbytes = C.c_size_t()
        N.check(lib.vnd_vn_decorrelate_workspace(frames, num_outs, C.byref(ep), C.byref(nbytes)), "vnd_vn_decorrelate_workspace")
        with torch.cuda.device(x32.device):
            work = torch.empty(nbytes.value, dtype=torch.uint8, device=x32.device)
            ps = R.device_program(program, x32.device)
            N.check(lib.vnd_vn_decorrelate_dev(C.byref(sx), C.byref(so), C.byref(ps), C.byref(ep), work.data_ptr(), nbytes.value,
                                               R.torch_stream_ptr(x32)), "vnd_vn_decorrelate_dev")
        return out
    xa = R.dense(x32)
    out = R.pinned_empty((frames + haas_delay, num_outs), np.float64 if out_f64 else np.float32)
    sx = R.host_signal(xa, mono_as_stereo=mono)
    so = R.host_signal(out)
    ps = program.host_struct()
    N.check(lib.vnd_vn_decorrelate_host(R.HostContext.get().handle, C.byref(sx), C.byref(so), C.byref(ps), C.byref(ep)), "vnd_vn_decorrelate_host")
    return out


def _haas(x32, *, delay: int, delayed_channel: int, mode_ms: bool, width):
    lib = N.lib()
    mono = x32.ndim == 1
    frames = x32.shape[0]
    args = (int(delay), int(delayed_channel), int(mode_ms), int(mono), int(width is not None), float(width) if width is not None else 0.0)
    if R.is_torch_tensor(x32):
        import torch

        if not x32.is_cuda:
            raise N.VndError(N.VND_EUNSUPPORTED, "haas", "CPU torch tensors are not supported (no CPU fallback)")
        out = torch.empty((frames + delay, 2), dtype=torch.float64, device=x32.device)
        sx, so = R.torch_signal(x32, mono_as_stereo=mono), R.torch_signal(out)
        with torch.cuda.device(x32.device):
            N.check(lib.vnd_haas_dev(C.byref(sx), C.byref(so), *args, R.torch_stream_ptr(x32)), "vnd_haas_dev")
        return out
    xa = R.dense(x32)
    out = R.pinned_empty((frames + delay, 2), np.float64)
    sx, so = R.host_signal(xa, mono_as_stereo=mono), R.host_signal(out)
    N.check(lib.vnd_haas_host(R.HostContext.get().handle, C.byref(sx), C.byref(so), *args), "vnd_haas_host")
    return out


# ------------------------------------------------------------------------------------------------
# Haas effect (decorrelation.py:163-230)
# ------------------------------------------------------------------------------------------------


class HaasEffect(Decorrelator):
    """Delays one channel (L/R, or mid/side in MS mode) by ``delay_time_seconds``; returns float64
    ``(n + round(delay * fs), 2)`` like the reference."""

    def __init__(self, *, sample_rate_hz: int, num_outs: int = 2, width: float | None = None, delayed_channel: int = 0,
                 delay_time_seconds: float = 0.02, mode: LayoutMode = LayoutMode.LR):
        self.sample_rate_hz = sample_rate_hz
        self.num_outs = num_outs
        self.width = width
        self.delayed_channel = delayed_channel
        self.delay_time_seconds = delay_time_seconds
        self.mode = mode

    @property
    def delay_len_samples(self) -> int:
        return round(self.delay_time_seconds * self.sample_rate_hz)  # Python's round-half-even, decorrelation.py:204

    def _check(self, x) -> None:
        if x.ndim not in (1, 2) or (x.ndim == 2 and x.shape[1] != 2):
            raise ValueError(f"could not broadcast input array from shape {tuple(x.shape)} into shape ({x.shape[0]},2)")
        if self.delayed_channel not in (0, 1, -1, -2):
            raise IndexError(f"index {self.delayed_channel} is out of bounds for axis 1 with size 2")

    def haas_delay(self, input_signal):
        """The delay alone (no width), as ``HaasEffect.haas_delay`` (decorrelation.py:202-230)."""
        self._check(input_signal)
        return _haas(to_float32(input_signal), delay=self.delay_len_samples, delayed_channel=self.delayed_channel % 2,
                     mode_ms=_is_mode(self.mode, LayoutMode.MS), width=None)

    def decorrelate(self, input_signal):
        input_signal = to_float32(input_signal if R.is_torch_tensor(input_signal) else np.asarray(input_signal))
        self._check(input_signal)
        return _haas(input_signal, delay=self.delay_len_samples, delayed_channel=self.delayed_channel % 2,
                     mode_ms=_is_mode(self.mode, LayoutMode.MS), width=self.width)


# ------------------------------------------------------------------------------------------------
# Velvet noise (decorrelation.py:326-546)
# ------------------------------------------------------------------------------------------------


class VelvetNoise(Decorrelator):
    """Velvet-noise decorrelator: a sparse FIR of ``num_impulses`` signed unit impulses per channel
    with a segmented decay envelope, applied anti-causally (``y[t] = sum c_k x[t + i_k]``), then
    optional M/S side-channel encode, width and RMS normalisation.

    Constructor arguments, defaults and attribute semantics are the reference's
    (decorrelation.py:355-362): the tap table is generated at construction from ``seed`` and
    regenerated only when ``num_outs``, ``num_impulses`` or the FIR length change; a new
    ``segment_envelope`` is picked up at call time."""

    def __init__(self, *, sample_rate_hz: int, num_outs: int = 2, width: float | None = None, duration_seconds: float = 0.03,
                 num_impulses: int = 30, segment_envelope: Sequence[float] = (0.85, 0.55, 0.35, 0.2),
                 log_distribution_strength: float = 1.0, normalizer: Callable[[Any, Any], None] | None = rms_normalize,
                 filtered_channels: Sequence[int] = (0, 1), mode: LayoutMode = LayoutMode.MS, seed: int | None = None):
        self.sample_rate_hz = sample_rate_hz
        self.num_outs = num_outs
        self.width = width
        self.duration_seconds = duration_seconds
        self.num_impulses = num_impulses
        self.segment_envelope = segment_envelope
        self.log_distribution_strength = log_distribution_strength
        self.normalizer = normalizer
        self.filtered_channels = filtered_channels
        self.mode = mode
        self.seed = seed
        if self.num_impulses >= self.fir_length_samples * 0.2:  # decorrelation.py:382-387
            raise ValueError(
                f"Velvet Noise Filter of length {self.fir_length_samples} with {self.num_impulses} impulses is not sparse. "
                f"(density={self.density:.2f})\n\tnum_impulses must be less than 20% the FIR length in samples."
            )
        if not self.segment_envelope:
            self.segment_envelope = IDENTITY_ENVELOPE
        self._velvet_noise: TapTable = self._generate()
        self._programs: dict = {}

    # ---- properties of the reference ------------------------------------------------------------
    @property
    def density(self) -> float:
        return self.num_impulses / self.duration_seconds

    @property
    def fir_length_samples(self) -> int:
        return int(round(self.sample_rate_hz * self.duration_seconds))

    @property
    def unfiltered_channels(self):
        return filter(lambda i: i not in self.filtered_channels, range(self.num_outs))

    @property
    def velvet_noise(self) -> TapTable:
        """The tap table; regenerated when ``num_outs``, ``num_impulses`` or the FIR length changed
        since it was made (decorrelation.py:368-379)."""
        t = self._velvet_noise
        if self.num_outs != t.num_outs or self.num_impulses != t.num_impluses or self.fir_length_samples != t.fir_length_samples:
            self._velvet_noise = self._generate()
            self._programs.clear()
        return self._velvet_noise

    def _generate(self) -> TapTable:
        return generate_tap_table(
            sample_rate_hz=self.sample_rate_hz, duration_seconds=self.duration_seconds, num_impulses=self.num_impulses,
            num_outs=self.num_outs, num_segments=len(self.segment_envelope), log_distribution_strength=self.log_distribution_strength,
            filtered_channels=self.filtered_channels, seed=self.seed,
        )

    @property
    def FIR(self) -> np.ndarray:
        """Dense float64 ``(fir_length_samples, len(filtered_channels))`` impulse responses
        (decorrelation.py:454-472)."""
        table = self.velvet_noise
        num_filters = len(self.filtered_channels)
        fir = np.zeros((self.fir_length_samples, num_filters))
        chans = np.nonzero(table.filtered)[0]
        if len(chans) != num_filters:
            raise ValueError("setting an array element with a sequence. The requested array has an inhomogeneous shape")
        for col, c in enumerate(chans):
            for s, seg in enumerate(table[c]):
                for indices, sign in ((seg[0], -1), (seg[1], 1)):
                    for i in indices:
                        fir[i, col] = self.segment_envelope[s] * sign
        return fir

    # ---- tap programs ---------------------------------------------------------------------------
    def tap_program(self, frames: int) -> TapProgram:
        """The packed program for a signal of ``frames`` samples (cached; the key includes the
        envelope because it may be replaced after construction, tests/test_decorrelation.py:148-158)."""
        table = self.velvet_noise
        env = self.segment_envelope
        max_index = int(table.index[table.filtered].max()) if table.filtered.any() and table.num_impulses else -1
        key = (min(frames, max_index + 1), tuple(env), env == IDENTITY_ENVELOPE)
        prog = self._programs.get(key)
        if prog is None:
            if len(self._programs) > 8:
                self._programs.clear()
            prog = segmented_program(table, env, frames)
            self._programs[key] = prog
        return prog

    # ---- the hot path ---------------------------------------------------------------------------
    def convolve(self, input_signal):
        """Sparse FIR on each filtered channel, other channels copied; float32 ``(n, num_outs)``
        (decorrelation.py:393-415).  ``input_signal`` must be 2-D with at least ``num_outs`` columns."""
        if input_signal.ndim != 2:
            raise IndexError(f"too many indices for array: array is {input_signal.ndim}-dimensional, but 2 were indexed")
        if input_signal.shape[1] < self.num_outs:
            raise IndexError(f"index {input_signal.shape[1]} is out of bounds for axis 1 with size {input_signal.shape[1]}")
        return _sparse_fir(input_signal, self.tap_program(input_signal.shape[0]), self.num_outs)

    def decorrelate(self, input_signal):
        """cast -> (mono -> stereo) -> FIR -> M/S encode -> width -> normaliser; float32
        ``(n, num_outs)`` (decorrelation.py:417-442)."""
        x = to_float32(input_signal if R.is_torch_tensor(input_signal) else np.asarray(input_signal))
        return self._decorrelate(x, haas=None)

    def _decorrelate(self, x, haas: "HaasEffect | None"):
        self._check_input(x)
        fused_norm = self.normalizer is None or self.normalizer is rms_normalize
        program = self.tap_program(x.shape[0])
        kw = dict(num_outs=self.num_outs, ms_encode=_is_mode(self.mode, LayoutMode.MS), width=self.width)
        if fused_norm:
            if haas is not None:
                return _vn_decorrelate(x, program, rms=self.normalizer is not None, haas_delay=haas.delay_len_samples,
                                       haas_channel=haas.delayed_channel % 2, out_f64=True, **kw)
            return _vn_decorrelate(x, program, rms=self.normalizer is not None, **kw)
        # user-supplied normaliser: run everything else fused, then hand (input, output) to it
        y = _vn_decorrelate(x, program, rms=False, **kw)
        x2 = x if x.ndim == 2 else (np.column_stack((x, x)) if not R.is_torch_tensor(x) else x[:, None].expand(-1, 2))
        self.normalizer(x2, y)
        return y

    def _check_input(self, x) -> int:
        """The shape checks of ``decorrelate`` on a cast signal (the reference's exceptions); returns the input's
        channel count, 2 for a mono signal."""
        if x.ndim == 1:
            in_channels = 2  # mono_to_stereo, passed to the kernel as a stride-0 broadcast
        elif x.ndim == 2:
            in_channels = x.shape[1]
        else:
            raise ValueError(f"Input shape invalid: Expected shape (num samples,) or (num samples, channels), but got shape {tuple(x.shape)}.")
        if in_channels < self.num_outs:
            raise IndexError(f"index {in_channels} is out of bounds for axis 1 with size {in_channels}")
        ms = _is_mode(self.mode, LayoutMode.MS)
        if ms and (in_channels != 2 or self.num_outs != 2):  # check_stereo in encode_signal_to_side_channel
            bad = (x.shape[0], in_channels) if in_channels != 2 else (x.shape[0], self.num_outs)
            raise ValueError(f"Input shape invalid: Expected shape (num samples, 2), but got shape {bad}.")
        if self.width is not None and self.num_outs != 2:
            raise ValueError(f"Input shape invalid: Expected shape (num samples, 2), but got shape {(x.shape[0], self.num_outs)}.")
        if self.normalizer is rms_normalize and in_channels != self.num_outs:
            raise ValueError(f"operands could not be broadcast together with shapes ({x.shape[0]},{self.num_outs}) ({in_channels},)")
        return in_channels


def _fusable(vn, haas) -> bool:
    return (
        isinstance(vn, VelvetNoise) and isinstance(haas, HaasEffect) and vn.num_outs == 2 and haas.width is None
        and _is_mode(haas.mode, LayoutMode.LR) and (vn.normalizer is None or vn.normalizer is rms_normalize)
        and haas.delayed_channel in (0, 1, -1, -2)
    )


# ------------------------------------------------------------------------------------------------
# Signal chain (decorrelation.py:71-153)
# ------------------------------------------------------------------------------------------------


class SignalChain:
    """Builder of cascaded decorrelators.  Stages are instantiated on the first call unless
    ``lazy=False``.  A ``VelvetNoise`` stage directly followed by an LR-mode ``HaasEffect`` without
    width is executed as one fused device pass (one read and one write per sample when the velvet
    stage has no normaliser; plus the RMS pre-pass otherwise)."""

    def __init__(self, *, sample_rate_hz: int, num_outs: int = 2, lazy: bool = True, _hot: bool = False, _decorrelators=None):
        if _decorrelators is not None:
            raise TypeError(
                "Cannot supply decorrelators directly, use ``SignalChain.velvet_noise``,"
                " ``SignalChain.haas_effect``, or ``SignalChain.stateless``."
            )
        self.sample_rate_hz = sample_rate_hz
        self.num_outs = num_outs
        self.lazy = lazy
        self._hot = _hot or not lazy
        self._decorrelators: list = []

    def haas_effect(self, **kwargs):
        self._add_decorrelator(HaasEffect, **kwargs)
        return self

    def velvet_noise(self, **kwargs):
        self._add_decorrelator(VelvetNoise, **kwargs)
        return self

    def white_noise(self, **kwargs):
        raise NotImplementedError("WhiteNoise is a dense FIR outside the sparse velvet-noise hot path; it is not provided by vndecorrelate_b200")

    def stateless(self, function, *args, **kwargs):
        make = lambda: partial(function, *args, **kwargs)  # noqa: E731
        self._decorrelators.append(make() if self._hot else make)
        return self

    def _add_decorrelator(self, cls, **kwargs) -> None:
        kwargs = self._validate(cls, **kwargs)

        def make():
            if "num_outs" in kwargs:  # the reference passes num_outs twice here (decorrelation.py:115-119)
                raise TypeError(f"{cls.__module__}.{cls.__name__}() got multiple values for keyword argument 'num_outs'")
            return cls(sample_rate_hz=self.sample_rate_hz, num_outs=self.num_outs, **kwargs)

        self._decorrelators.append(make() if self._hot else make)

    def _validate(self, cls, *, sample_rate_hz: int | None = None, **kwargs) -> dict[str, Any]:
        if sample_rate_hz is not None and sample_rate_hz != self.sample_rate_hz:
            raise TypeError(
                f"{sample_rate_hz=} was supplied to {cls} but differs from the sample rate of the enclosing ``SignalChain`` ({self.sample_rate_hz})"
            )
        return kwargs

    def _init_decorrelators(self) -> None:
        if self._hot:
            return
        self._decorrelators = [make() for make in self._decorrelators]
        self._hot = True

    def __call__(self, input_signal):
        self._init_decorrelators()
        stages = self._decorrelators
        sig = input_signal
        i = 0
        while i < len(stages):
            if i + 1 < len(stages) and _fusable(stages[i], stages[i + 1]):
                x = to_float32(sig if R.is_torch_tensor(sig) else np.asarray(sig))
                sig = stages[i]._decorrelate(x, haas=stages[i + 1])
                i += 2
            else:
                sig = stages[i](sig)
                i += 1
        return sig


# ------------------------------------------------------------------------------------------------
# many clips in one call
# ------------------------------------------------------------------------------------------------


def _batch_stages(d) -> "tuple[VelvetNoise, HaasEffect | None]":
    """The (velvet noise, fused Haas or None) pair a batch decorrelator runs as."""
    if isinstance(d, VelvetNoise):
        vn, haas = d, None
    elif isinstance(d, SignalChain):
        d._init_decorrelators()  # a lazy chain is instantiated as its first call would
        stages = d._decorrelators
        if len(stages) == 1 and isinstance(stages[0], VelvetNoise):
            vn, haas = stages[0], None
        elif len(stages) == 2 and _fusable(stages[0], stages[1]):
            vn, haas = stages
        else:
            names = ", ".join(type(st).__name__ for st in stages) or "no stages"
            raise NotImplementedError("decorrelate_batch runs a SignalChain of one VelvetNoise, or of a VelvetNoise followed by an LR-mode "
                                      f"HaasEffect without width; this chain has {names}")
    else:
        raise NotImplementedError(f"decorrelate_batch takes VelvetNoise or SignalChain decorrelators, not {type(d).__name__}")
    if vn.normalizer is not None and vn.normalizer is not rms_normalize:
        raise NotImplementedError("decorrelate_batch fuses rms_normalize or no normaliser; a user-supplied normaliser runs clip by clip")
    return vn, haas


def _batch_settings(vn: VelvetNoise, haas: "HaasEffect | None") -> dict:
    """What the clips of one batch must share (one epilogue and one apply_gain flag for the whole launch)."""
    return {
        "num_outs": vn.num_outs,
        "mode": "MS" if _is_mode(vn.mode, LayoutMode.MS) else "LR",
        "width": vn.width,
        "normalizer": "rms_normalize" if vn.normalizer is rms_normalize else None,
        "Haas stage": haas is not None,
        "Haas delay": haas.delay_len_samples if haas is not None else 0,
        "Haas delayed_channel": haas.delayed_channel % 2 if haas is not None else 0,
        # multiplying by 1.0 is not payload-safe for NaN, so the identity envelope skips the multiply (decorrelation.py:411)
        "identity segment_envelope": vn.segment_envelope == IDENTITY_ENVELOPE,
    }


def _check_offsets(offsets: np.ndarray, n: int, rows: int) -> None:
    """The frame offsets of a packed batch of ``n`` clips: from 0 to ``rows``, never decreasing (the device entry points
    cannot check them)."""
    if len(offsets) != n + 1 or offsets[0] != 0 or offsets[-1] != rows:
        raise ValueError(f"frame offsets must run from 0 to {rows} with one entry per clip and one more")
    if np.any(np.diff(offsets) < 0):
        raise ValueError("frame offsets must not decrease")


def _check_batch_layout(offsets: np.ndarray, program_of_clip: np.ndarray, n_programs: int, rows: int) -> None:
    """The packed layout vnd_vn_decorrelate_batch_* reads: offsets from 0 to ``rows``, never decreasing, and a program
    index in range for every clip (the device entry point cannot check these)."""
    _check_offsets(offsets, len(program_of_clip), rows)
    if len(program_of_clip) and (program_of_clip.min() < 0 or program_of_clip.max() >= n_programs):
        raise ValueError(f"program indices must lie in [0, {n_programs})")


def _batch_programs(filters: "Sequence[VelvetNoise]", lengths) -> "tuple[list[TapProgram], np.ndarray]":
    """The distinct tap programs of a batch and the index of each clip's one.  ``tap_program`` caches one program for
    every length beyond the filter, so all such clips of one filter share it; shorter clips get their truncated one."""
    index: dict[int, int] = {}
    progs: list[TapProgram] = []
    prog_of = np.empty(len(filters), dtype=np.int32)
    for i, (vn, L) in enumerate(zip(filters, lengths)):
        prog = vn.tap_program(int(L))
        if id(prog) not in index:
            index[id(prog)] = len(progs)
            progs.append(prog)
        prog_of[i] = index[id(prog)]
    return progs, prog_of


def _batch_program(progs: "list[TapProgram]") -> TapProgram:
    """One SEGMENTED program holding the k channels of every distinct filter (k = their common channel count, 2 for the
    stereo calls): filter j = channels [j k, (j + 1) k)."""
    k = progs[0].channels
    if any(p.channels != k for p in progs):
        raise ValueError(f"the filters of one batch need one channel count, got {sorted({p.channels for p in progs})}")
    words = np.concatenate([p.words for p in progs]).astype(np.int32, copy=False)
    offsets = np.concatenate([[0]] + [p.offsets[1:].astype(np.int64) + base for p, base in
                                      zip(progs, np.cumsum([0] + [p.words.size for p in progs[:-1]]))]).astype(np.int32)
    return TapProgram(np.ascontiguousarray(words), offsets, k * len(progs), N.ORDER_SEGMENTED, progs[0].apply_gain, max(p.halo for p in progs),
                      max(p.max_channel_words for p in progs))


def _pack_clips(xp: np.ndarray, clips, offsets: np.ndarray) -> None:
    """Copy numpy clips into their rows of the packed (rows, k) array: the first k columns, cast to its dtype (a mono
    clip into both columns of a stereo array).  Large batches
    are copied by several threads: numpy releases the GIL for the copies, and one thread does not reach the host's
    memory bandwidth."""

    def put(i):
        x, a, b = clips[i], offsets[i], offsets[i + 1]
        if x.ndim == 1:
            xp[a:b, 0] = x
            xp[a:b, 1] = x
        else:
            xp[a:b] = x[:, :xp.shape[1]]

    if xp.nbytes < 64 << 20 or len(clips) < 2:
        for i in range(len(clips)):
            put(i)
        return
    from concurrent.futures import ThreadPoolExecutor

    with ThreadPoolExecutor(max_workers=min(8, os.cpu_count() or 1, len(clips))) as pool:
        list(pool.map(put, range(len(clips))))


def _pack_tensors(clips, rows: int, device, cols: int = 2, dtype=None):
    """The CUDA clips packed into one (rows, cols) tensor of ``dtype``, float32 by default: the first ``cols`` columns of
    each clip (a mono clip into both columns of a stereo tensor)."""
    import torch

    dtype = torch.float32 if dtype is None else dtype
    if not rows:
        return torch.empty((0, cols), dtype=dtype, device=device)
    return torch.cat([(x[:, :cols] if x.ndim == 2 else x[:, None].expand(-1, cols)).to(dtype) for x in clips])


def _batch_device(input_signals, is_array: bool, where: str):
    """``(torch_in, device)`` of a batch's clips: all CUDA tensors on one device, or all numpy (device None).  Mixed
    clips and clips on several devices raise ``ValueError``, CPU tensors ``VndError(VND_EUNSUPPORTED)``."""
    torch_in = R.is_torch_tensor(input_signals) if is_array else any(R.is_torch_tensor(c) for c in input_signals)
    if not torch_in:
        return False, None
    if is_array:
        clips_in = [input_signals]
    else:
        clips_in = list(input_signals)
        if not all(R.is_torch_tensor(c) for c in clips_in):
            raise ValueError("clips must be all numpy arrays or all CUDA tensors")
    if not all(c.is_cuda for c in clips_in):
        raise N.VndError(N.VND_EUNSUPPORTED, where, "CPU torch tensors are not supported (no CPU fallback); pass CUDA tensors or numpy arrays")
    device = clips_in[0].device if clips_in else None
    if any(c.device != device for c in clips_in):
        raise ValueError("all clips must be on one CUDA device")
    return True, device


def _cast_clips(input_signals, is_array: bool, torch_in: bool):
    """``(x3, clips)``: the clips cast with ``to_float32`` as the single-clip calls cast them, and for an array of clips
    the cast array itself (None for a list)."""
    if is_array:
        x3 = to_float32(input_signals if torch_in else np.asarray(input_signals))
        return x3, [x3[i] for i in range(int(x3.shape[0]))]
    return None, [to_float32(c if torch_in else np.asarray(c)) for c in input_signals]


def _sums_pairwise(x) -> bool:
    """True when the single-clip path would sum this signal's squares in numpy's pairwise order (a planar, i.e.
    column-major, stereo signal); the packed batch is C-order, which numpy sums frame by frame."""
    if x.ndim != 2 or x.shape[0] <= 1 or x.shape[1] <= 1:
        return False
    if R.is_torch_tensor(x):
        return x.stride(0) == 1 and x.stride(1) >= x.shape[0]
    xa = R.dense(x)
    return not xa.flags.c_contiguous


def decorrelate_batch(input_signals, decorrelator):
    """Decorrelate many clips in one call: element ``i`` of the result is byte-identical (dtype, shape, bytes) to
    ``decorrelator_i(input_signals[i])``, computed with a fixed number of launches for the whole batch.

    ``input_signals``: a sequence of clips - numpy arrays or CUDA tensors, ``(frames_i, 2)`` or mono ``(frames_i,)``,
    any length including 0, cast per clip with ``to_float32`` - or one equal-length ``(n_clips, frames, 2)`` array or
    CUDA tensor, returned as one ``(n_clips, frames + haas_delay, 2)`` array.  ``decorrelator``: one ``VelvetNoise``,
    or a ``SignalChain`` of a ``VelvetNoise`` alone or followed by an LR ``HaasEffect`` without width, shared by all
    clips, or a sequence of them, one per clip (e.g. the strengths ``optimize_velvet_noise_batch`` found).

    The clips must share ``num_outs == 2``, ``mode``, ``width``, the normaliser (None or ``rms_normalize``), the Haas
    delay and delayed channel, and whether the envelope is the identity ``(1.0,)``; otherwise ``ValueError`` names the
    setting, before any device work.  Numpy in gives numpy out (views into one page-locked block); CUDA tensors in give
    CUDA tensors out, on torch's current stream."""
    is_array = R.is_torch_tensor(input_signals) or isinstance(input_signals, np.ndarray)
    if is_array and input_signals.ndim != 3:
        raise ValueError(f"an array of clips must be (n_clips, frames, 2), got shape {tuple(input_signals.shape)}; pass other clips as a list")
    if is_array and input_signals.shape[2] != 2:
        raise ValueError(f"an array of clips must be (n_clips, frames, 2), got shape {tuple(input_signals.shape)}")
    n = int(input_signals.shape[0]) if is_array else len(input_signals)
    shared = isinstance(decorrelator, (Decorrelator, SignalChain))  # one for all clips (an unsupported one raises below)
    decs = [decorrelator] * n if shared else list(decorrelator)
    if len(decs) != n:
        raise ValueError(f"{len(decs)} decorrelators for {n} clips: pass one decorrelator, or one per clip")

    # decorrelators and the settings they must share
    stages: dict[int, tuple] = {}
    for d in ([decorrelator] if shared else decs):
        if id(d) not in stages:
            stages[id(d)] = _batch_stages(d)
    pairs = [stages[id(d)] for d in decs]
    settings = None
    for vn, haas in (stages.values() if n else []):
        cur = _batch_settings(vn, haas)
        if settings is None:
            settings = cur
            continue
        for key, value in cur.items():
            if value != settings[key]:
                raise ValueError(f"decorrelate_batch needs one {key} for every clip, got {settings[key]!r} and {value!r}")
    if settings is None and shared:
        settings = _batch_settings(*stages[id(decorrelator)])
    if settings is not None and settings["num_outs"] != 2:
        raise ValueError(f"decorrelate_batch decorrelates stereo clips: num_outs must be 2, got {settings['num_outs']}")
    delay = settings["Haas delay"] if settings else 0
    out_f64 = bool(settings and settings["Haas stage"])

    # clips: cast, checked as the single-clip call checks them
    torch_in, device = _batch_device(input_signals, is_array, "decorrelate_batch")
    if torch_in:
        import torch
    x3, clips = _cast_clips(input_signals, is_array, torch_in)
    for (vn, _), x in zip(pairs, clips):
        vn._check_input(x)
    if n == 0:
        dt = np.float64 if out_f64 else np.float32
        if not is_array:
            return []
        if torch_in:
            return torch.empty((0, int(input_signals.shape[1]) + delay, 2), dtype=torch.float64 if out_f64 else torch.float32, device=input_signals.device)
        return np.empty((0, int(input_signals.shape[1]) + delay, 2), dtype=dt)

    # programs: one per distinct (filter, truncation), shared by the clips that use it
    lengths = np.array([int(x.shape[0]) for x in clips], dtype=np.int64)
    offsets = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lengths, out=offsets[1:])
    rows = int(offsets[-1])
    progs, prog_of = _batch_programs([vn for vn, _ in pairs], lengths)
    program = _batch_program(progs)
    _check_batch_layout(offsets, prog_of, len(progs), rows)
    vn0 = pairs[0][0]
    haas_ch = settings["Haas delayed_channel"]
    ep = N.EpilogueStruct(int(settings["mode"] == "MS"), int(vn0.width is not None), float(vn0.width) if vn0.width is not None else 0.0,
                          int(settings["normalizer"] is not None), int(delay), int(haas_ch))
    out_dt = N.VND_F64 if out_f64 else N.VND_F32
    starts = offsets[:-1] + np.arange(n, dtype=np.int64) * delay
    lib = N.lib()

    if torch_in:
        xp = x3.contiguous().view(-1, 2) if is_array else _pack_tensors(clips, rows, device)
        if xp.data_ptr() % 8:  # the kernels load one float32 pair per row
            xp = xp.clone()
        out = torch.empty((rows + n * delay, 2), dtype=torch.float64 if out_f64 else torch.float32, device=device)
        stream = R.torch_stream_ptr(xp)
        with torch.cuda.device(device):
            d_offs = torch.from_numpy(offsets).to(device)
            d_prog_of = torch.from_numpy(prog_of).to(device)
            ps = R.device_program(program, device)
            nbytes = C.c_size_t()
            N.check(lib.vnd_vn_decorrelate_batch_workspace(rows, n, C.byref(ep), C.byref(nbytes)), "vnd_vn_decorrelate_batch_workspace")
            work = torch.empty(max(nbytes.value, 16), dtype=torch.uint8, device=device)
            rc = lib.vnd_vn_decorrelate_batch_dev(xp.data_ptr(), N.VND_F32, rows, d_offs.data_ptr(), n, d_prog_of.data_ptr(), C.byref(ps), C.byref(ep),
                                                  out.data_ptr(), out_dt, work.data_ptr(), nbytes.value, stream)
            if rc == N.VND_EUNSUPPORTED:
                # the filter's halo does not fit the batched kernel: clip by clip through the single-clip device path
                for i in range(n):
                    a, L, o = int(offsets[i]), int(lengths[i]), int(starts[i])
                    _vn_decorrelate_into(xp[a:a + L], out[o:o + L + delay], progs[prog_of[i]], ep, stream)
            else:
                N.check(rc, "vnd_vn_decorrelate_batch_dev")
        results = out.view(n, -1, 2) if is_array else [out[int(o):int(o) + int(L) + delay] for o, L in zip(starts, lengths)]
    else:
        if is_array:
            xp = np.ascontiguousarray(x3).reshape(-1, 2)  # already packed: a view when the input is C-ordered float32
        else:
            xp = R.pinned_empty((rows, 2), np.float32)  # page-locked (within the pool's cap): uploaded by DMA, no staging copy
            _pack_clips(xp, clips, offsets)
        if xp.ctypes.data % 8:  # the kernels load one float32 pair per row
            xp = xp.copy()
        out = R.pinned_empty((rows + n * delay, 2), np.float64 if out_f64 else np.float32)
        ps = program.host_struct()
        N.check(lib.vnd_vn_decorrelate_batch_host(R.HostContext.get().handle, xp.ctypes.data, N.VND_F32, rows, offsets.ctypes.data, n,
                                                  prog_of.ctypes.data, C.byref(ps), C.byref(ep), out.ctypes.data if out.size else None, out_dt),
                "vnd_vn_decorrelate_batch_host")
        results = out.reshape(n, -1, 2) if is_array else [out[o:o + L + delay] for o, L in zip(starts, lengths)]

    if settings["normalizer"] is not None:
        # numpy sums a column-major clip pairwise, not frame by frame: such clips keep the single-clip path's order
        for i, ((vn, haas), x) in enumerate(zip(pairs, clips)):
            if _sums_pairwise(x):
                y = vn._decorrelate(x, haas)
                if torch_in:
                    results[i].copy_(y)
                else:
                    results[i][...] = y
    return results


def _vn_decorrelate_into(x32, out, program: TapProgram, ep, stream) -> None:
    """vnd_vn_decorrelate_dev of one packed (frames, 2) float32 clip into a slice of a batch's output tensor."""
    import torch

    lib = N.lib()
    nbytes = C.c_size_t()
    N.check(lib.vnd_vn_decorrelate_workspace(x32.shape[0], 2, C.byref(ep), C.byref(nbytes)), "vnd_vn_decorrelate_workspace")
    work = torch.empty(max(nbytes.value, 16), dtype=torch.uint8, device=x32.device)
    sx, so = R.torch_signal(x32), R.torch_signal(out)
    ps = R.device_program(program, x32.device)
    N.check(lib.vnd_vn_decorrelate_dev(C.byref(sx), C.byref(so), C.byref(ps), C.byref(ep), work.data_ptr(), nbytes.value, stream),
            "vnd_vn_decorrelate_dev")


def _haas_table(haases: "Sequence[HaasEffect]", clips, shared: bool) -> np.ndarray:
    """The ``vnd_haas_clip`` record of every clip (``N.HAAS_CLIP_DTYPE``), checked as ``HaasEffect.decorrelate`` checks
    its clip: the first clip the single call would reject raises that call's exception, with the clip's index.  The
    attributes of the effects and the shapes of the clips are read once each; the rest is vectorised."""
    n = len(clips)
    src = haases[:1] if shared else haases
    delays = np.array([h.delay_len_samples for h in src], dtype=object)
    channels = np.array([h.delayed_channel for h in src], dtype=object)
    mode_ms = np.array([h.mode for h in src], dtype=object) == LayoutMode.MS
    widths = np.array([h.width for h in src], dtype=object)
    use_width = widths != None  # noqa: E711 - elementwise
    ndim = np.fromiter((x.ndim for x in clips), dtype=np.int64, count=n)
    cols = np.fromiter((x.shape[1] if x.ndim == 2 else 2 for x in clips), dtype=np.int64, count=n)
    bad_shape = ((ndim != 1) & (ndim != 2)) | (cols != 2)
    bad_channel = np.broadcast_to(~np.isin(channels, (0, 1, -1, -2)), (n,))
    bad_delay = np.broadcast_to((delays < 0) | (delays >= 2**31), (n,))
    bad = np.flatnonzero(bad_shape | bad_channel | bad_delay)
    if bad.size:
        i = int(bad[0])
        try:
            haases[i]._check(clips[i])
        except (ValueError, IndexError) as e:
            raise type(e)(f"clip {i}: {e}") from None
        raise ValueError(f"clip {i}: the Haas delay of {haases[i].delay_len_samples} frames must lie in [0, 2**31)")
    table = np.zeros(n, dtype=N.HAAS_CLIP_DTYPE)
    table["delay"] = delays.astype(np.int64)
    table["delayed_channel"] = channels.astype(np.int64) % 2
    table["mode_ms"] = mode_ms
    table["mono"] = ndim == 1
    table["use_width"] = use_width
    table["width"] = np.where(use_width, widths, 0.0).astype(np.float64)
    return table


def _haas_offsets(lengths: np.ndarray, delays: np.ndarray) -> "tuple[np.ndarray, np.ndarray]":
    """``(frame_offsets, out_offsets)`` of a packed Haas batch: clip ``i`` is input rows ``[frame_offsets[i],
    frame_offsets[i + 1])`` and output rows from ``out_offsets[i] = frame_offsets[i] + sum_{j < i} delays[j]``."""
    n = len(lengths)
    offsets = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(lengths, out=offsets[1:])
    _check_offsets(offsets, n, int(offsets[-1]))
    out_offsets = offsets[:-1].copy()
    out_offsets[1:] += np.cumsum(delays[:-1], dtype=np.int64)
    return offsets, out_offsets


def _packed_base(clips, offsets: np.ndarray, torch_in: bool) -> "int | None":
    """The address of row 0 when the clips are already consecutive row ranges of one C-order (rows, 2) float32 buffer
    (e.g. the views ``decorrelate_batch`` returns without a Haas stage), else None.  Only the clips' own rows are read
    from it, so the clips may come from separate allocations as long as their addresses line up."""
    n = len(clips)
    if torch_in:
        import torch

        if not all(x.dtype == torch.float32 and x.ndim == 2 and x.shape[1] == 2 and x.stride(1) == 1 and (x.shape[0] <= 1 or x.stride(0) == 2)
                   for x in clips):
            return None
        ptrs = np.fromiter((x.data_ptr() for x in clips), dtype=np.int64, count=n)
    else:
        if not all(x.dtype == np.float32 and x.ndim == 2 and x.shape[1] == 2 and x.strides[1] == 4 and (x.shape[0] <= 1 or x.strides[0] == 8)
                   for x in clips):
            return None
        ptrs = np.fromiter((x.ctypes.data for x in clips), dtype=np.int64, count=n)
    used = np.diff(offsets) > 0
    if not used.any():
        return None
    starts = offsets[:-1][used]
    base = int(ptrs[used][0] - 8 * starts[0])
    if base % 8 or not np.array_equal(ptrs[used], base + 8 * starts):
        return None
    return base


def haas_effect_batch(input_signals, haas_effect):
    """Apply the Haas effect to many clips in one call: element ``i`` of the result is byte-identical (dtype float64,
    shape, bytes) to ``haas_effect_i.decorrelate(input_signals[i])``, computed with one launch for the whole batch.

    ``input_signals``: a sequence of clips - numpy arrays or CUDA tensors, ``(frames_i, 2)`` or mono ``(frames_i,)``,
    any length including 0, cast per clip with ``to_float32`` - or one ``(n_clips, frames, 2)`` array or CUDA tensor,
    returned as one ``(n_clips, frames + delay, 2)`` array (its clips must then share one delay).  ``haas_effect``: one
    ``HaasEffect`` shared by all clips, or a sequence with one per clip (e.g. with the delays
    ``optimize_haas_delay_batch`` found); each clip's delay, delayed channel, mode and width are its own.

    Every error is raised before any device work, with the index of the clip it concerns.  Numpy in gives numpy out
    (views into one page-locked block); CUDA tensors in give CUDA tensors out (views into one tensor), on torch's
    current stream.  Clips that already are consecutive rows of one (rows, 2) float32 buffer, such as the output of
    ``decorrelate_batch`` without a Haas stage, are read in place."""
    is_array = R.is_torch_tensor(input_signals) or isinstance(input_signals, np.ndarray)
    if is_array and (input_signals.ndim != 3 or input_signals.shape[2] != 2):
        raise ValueError(f"an array of clips must be (n_clips, frames, 2), got shape {tuple(input_signals.shape)}; pass other clips as a list")
    n = int(input_signals.shape[0]) if is_array else len(input_signals)
    shared = isinstance(haas_effect, HaasEffect)
    haases = [haas_effect] * n if shared else list(haas_effect)
    if len(haases) != n:
        raise ValueError(f"{len(haases)} Haas effects for {n} clips: pass one HaasEffect, or one per clip")
    if not all(isinstance(h, HaasEffect) for h in (haases[:1] if shared else haases)):
        raise TypeError("haas_effect_batch takes a HaasEffect or a sequence of them")
    torch_in, device = _batch_device(input_signals, is_array, "haas_effect_batch")
    if torch_in:
        import torch
    raw = input_signals if is_array or torch_in else [np.asarray(c) for c in input_signals]
    table = _haas_table(haases, [raw[i] for i in range(n)], shared)
    delays = table["delay"].astype(np.int64)
    if is_array and n and np.any(delays != delays[0]):
        raise ValueError("the clips of an (n_clips, frames, 2) array need one Haas delay; pass clips with different delays as a list")
    if n == 0:
        if not is_array:
            return []
        shape = (0, int(input_signals.shape[1]) + (haas_effect.delay_len_samples if shared else 0), 2)
        return torch.empty(shape, dtype=torch.float64, device=input_signals.device) if torch_in else np.empty(shape, dtype=np.float64)

    x3, clips = _cast_clips(raw, is_array, torch_in)
    lengths = np.fromiter((x.shape[0] for x in clips), dtype=np.int64, count=n)
    offsets, out_offsets = _haas_offsets(lengths, delays)
    rows, out_rows = int(offsets[-1]), int(offsets[-1] + delays.sum())
    lib = N.lib()

    keep = None  # the packed input, when the clips are packed here
    if torch_in:
        if is_array:
            keep = x3.contiguous().view(-1, 2)
            base = keep.data_ptr()
        else:
            base = _packed_base(clips, offsets, True)
            if base is None:
                keep = _pack_tensors(clips, rows, device)
                base = keep.data_ptr()
        if base % 8:  # the kernel loads one float32 pair per row
            keep = keep.clone()
            base = keep.data_ptr()
        out = torch.empty((out_rows, 2), dtype=torch.float64, device=device)
        with torch.cuda.device(device):
            meta = torch.from_numpy(np.concatenate([table.view(np.int64), offsets, out_offsets])).to(device)
            m = meta.data_ptr()
            N.check(lib.vnd_haas_batch_dev(base if rows else None, rows, m + 32 * n, n, m, m + 32 * n + 8 * (n + 1), out_rows,
                                           out.data_ptr() if out_rows else None, R.torch_stream_ptr(out)), "vnd_haas_batch_dev")
        results = out.view(n, -1, 2) if is_array else [out[int(o):int(o) + int(L) + int(d)] for o, L, d in zip(out_offsets, lengths, delays)]
    else:
        if is_array:
            keep = np.ascontiguousarray(x3).reshape(-1, 2)  # already packed: a view when the input is C-ordered float32
            base = keep.ctypes.data
        else:
            base = _packed_base(clips, offsets, False)
            if base is None:
                keep = R.pinned_empty((rows, 2), np.float32)  # page-locked (within the pool's cap): uploaded by DMA, no staging copy
                _pack_clips(keep, clips, offsets)
                base = keep.ctypes.data
        out = R.pinned_empty((out_rows, 2), np.float64)
        N.check(lib.vnd_haas_batch_host(R.HostContext.get().handle, base if rows else None, rows, offsets.ctypes.data, n, table.ctypes.data,
                                        out.ctypes.data if out_rows else None), "vnd_haas_batch_host")
        results = out.reshape(n, -1, 2) if is_array else [out[o:o + L + d] for o, L, d in zip(out_offsets, lengths, delays)]
    return results


# ------------------------------------------------------------------------------------------------
# live signals, block by block
# ------------------------------------------------------------------------------------------------


def _live_step(blocks, final, n: int, device, who: str):
    """``(blocks, fin, is_t, given, torch_in)`` of one step of ``n`` live signals: one block or None per signal (``given``:
    the signals with a block), all numpy or all CUDA tensors on ``device`` when it is set, and ``final`` as one bool
    per signal (``fin``).  Raises, naming the signal, before any device work."""
    blocks = list(blocks)
    if len(blocks) != n:
        raise ValueError(f"{len(blocks)} blocks for {n} signals: pass one block (or None) per signal")
    if isinstance(final, (bool, np.bool_)):
        fin = np.full(n, bool(final))
    else:
        fin = np.array([bool(f) for f in final], dtype=bool)
        if fin.size != n:
            raise ValueError(f"{fin.size} final flags for {n} signals: pass one bool, or one per signal")
    is_t = [R.is_torch_tensor(b) for b in blocks]
    given = [i for i, b in enumerate(blocks) if b is not None]
    torch_in = bool(given) and is_t[given[0]]
    for i in given:
        if is_t[i] != torch_in:
            raise ValueError(f"signal {i}: the blocks of one step must be all numpy arrays or all CUDA tensors")
    if torch_in:
        for i in given:
            if not blocks[i].is_cuda:
                raise N.VndError(N.VND_EUNSUPPORTED, who,
                                 f"signal {i}: CPU torch tensors are not supported (no CPU fallback); pass CUDA tensors or numpy arrays")
        device = device if device is not None else blocks[given[0]].device
        import torch

        device = torch.device(device)
        for i in given:
            if blocks[i].device != device:
                raise ValueError(f"signal {i}: the block is on {blocks[i].device}, this {who} on {device}")
    return blocks, fin, is_t, given, torch_in


def _live_device(clips, torch_in: bool, device):
    """The torch device a step runs on: its tensors', else the object's, else torch's current one."""
    import torch

    if torch_in:
        return next(x.device for x in clips if R.is_torch_tensor(x))
    return torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")


def _live_results(out, out_offsets: np.ndarray, torch_in: bool, launched: bool, stream):
    """Each signal's rows of a step's output ``out``: views of it for tensor input, else views of one page-locked copy,
    complete when this returns."""
    import torch

    bounds = zip(out_offsets[:-1].tolist(), out_offsets[1:].tolist())
    if torch_in:
        return [out[a:b] for a, b in bounds]
    host = R.pinned_empty(tuple(out.shape), np.float64 if out.dtype == torch.float64 else np.float32)
    if out.shape[0]:
        torch.from_numpy(host).copy_(out, non_blocking=True)
    if launched:
        stream.synchronize()  # the output is read, and the page-locked input may be reused, from here on
    return [host[a:b] for a, b in bounds]


class BlockStepPlan:
    """What one step of live signals does (``plan_block_step``), per signal: ``total`` frames received after the step,
    ``ready`` frames emitted after it, ``out_offsets`` (n + 1) of the step's outputs - signal ``i`` emits its frames
    ``[emitted[i], ready[i])`` -, ``history_start``, the first frame of the history the step leaves (``total - H``), and
    the ``(received, emitted)`` state the next step starts from: zero for a signal whose step was final."""

    __slots__ = ("total", "ready", "out_offsets", "history_start", "next_received", "next_emitted")

    def __init__(self, total, ready, out_offsets, history_start, next_received, next_emitted):
        self.total, self.ready, self.out_offsets = total, ready, out_offsets
        self.history_start, self.next_received, self.next_emitted = history_start, next_received, next_emitted


def plan_block_step(received, emitted, lengths, final, latency, tail, history: int) -> BlockStepPlan:
    """The step planner of ``BlockDecorrelator``, vectorised over signals (int64 arrays, ``final`` bool).  A signal that
    has received ``T`` frames has emitted ``max(0, T - latency)`` of them after a non-final step, and ``T + tail`` after
    its final step; ``latency`` is the filter's look-ahead ``A`` (0 for the Haas effect alone) and ``tail`` the Haas
    delay ``d`` (0 for velvet noise alone)."""
    total = received + lengths
    ready = np.where(final, total + tail, np.maximum(total - latency, 0))
    out_offsets = np.zeros(len(total) + 1, dtype=np.int64)
    np.cumsum(ready - emitted, out=out_offsets[1:])
    zero = np.zeros_like(total)
    return BlockStepPlan(total, ready, out_offsets, total - history, np.where(final, zero, total), np.where(final, zero, ready))


def _block_stages(d) -> "tuple[VelvetNoise | None, HaasEffect | None]":
    """The (velvet noise, Haas) stages a live decorrelator runs as, either of them None."""
    if isinstance(d, VelvetNoise):
        vn, haas = d, None
    elif isinstance(d, HaasEffect):
        vn, haas = None, d
    elif isinstance(d, SignalChain):
        d._init_decorrelators()
        stages = d._decorrelators
        kinds = tuple(type(st) for st in stages)
        if kinds == (VelvetNoise,):
            vn, haas = stages[0], None
        elif kinds == (HaasEffect,):
            vn, haas = None, stages[0]
        elif kinds == (VelvetNoise, HaasEffect):
            vn, haas = stages
        else:
            names = ", ".join(getattr(st, "__name__", type(st).__name__) for st in stages) or "no stages"
            raise NotImplementedError(f"BlockDecorrelator runs a SignalChain of [VelvetNoise], [HaasEffect] or [VelvetNoise, HaasEffect]; "
                                      f"this chain has {names}")
    else:
        raise NotImplementedError(f"BlockDecorrelator takes VelvetNoise, HaasEffect or SignalChain decorrelators, not {type(d).__name__}")
    if vn is not None and vn.normalizer is not None:
        raise NotImplementedError("rms_normalize and other normalisers scale by statistics of the whole signal, which a block cannot know; "
                                  "pass normalizer=None to the VelvetNoise")
    return vn, haas


_STEREO0 = np.empty((0, 2), np.float32)


class BlockDecorrelator:
    """Decorrelates ``n_signals`` live signals that arrive block by block, one launch per step for all of them (two for a
    velvet-noise + Haas chain).

    ``decorrelator``: one ``VelvetNoise`` with ``normalizer=None``, ``HaasEffect``, or ``SignalChain`` of
    ``[VelvetNoise]``, ``[HaasEffect]`` or ``[VelvetNoise, HaasEffect]``, shared by all signals, or a sequence with one
    per signal.  Velvet-noise filters of different signals must share what ``decorrelate_batch`` needs them to share
    (``ValueError`` otherwise); Haas settings are each signal's own.

    ``process(blocks, final=False)`` takes one block per signal - a numpy array or CUDA tensor, ``(frames, 2)`` or mono
    ``(frames,)``, any dtype ``to_float32`` accepts, or None / empty for a signal that received nothing - and returns one
    output per signal.  Concatenating signal ``i``'s outputs up to and including its final step gives the bytes (dtype,
    shape and values) of ``decorrelator_i(np.concatenate(its blocks))``, however the input was cut.  After its final step
    a signal starts over.

    Latency: with ``A_i = latency_frames[i]`` (the filter's largest tap index; 0 for the Haas effect alone), ``d_i`` the
    Haas delay and ``T_i`` the frames received, a signal has emitted ``max(0, T_i - A_i)`` frames after a non-final step
    (``T_i`` for the Haas effect alone), and ``T_i`` (velvet noise) or ``T_i + d_i`` (Haas, chain) after its final step.
    Outputs are float32 for velvet noise and float64 with a Haas stage, as the one-shot call returns them.  Numpy blocks
    give numpy outputs (views of one page-locked block); CUDA tensors give CUDA tensors, on torch's current stream.
    Every error is raised before any device work and names the signal."""

    def __init__(self, decorrelator, n_signals: int = 1, device=None):
        n = int(n_signals)
        if n < 1:
            raise ValueError(f"n_signals must be at least 1, got {n_signals}")
        shared = isinstance(decorrelator, (Decorrelator, SignalChain)) or not hasattr(decorrelator, "__iter__")  # else one per signal
        decs = [decorrelator] * n if shared else list(decorrelator)
        if len(decs) != n:
            raise ValueError(f"{len(decs)} decorrelators for {n} signals: pass one decorrelator, or one per signal")
        stages: dict[int, tuple] = {}
        for d in ([decorrelator] if shared else decs):
            if id(d) not in stages:
                stages[id(d)] = _block_stages(d)
        pairs = [stages[id(d)] for d in decs]
        kind = (pairs[0][0] is not None, pairs[0][1] is not None)
        for i, (vn, haas) in enumerate(pairs):
            if (vn is not None, haas is not None) != kind:
                raise ValueError(f"signal {i}: every signal needs the same stages (velvet noise, Haas effect or both)")
        self.n_signals = n
        self.device = device
        self._vn_stage, self._haas_stage = kind
        self.latency_frames = np.zeros(n, dtype=np.int64)
        self._H_vn = self._H_haas = 0
        if self._vn_stage:
            settings = None
            for i, (vn, _) in enumerate(pairs):
                cur = _batch_settings(vn, None)
                if settings is None:
                    settings = cur
                for key, value in cur.items():
                    if value != settings[key]:
                        raise ValueError(f"signal {i}: BlockDecorrelator needs one {key} for every signal, got {settings[key]!r} and {value!r}")
            if settings["num_outs"] != 2:
                raise ValueError(f"BlockDecorrelator decorrelates stereo signals: num_outs must be 2, got {settings['num_outs']}")
            vns = [vn for vn, _ in pairs]
            progs, self._prog_of = _batch_programs(vns, np.full(n, np.iinfo(np.int64).max))
            self._program = _batch_program(progs)
            self.latency_frames = np.array([max(p.halo - 1, 0) for p in progs], dtype=np.int64)[self._prog_of]
            self._H_vn = int(self.latency_frames.max())
            vn0 = vns[0]
            self._ep = N.EpilogueStruct(int(settings["mode"] == "MS"), int(vn0.width is not None), float(vn0.width) if vn0.width is not None else 0.0,
                                        0, 0, 0)
            ps = self._program.host_struct()
            rc = N.lib().vnd_vn_block_step_dev(None, 0, None, 0, None, None, None, C.byref(ps), C.byref(self._ep), None, None, self._H_vn, None, 0,
                                               None, None)  # no signals: checks the filter, launches nothing
            if rc == N.VND_EUNSUPPORTED:
                raise NotImplementedError(f"a filter reading {self._H_vn} frames ahead does not fit the block-step kernel's shared memory; "
                                          "decorrelate such signals whole")
            N.check(rc, "vnd_vn_block_step_dev")
        self._tail = np.zeros(n, dtype=np.int64)
        if self._haas_stage:
            haases = [h for _, h in pairs]
            self._table = _haas_table(haases, [_STEREO0] * n, shared)
            self._tail = self._table["delay"].astype(np.int64)
            self._H_haas = int(self._tail.max())
        self._received = np.zeros(n, dtype=np.int64)
        self._emitted = np.zeros(n, dtype=np.int64)
        self._mono = np.full(n, -1, dtype=np.int8)  # -1: not known yet (no frame since the signal started)
        self._dev = None  # device state, made at the first launch

    # ---- host side ------------------------------------------------------------------------------
    def _blocks(self, blocks, final):
        """``(torch_in, clips, lengths, final, mono)`` of one step, every check done; no device work."""
        n = self.n_signals
        blocks, fin, is_t, given, torch_in = _live_step(blocks, final, n, self.device, "BlockDecorrelator")
        clips = [_STEREO0 if b is None else to_float32(b if t else np.asarray(b)) for b, t in zip(blocks, is_t)]
        for i in given:
            x = clips[i]
            if x.ndim not in (1, 2) or (x.ndim == 2 and x.shape[1] != 2):
                raise ValueError(f"signal {i}: a block must be (frames, 2) or mono (frames,), got shape {tuple(x.shape)}")
        lengths = np.fromiter((x.shape[0] for x in clips), dtype=np.int64, count=n)
        mono = np.fromiter((x.ndim == 1 for x in clips), dtype=np.int8, count=n)
        clash = (lengths > 0) & (self._mono >= 0) & (mono != self._mono)
        if clash.any():
            i = int(np.flatnonzero(clash)[0])
            was = "mono" if self._mono[i] else "stereo"
            raise ValueError(f"signal {i}: a {'mono' if mono[i] else 'stereo'} block for a {was} signal; a signal keeps its layout until its final step")
        mono = np.where(lengths > 0, mono, self._mono)
        return torch_in, clips, lengths, fin, mono

    def _device_state(self, device):
        import torch

        if self._dev is None:
            self.device = device
            n = self.n_signals
            st = {"vn": None, "haas": None}
            if self._vn_stage:
                st["vn"] = [torch.zeros((n, self._H_vn, 2), dtype=torch.float32, device=device) for _ in range(2)]
                st["program"] = R.device_program(self._program, device)
                st["prog_of"] = torch.from_numpy(self._prog_of).to(device)
            if self._haas_stage:
                st["haas"] = [torch.zeros((n, self._H_haas, 2), dtype=torch.float32, device=device) for _ in range(2)]
                st["table"] = None
                st["mono"] = None
            self._dev = st
        return self._dev

    # ---- one step -------------------------------------------------------------------------------
    def process(self, blocks, final=False):
        """One step: ``blocks`` has one block (or None) per signal, ``final`` is a bool or one bool per signal.  Returns
        each signal's output frames that became ready in this step (see the class documentation)."""
        torch_in, clips, lengths, fin, mono = self._blocks(blocks, final)
        import torch

        device = _live_device(clips, torch_in, self.device)
        n = self.n_signals
        offsets = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(lengths, out=offsets[1:])
        plan = plan_block_step(self._received, self._emitted, lengths, fin, self.latency_frames, self._tail,
                               self._H_vn if self._vn_stage else self._H_haas)
        # a chain's Haas stage reads the velvet-noise output: its block is what the velvet-noise stage emits in this step
        vn_oo = plan_block_step(self._received, self._emitted, lengths, fin, self.latency_frames, 0, 0).out_offsets if self._vn_stage else None
        rows, out_rows = int(offsets[-1]), int(plan.out_offsets[-1])
        vn_rows = int(vn_oo[-1]) if self._vn_stage else 0
        launch_vn = self._vn_stage and rows + vn_rows > 0
        haas_rows = vn_rows if self._vn_stage else rows
        launch_haas = self._haas_stage and haas_rows + out_rows > 0
        out_dtype = torch.float64 if self._haas_stage else torch.float32

        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device)
            out = torch.empty((0, 2), dtype=out_dtype, device=device)
            if launch_vn or launch_haas:
                st = self._device_state(device)
                tables = [offsets, self._received, self._emitted, plan.out_offsets] + ([vn_oo] if self._vn_stage else [])
                meta = torch.from_numpy(np.concatenate(tables)).to(device)
                m = meta.data_ptr()
                d_offs, d_recv, d_emit, d_oo, d_vn_oo = (m + 8 * k for k in (0, n + 1, 2 * n + 1, 3 * n + 1, 4 * n + 2))
                keep, x_ptr = self._pack(clips, offsets, rows, torch_in, device)
                lib = N.lib()
                y = None
                if launch_vn:
                    y = torch.empty((vn_rows, 2), dtype=torch.float32, device=device)
                    h_in, h_out = st["vn"]
                    N.check(lib.vnd_vn_block_step_dev(x_ptr, rows, d_offs, n, d_recv, d_emit, st["prog_of"].data_ptr(), C.byref(st["program"]),
                                                      C.byref(self._ep), h_in.data_ptr(), h_out.data_ptr(), self._H_vn, d_vn_oo, vn_rows,
                                                      y.data_ptr() if vn_rows else None, stream.cuda_stream), "vnd_vn_block_step_dev")
                    st["vn"] = [h_out, h_in]
                    out = y
                if launch_haas:
                    h_mono = np.zeros(n, np.int32) if self._vn_stage else np.maximum(mono, 0).astype(np.int32)
                    if st["mono"] is None or not np.array_equal(st["mono"], h_mono):  # the records change only with a layout
                        table = self._table.copy()
                        table["mono"] = h_mono
                        st["table"], st["mono"] = torch.from_numpy(table.view(np.uint8)).to(device), h_mono
                    if self._vn_stage:
                        hx, h_offs, h_recv = (y.data_ptr() if vn_rows else None), d_vn_oo, d_emit
                    else:
                        hx, h_offs, h_recv = x_ptr, d_offs, d_recv
                    out = torch.empty((out_rows, 2), dtype=torch.float64, device=device)
                    h_in, h_out = st["haas"]
                    N.check(lib.vnd_haas_block_step_dev(hx, haas_rows, h_offs, n, h_recv, st["table"].data_ptr(), h_in.data_ptr(), h_out.data_ptr(),
                                                        self._H_haas, d_oo, out_rows, out.data_ptr() if out_rows else None, stream.cuda_stream),
                            "vnd_haas_block_step_dev")
                    st["haas"] = [h_out, h_in]
            results = _live_results(out, plan.out_offsets, torch_in, launch_vn or launch_haas, stream)
        self._received, self._emitted = plan.next_received, plan.next_emitted
        self._mono = np.where(fin, -1, mono).astype(np.int8)
        return results

    @staticmethod
    def _pack(clips, offsets, rows: int, torch_in: bool, device):
        """``(keep, address)`` of the step's blocks as one float32 (rows, 2) buffer on the device (a mono block in both
        columns); ``keep`` holds what the address points into.  CUDA blocks that already are consecutive rows of one
        buffer are read in place."""
        import torch

        if not rows:
            return None, None
        if torch_in:
            empty = torch.empty((0, 2), dtype=torch.float32, device=device)
            ts = [x if R.is_torch_tensor(x) else empty for x in clips]
            base = _packed_base(ts, offsets, True)
            if base is not None:
                return ts, base
            xp = _pack_tensors(ts, rows, device)
            if xp.data_ptr() % 8:  # the kernels load one float32 pair per row
                xp = xp.clone()
            return xp, xp.data_ptr()
        xh = R.pinned_empty((rows, 2), np.float32)  # page-locked: uploaded by DMA
        _pack_clips(xh, clips, offsets)
        xp = torch.from_numpy(xh).to(device, non_blocking=True)
        return (xh, xp), xp.data_ptr()


class BlockConvolver:
    """Convolves ``n_signals`` live multichannel signals that arrive block by block with their velvet-noise filters, one
    launch per step for all signals and channels: the streaming form of ``VelvetNoise.convolve``.

    ``filters``: one ``VelvetNoise`` shared by all signals, or a sequence with one per signal.  They must share
    ``num_outs`` and whether the envelope is the identity ``(1.0,)`` (``ValueError`` naming the signal otherwise);
    ``mode``, ``width`` and ``normalizer`` are ignored, as ``convolve`` ignores them.

    ``process(blocks, final=False)`` takes one block per signal - a 2-D numpy array or CUDA tensor ``(frames, >=
    num_outs)`` of any dtype ``convolve`` accepts, or None for a signal that received nothing - and returns one float32
    ``(frames, num_outs)`` output per signal.  Concatenating signal ``i``'s outputs up to and including its final step
    gives the bytes (dtype, shape and values) of ``filters_i.convolve(np.concatenate(its blocks))``, however the input
    was cut.  After its final step a signal starts over.  Only the first ``num_outs`` columns are read; a signal keeps
    its column count until its final step, as ``np.concatenate`` requires.

    Latency: with ``A_i = latency_frames[i]`` (the filter's largest tap index) and ``T_i`` the frames received, a signal
    has emitted ``max(0, T_i - A_i)`` frames after a non-final step and ``T_i`` after its final step.

    Arithmetic: the compute dtype of ``convolve`` - float32 for float32, float16 and integers of up to 2 bytes, float64
    for float64 and wider integers.  The first non-empty block fixes it for the object, and a block of the other compute
    dtype raises ``ValueError``: the concatenation of both would run in float64, which the steps already emitted did not.
    Numpy blocks give numpy outputs (views of one page-locked block); CUDA tensors give CUDA tensors, on torch's current
    stream.  Every error is raised before any device work and names the signal."""

    def __init__(self, filters, n_signals: int = 1, device=None):
        n = int(n_signals)
        if n < 1:
            raise ValueError(f"n_signals must be at least 1, got {n_signals}")
        shared = isinstance(filters, VelvetNoise) or not hasattr(filters, "__iter__")
        if shared and not isinstance(filters, VelvetNoise):
            raise TypeError(f"BlockConvolver takes a VelvetNoise, or one per signal, not {type(filters).__name__}")
        vns = [filters] * n if shared else list(filters)
        if len(vns) != n:
            raise ValueError(f"{len(vns)} filters for {n} signals: pass one VelvetNoise, or one per signal")
        for i, vn in enumerate(vns):
            if not isinstance(vn, VelvetNoise):
                raise TypeError(f"signal {i}: BlockConvolver takes VelvetNoise filters, not {type(vn).__name__}")
        settings = [(vn.num_outs, vn.segment_envelope == IDENTITY_ENVELOPE) for vn in (vns[:1] if shared else vns)]
        for i, cur in enumerate(settings):
            for key, a, b in zip(("num_outs", "identity segment_envelope"), settings[0], cur):
                if a != b:
                    raise ValueError(f"signal {i}: BlockConvolver needs one {key} for every signal, got {a!r} and {b!r}")
        self.n_signals = n
        self.device = device
        self.num_outs = int(settings[0][0])
        progs, self._prog_of = _batch_programs(vns, np.full(n, np.iinfo(np.int64).max))
        self._program = _batch_program(progs)
        self.latency_frames = np.array([max(p.halo - 1, 0) for p in progs], dtype=np.int64)[self._prog_of]
        self._H = int(self.latency_frames.max())
        ps = self._program.host_struct()
        N.check(N.lib().vnd_fir_block_step_dev(None, N.VND_F32, 0, self.num_outs, None, 0, None, None, None, C.byref(ps), None, None, self._H,
                                               None, 0, None, None), "vnd_fir_block_step_dev")  # no signals: checks the filter only
        self._received = np.zeros(n, dtype=np.int64)
        self._emitted = np.zeros(n, dtype=np.int64)
        self._cols = np.full(n, -1, dtype=np.int64)  # -1: not known yet (no block since the signal started)
        self._dtype = None  # the compute dtype, numpy's; fixed by the first non-empty block
        self._dev = None  # device state, made at the first launch

    def _blocks(self, blocks, final):
        """``(torch_in, blocks, lengths, final, cols, dtype)`` of one step, every check done; no device work."""
        n, k = self.n_signals, self.num_outs
        blocks, fin, is_t, given, torch_in = _live_step(blocks, final, n, self.device, "BlockConvolver")
        if not torch_in:
            blocks = [None if b is None else np.asarray(b) for b in blocks]
        cols = self._cols.copy()
        dtype = self._dtype
        for i in given:
            x = blocks[i]
            if x.ndim != 2:  # convolve's exceptions (decorrelation.py:393-415)
                raise IndexError(f"signal {i}: too many indices for array: array is {x.ndim}-dimensional, but 2 were indexed")
            if x.shape[1] < k:
                raise IndexError(f"signal {i}: index {x.shape[1]} is out of bounds for axis 1 with size {x.shape[1]}")
            if cols[i] >= 0 and x.shape[1] != cols[i]:
                raise ValueError(f"signal {i}: a block of {x.shape[1]} columns for a signal of {cols[i]}; a signal keeps its column count "
                                 "until its final step")
            cols[i] = x.shape[1]
            dt = np.dtype(str(_fir_tensor_dtype(x)).replace("torch.", "")) if torch_in else _fir_compute_dtype(x.dtype)
            if dtype is None and x.shape[0]:
                dtype = dt
            if dtype is not None and dt != dtype:
                raise ValueError(f"signal {i}: a block computed in {dt} for a BlockConvolver computing in {dtype}; convolve the "
                                 f"concatenation of both in one dtype, or use a BlockConvolver for each")
        lengths = np.array([0 if b is None else int(b.shape[0]) for b in blocks], dtype=np.int64)
        return torch_in, blocks, lengths, fin, cols, dtype

    def process(self, blocks, final=False):
        """One step: ``blocks`` has one block (or None) per signal, ``final`` is a bool or one bool per signal.  Returns
        each signal's output frames that became ready in this step (see the class documentation)."""
        torch_in, blocks, lengths, fin, cols, dtype = self._blocks(blocks, final)
        import torch

        device = _live_device(blocks, torch_in, self.device)
        n, k = self.n_signals, self.num_outs
        offsets = np.zeros(n + 1, dtype=np.int64)
        np.cumsum(lengths, out=offsets[1:])
        plan = plan_block_step(self._received, self._emitted, lengths, fin, self.latency_frames, 0, self._H)
        rows, out_rows = int(offsets[-1]), int(plan.out_offsets[-1])
        launch = rows + out_rows > 0
        with torch.cuda.device(device):
            stream = torch.cuda.current_stream(device)
            out = torch.empty((out_rows, k), dtype=torch.float32, device=device)
            if launch:
                st = self._device_state(device, dtype)
                meta = torch.from_numpy(np.concatenate([offsets, self._received, self._emitted, plan.out_offsets])).to(device)
                m = meta.data_ptr()
                keep, x_ptr = self._pack(blocks, offsets, rows, torch_in, device, dtype)
                h_in, h_out = st["history"]
                N.check(N.lib().vnd_fir_block_step_dev(x_ptr, N.VND_F64 if dtype == np.float64 else N.VND_F32, rows, k, m, n, m + 8 * (n + 1),
                                                       m + 8 * (2 * n + 1), st["prog_of"].data_ptr(), C.byref(st["program"]),
                                                       h_in.data_ptr() if self._H else None, h_out.data_ptr() if self._H else None, self._H,
                                                       m + 8 * (3 * n + 1), out_rows, out.data_ptr() if out_rows else None, stream.cuda_stream),
                        "vnd_fir_block_step_dev")
                st["history"] = [h_out, h_in]
            results = _live_results(out, plan.out_offsets, torch_in, launch, stream)
        self._received, self._emitted = plan.next_received, plan.next_emitted
        self._cols = np.where(fin, -1, cols)
        self._dtype = dtype
        return results

    def _device_state(self, device, dtype):
        import torch

        if self._dev is None:
            self.device = device
            tdt = torch.float64 if dtype == np.float64 else torch.float32
            self._dev = {"history": [torch.zeros((self.n_signals, self._H, self.num_outs), dtype=tdt, device=device) for _ in range(2)],
                         "program": R.device_program(self._program, device), "prog_of": torch.from_numpy(self._prog_of).to(device)}
        return self._dev

    def _pack(self, blocks, offsets, rows: int, torch_in: bool, device, dtype):
        """``(keep, address)`` of the step's blocks as one C-order (rows, num_outs) buffer of the compute dtype on the
        device; ``keep`` holds what the address points into.  The only non-empty block of a step is read in place when it
        already is such a buffer."""
        import torch

        if not rows:
            return None, None
        k = self.num_outs
        full = [b for b in blocks if b is not None and b.shape[0]]
        one = full[0] if len(full) == 1 else None
        if torch_in:
            tdt = torch.float64 if dtype == np.float64 else torch.float32
            if one is not None and one.dtype == tdt and one.shape[1] == k and one.is_contiguous():
                return one, one.data_ptr()
            xp = _pack_tensors(full, rows, device, cols=k, dtype=tdt)
            return xp, xp.data_ptr()
        if one is not None and one.dtype == dtype and one.shape[1] == k and one.flags.c_contiguous:
            xp = torch.from_numpy(one).to(device, non_blocking=True)
            return xp, xp.data_ptr()
        xh = R.pinned_empty((rows, k), dtype)  # page-locked: uploaded by DMA
        _pack_clips(xh, [b if b is not None else np.empty((0, k), dtype) for b in blocks], offsets)
        xp = torch.from_numpy(xh).to(device, non_blocking=True)
        return (xh, xp), xp.data_ptr()


# ------------------------------------------------------------------------------------------------
# function path (decorrelation.py:549-660)
# ------------------------------------------------------------------------------------------------


def generate_velvet_noise(*, duration_seconds: float, num_impulses: int, num_outs: int = 2, sample_rate_hz: int = 44100,
                          segment_envelope: Sequence[float] = (0.85, 0.55, 0.35, 0.2), log_distribution_strength: float = 1.0,
                          seed: int | None = None) -> np.ndarray:
    """Dense float32 ``(int(duration * fs), num_outs)`` velvet-noise FIR for ``convolve_velvet_noise``."""
    return generate_dense_fir(duration_seconds=duration_seconds, num_impulses=num_impulses, num_outs=num_outs, sample_rate_hz=sample_rate_hz,
                              segment_envelope=segment_envelope, log_distribution_strength=log_distribution_strength, seed=seed)


def convolve_velvet_noise(input_signal, velvet_noise_filters):
    """Stateless sparse FIR: for each non-zero of each FIR column in ascending index order,
    ``y[:n - i] += x[i:] * value``; float32 output with the input's shape (decorrelation.py:630-660)."""
    if input_signal.ndim == 1:  # the reference indexes [:, channel] on the 1-D input (decorrelation.py:650)
        raise IndexError("too many indices for array: array is 1-dimensional, but 2 were indexed")
    fir = velvet_noise_filters.detach().cpu().numpy() if R.is_torch_tensor(velvet_noise_filters) else np.asarray(velvet_noise_filters)
    if input_signal.shape[1] > 1:
        check_equal_length(input_signal, fir, dim=1)
    program = ascending_program(fir, input_signal.shape[0])
    return _sparse_fir(input_signal, program, input_signal.shape[1])
