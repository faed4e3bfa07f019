"""ctypes binding of ``libvnd_b200.so`` (``include/vnd_b200.h``).

The library is built in-tree by ``vndecorrelate_b200/csrc/build.sh`` (``__graft_entry__.build()``
runs it).  There is no fallback: if the library is missing, or no CUDA device is present, every
compute entry point raises — a result never silently comes from somewhere else.
"""

from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("VND_B200_LIB") or os.path.join(_HERE, "_lib", "libvnd_b200.so")  # the override is for A/B builds of the kernels
BUILD_SCRIPT = os.path.join(_HERE, "csrc", "build.sh")

VND_OK, VND_EINVAL, VND_ECUDA, VND_EUNSUPPORTED, VND_ENOMEM, VND_EPROGRAM = 0, -1, -2, -3, -4, -5
VND_F32, VND_F64 = 0, 1
ORDER_SEGMENTED, ORDER_ASCENDING, ORDER_ASCENDING_F64 = 0, 1, 2
OBJ_SLOTS, HAAS_SLOTS = 12, 8


class VndError(RuntimeError):
    """A non-zero status from the native library."""

    def __init__(self, status: int, where: str, detail: str):
        self.status = status
        super().__init__(f"{where}: {detail}" if detail else where)


class TapProgramStruct(C.Structure):
    _fields_ = [
        ("words", C.c_void_p),
        ("offsets", C.c_void_p),
        ("n_words", C.c_int64),
        ("channels", C.c_int32),
        ("order", C.c_int32),
        ("apply_gain", C.c_int32),
        ("halo", C.c_int32),
        ("max_channel_words", C.c_int32),
    ]


class SignalStruct(C.Structure):
    _fields_ = [
        ("data", C.c_void_p),
        ("frames", C.c_int64),
        ("channels", C.c_int32),
        ("dtype", C.c_int32),
        ("stride_t", C.c_int64),
        ("stride_c", C.c_int64),
    ]


class EpilogueStruct(C.Structure):
    _fields_ = [
        ("ms_encode", C.c_int32),
        ("use_width", C.c_int32),
        ("width", C.c_double),
        ("rms_normalize", C.c_int32),
        ("haas_delay", C.c_int32),
        ("haas_channel", C.c_int32),
    ]


# vnd_haas_clip, one record per clip of vnd_haas_batch_dev (32 bytes)
HAAS_CLIP_DTYPE = np.dtype([("delay", "<i4"), ("delayed_channel", "<i4"), ("mode_ms", "<i4"), ("mono", "<i4"), ("use_width", "<i4"),
                            ("reserved", "<i4"), ("width", "<f8")])
assert HAAS_CLIP_DTYPE.itemsize == 32

# vnd_vn_stereo_cand, one record per candidate of vnd_vn_stereo_objective_dev (16 bytes)
VN_STEREO_CAND_DTYPE = np.dtype([("ms_encode", "<i4"), ("use_width", "<i4"), ("w_mid", "<f4"), ("w_side", "<f4")])
assert VN_STEREO_CAND_DTYPE.itemsize == 16


# name -> (restype, argtypes); every symbol include/vnd_b200.h declares
_P = C.POINTER
SIGNATURES = {
    "vnd_abi_version": (C.c_int, []),
    "vnd_version": (C.c_char_p, []),
    "vnd_status_string": (C.c_char_p, [C.c_int]),
    "vnd_last_error": (C.c_char_p, []),
    "vnd_device_count": (C.c_int, [_P(C.c_int)]),
    "vnd_sparse_fir_dev": (C.c_int, [_P(SignalStruct), _P(SignalStruct), _P(TapProgramStruct), C.c_void_p]),
    "vnd_vn_decorrelate_workspace": (C.c_int, [C.c_int64, C.c_int32, _P(EpilogueStruct), _P(C.c_size_t)]),
    "vnd_vn_decorrelate_dev": (C.c_int, [_P(SignalStruct), _P(SignalStruct), _P(TapProgramStruct), _P(EpilogueStruct), C.c_void_p, C.c_size_t, C.c_void_p]),
    "vnd_vn_decorrelate_batch_workspace": (C.c_int, [C.c_int64, C.c_int32, _P(EpilogueStruct), _P(C.c_size_t)]),
    "vnd_vn_decorrelate_batch_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, _P(TapProgramStruct),
                                               _P(EpilogueStruct), C.c_void_p, C.c_int32, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vnd_colsumsq_seq_f32_dev": (C.c_int, [_P(SignalStruct), C.c_void_p, C.c_void_p]),
    "vnd_haas_dev": (C.c_int, [_P(SignalStruct), _P(SignalStruct), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_void_p]),
    "vnd_haas_batch_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "vnd_vn_block_step_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, _P(TapProgramStruct),
                                        _P(EpilogueStruct), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "vnd_haas_block_step_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                          C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "vnd_fir_block_step_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                         _P(TapProgramStruct), C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "vnd_stereo_op_dev": (C.c_int, [_P(SignalStruct), _P(SignalStruct), C.c_int32, C.c_double, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vnd_dsp_workspace": (C.c_int, [C.c_int64, _P(C.c_size_t)]),
    "vnd_rms_normalize_dev": (C.c_int, [_P(SignalStruct), C.c_int32, _P(SignalStruct), C.c_int32, C.c_int32, C.c_double, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vnd_peak_normalize_dev": (C.c_int, [_P(SignalStruct), C.c_int32, C.c_int32, C.c_double, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vnd_polar_dev": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.c_size_t, C.c_void_p]),
    "vnd_rms_normalize_host": (C.c_int, [C.c_void_p, _P(SignalStruct), C.c_int32, _P(SignalStruct), C.c_int32, C.c_int32, C.c_double]),
    "vnd_peak_normalize_host": (C.c_int, [C.c_void_p, _P(SignalStruct), C.c_int32, C.c_int32, C.c_double]),
    "vnd_polar_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                 C.c_void_p]),
    "vnd_objective_workspace": (C.c_int, [C.c_int64, C.c_int32, C.c_int32, _P(C.c_size_t)]),
    "vnd_vn_objective_batch_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int64, _P(TapProgramStruct), C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vnd_haas_objective_batch_dev": (C.c_int, [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vnd_haas_objective_pairs_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                               C.c_void_p]),
    "vnd_vn_objective_runs_workspace": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, _P(C.c_size_t)]),
    "vnd_vn_objective_runs_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, _P(TapProgramStruct), C.c_void_p, C.c_void_p,
                                            C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vnd_vn_stereo_objective_workspace": (C.c_int, [C.c_int64, C.c_int32, _P(C.c_size_t)]),
    "vnd_vn_stereo_objective_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _P(TapProgramStruct), C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                              C.c_size_t, C.c_void_p]),
    "vnd_haas_effect_objective_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "vnd_vn_stereo_rms_objective_workspace": (C.c_int, [C.c_int64, C.c_int32, _P(C.c_size_t)]),
    "vnd_vn_stereo_rms_objective_dev": (C.c_int, [C.c_void_p, C.c_int64, C.c_int64, _P(TapProgramStruct), C.c_void_p, C.c_int32, C.c_void_p,
                                                  C.c_void_p, C.c_void_p, C.c_size_t, C.c_void_p]),
    "vnd_ctx_create": (C.c_int, [C.c_int, _P(C.c_void_p)]),
    "vnd_ctx_destroy": (C.c_int, [C.c_void_p]),
    "vnd_host_alloc": (C.c_int, [C.c_size_t, _P(C.c_void_p)]),
    "vnd_ctx_host_alloc": (C.c_int, [C.c_void_p, C.c_size_t, _P(C.c_void_p)]),
    "vnd_host_free": (C.c_int, [C.c_void_p]),
    "vnd_sparse_fir_host": (C.c_int, [C.c_void_p, _P(SignalStruct), _P(SignalStruct), _P(TapProgramStruct)]),
    "vnd_vn_decorrelate_host": (C.c_int, [C.c_void_p, _P(SignalStruct), _P(SignalStruct), _P(TapProgramStruct), _P(EpilogueStruct)]),
    "vnd_vn_decorrelate_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p,
                                                _P(TapProgramStruct), _P(EpilogueStruct), C.c_void_p, C.c_int32]),
    "vnd_haas_host": (C.c_int, [C.c_void_p, _P(SignalStruct), _P(SignalStruct), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double]),
    "vnd_haas_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "vnd_stereo_op_host": (C.c_int, [C.c_void_p, _P(SignalStruct), _P(SignalStruct), C.c_int32, C.c_double]),
    "vnd_vn_objective_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int64, C.c_int64, _P(TapProgramStruct), C.c_void_p]),
    "vnd_haas_objective_batch_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]),
    "vnd_haas_objective_pairs_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                                C.c_void_p]),
    "vnd_vn_objective_runs_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, _P(TapProgramStruct), C.c_void_p,
                                             C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64]),
    "vnd_vn_stereo_objective_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, _P(TapProgramStruct), C.c_void_p, C.c_int32, C.c_void_p]),
    "vnd_haas_effect_objective_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]),
    "vnd_vn_stereo_rms_objective_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int64, _P(TapProgramStruct), C.c_void_p, C.c_int32,
                                                   C.c_void_p, C.c_void_p]),
    "vnd_sparse_fir_stream_host": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, _P(TapProgramStruct), C.c_int32]),
    "vnd_launch_count": (C.c_int64, []),
}

_lib = None
_lock = threading.Lock()


def build(force: bool = False) -> str:
    """Compile the CUDA sources for sm_100a into ``_lib/libvnd_b200.so`` (nvcc cross-compiles
    without a GPU).  Rebuilds when a source is newer than the library."""
    src_dir = os.path.join(_HERE, "csrc")
    sources = [os.path.join(src_dir, f) for f in os.listdir(src_dir)] + [os.path.join(_HERE, "..", "include", "vnd_b200.h")]
    stale = force or not os.path.exists(LIB_PATH) or any(os.path.getmtime(s) > os.path.getmtime(LIB_PATH) for s in sources if os.path.exists(s))
    if stale:
        subprocess.run(["bash", BUILD_SCRIPT], check=True)
    return LIB_PATH


def lib() -> C.CDLL:
    """The loaded library, with argument types set.  Raises if it has not been built."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise VndError(VND_EUNSUPPORTED, "libvnd_b200.so",
                               f"not built at {LIB_PATH}; run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(there is no CPU fallback)")
            handle = C.CDLL(LIB_PATH)
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(handle, name)  # AttributeError here means the header and the library disagree
                fn.restype = res
                fn.argtypes = args
            if handle.vnd_abi_version() != 1:
                raise VndError(VND_EUNSUPPORTED, "libvnd_b200.so", "ABI version mismatch")
            _lib = handle
    return _lib


def check(status: int, where: str) -> None:
    if status != VND_OK:
        l = lib()
        detail = l.vnd_last_error().decode(errors="replace")
        name = l.vnd_status_string(status).decode()
        raise VndError(status, where, f"{name}: {detail}")


def launch_count() -> int:
    return int(lib().vnd_launch_count())
