"""ctypes binding of libhmmb200.so (include/hmmb200.h) — the only route from the Python
drop-in modules to the CUDA kernels.  There is no CPU fallback: a missing library or a
missing CUDA device raises ``HmmbError`` / ``OSError`` loudly.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Sequence

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libhmmb200.so")

HMMB_OK = 0
ERR_CUDA, ERR_ARG, ERR_OOM, ERR_EMPTY, ERR_RANGE, ERR_UNSUPPORTED = -1, -2, -3, -4, -5, -6

ALLREDUCE_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_int64, ctypes.c_void_p)

# every symbol include/hmmb200.h declares: (name, restype, argtypes)
_c = ctypes
_dp = _c.POINTER(_c.c_double)
_ip = _c.POINTER(_c.c_int32)
_lp = _c.POINTER(_c.c_int64)
SYMBOLS = [
    ("hmmb_init", _c.c_int, [_c.c_int]),
    ("hmmb_shutdown", _c.c_int, []),
    ("hmmb_last_error", _c.c_char_p, []),
    ("hmmb_version", _c.c_char_p, []),
    ("hmmb_device_info", _c.c_int, [_ip, _ip, _ip, _lp]),
    ("hmmb_set_stream", _c.c_int, [_c.c_void_p]),
    ("hmmb_get_stream", _c.c_void_p, []),
    ("hmmb_synchronize", _c.c_int, []),
    ("hmmb_host_alloc", _c.c_void_p, [_c.c_int64]),
    ("hmmb_host_free", _c.c_int, [_c.c_void_p]),
    ("hmmb_launch_count", _c.c_int64, []),
    ("hmmb_phase_ms", _c.c_double, [_c.c_char_p, _lp]),
    ("hmmb_phase_reset", _c.c_int, []),
    ("hmmb_set_profiling", _c.c_int, [_c.c_int]),
    ("hmmb_peak_probe", _c.c_int, [_c.c_int, _dp]),
    ("hmmb_comm_unique_id", _c.c_int, [_c.c_void_p, _c.c_int]),
    ("hmmb_comm_init", _c.c_int, [_c.c_int, _c.c_int, _c.c_void_p]),
    ("hmmb_comm_allreduce", _c.c_int, [_c.c_void_p, _c.c_int64, _c.c_void_p]),
    ("hmmb_comm_rank", _c.c_int, [_ip, _ip]),
    ("hmmb_comm_destroy", _c.c_int, []),
    ("hmmb_vq_encode", _c.c_int, [_c.c_void_p, _c.c_int64, _c.c_void_p, _c.c_int, _c.c_void_p]),
    ("hmmb_vq_encode_dev", _c.c_int, [_c.c_void_p, _c.c_int64, _c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p]),
    ("hmmb_vq_encode_ex", _c.c_int, [_c.c_void_p, _c.c_int64, _c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_int64,
                                     _lp]),
    ("hmmb_lbg_fit", _c.c_int, [_c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _c.c_double, _c.c_void_p,
                                _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
    ("hmmb_lbg_fit_ex", _c.c_int, [_c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _c.c_double, _c.c_void_p,
                                   _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
    ("hmmb_bw_create", _c.c_int, [_c.POINTER(_c.c_void_p), _c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p,
                                  _c.c_int64, _c.c_int, _c.c_int, _c.c_int]),
    ("hmmb_bw_create_ex", _c.c_int, [_c.POINTER(_c.c_void_p), _c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p,
                                     _c.c_int64, _c.c_int, _c.c_int, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p,
                                     _c.c_void_p]),
    ("hmmb_bw_destroy", _c.c_int, [_c.c_void_p]),
    ("hmmb_bw_set_params", _c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
    ("hmmb_bw_set_dist", _c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_void_p]),
    ("hmmb_bw_set_overlap", _c.c_int, [_c.c_void_p, _c.c_int]),
    ("hmmb_bw_iterate", _c.c_int, [_c.c_void_p, _c.c_int, _c.c_double, _c.c_int, _c.c_int]),
    ("hmmb_bw_get_params", _c.c_int, [_c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
    ("hmmb_bw_get_history", _c.c_int, [_c.c_void_p, _c.c_void_p, _c.c_int, _c.c_void_p]),
    ("hmmb_bw_get_seq_ll", _c.c_int, [_c.c_void_p, _c.c_void_p]),
    ("hmmb_bw_total_frames", _c.c_int64, [_c.c_void_p]),
    ("hmmb_bw_kernel_family", _c.c_char_p, [_c.c_void_p]),
    ("hmmb_bw_diagnostics", _c.c_int, [_c.c_void_p, _lp, _lp]),
    ("hmmb_bw_thin_states", _c.c_int, [_c.c_void_p, _lp]),
    ("hmmb_bw_fit", _c.c_int, [_c.c_void_p, _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int,
                               _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_double, _c.c_int, _c.c_void_p,
                               _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
    ("hmmb_mfcc_frames", _c.c_int, [_c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_double, _c.c_void_p]),
    ("hmmb_frames_json_scan", _c.c_int64, [_c.c_char_p, _c.c_int64, _c.c_void_p, _c.c_int64]),
    ("hmmb_score", _c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int64, _c.c_int, _c.c_int, _c.c_int,
                              _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
    ("hmmb_viterbi", _c.c_int, [_c.c_void_p, _c.c_int, _c.c_int, _c.c_void_p, _c.c_int64, _c.c_void_p, _c.c_int, _c.c_int,
                                _c.c_int, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p, _c.c_void_p]),
]


class HmmbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"libhmmb200 error {code}: {msg}")
        self.code = code


_lib = None


def load(build_if_missing: bool = True):
    """Load (and on first use, if absent, build) libhmmb200.so and bind every symbol."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        if not build_if_missing:
            raise OSError(f"{LIB_PATH} not built; run `python -m hmm_training_b200.build`")
        from . import build as _build
        _build.build()
    lib = ctypes.CDLL(LIB_PATH)
    for name, res, args in SYMBOLS:
        fn = getattr(lib, name)  # AttributeError if the .so lacks a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> int:
    if rc < 0:
        msg = load().hmmb_last_error().decode(errors="replace")
        code_to_exc = {ERR_EMPTY: IndexError, ERR_RANGE: IndexError}
        if rc in code_to_exc and "No raw data" not in msg:
            raise code_to_exc[rc](msg)  # same exception class the reference raises
        if rc == ERR_EMPTY:
            raise ValueError(msg)  # codevector_functions.py:445-446
        raise HmmbError(rc, msg)
    return rc


def init(device: Optional[int] = None) -> None:
    check(load().hmmb_init(-1 if device is None else int(device)))


def ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(ctypes.c_void_p)


def c_f64(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float64)


def phase_ms(name: str):
    n = ctypes.c_int64(0)
    ms = load().hmmb_phase_ms(name.encode(), ctypes.byref(n))
    return ms, n.value


def device_info():
    sm, maj, mnr = ctypes.c_int32(), ctypes.c_int32(), ctypes.c_int32()
    mem = ctypes.c_int64()
    check(load().hmmb_device_info(ctypes.byref(sm), ctypes.byref(maj), ctypes.byref(mnr), ctypes.byref(mem)))
    return {"sm_count": sm.value, "cc": (maj.value, mnr.value), "global_mem": mem.value}


def pack_sequences(observations: Sequence[np.ndarray], M: int):
    """List of per-sequence integer arrays -> (obs, offsets int64[R+1]) in the narrowest
    unsigned dtype that holds M-1 (negative codewords are rejected here, as numpy indexing
    with them would silently wrap in the reference)."""
    R = len(observations)
    lens = np.fromiter((len(o) for o in observations), dtype=np.int64, count=R)
    offsets = np.zeros(R + 1, dtype=np.int64)
    np.cumsum(lens, out=offsets[1:])
    if R == 0 or offsets[-1] == 0:
        return np.zeros(0, np.uint8), offsets
    flat = np.concatenate([np.asarray(o).reshape(-1) for o in observations])
    if flat.dtype.kind not in "iu":
        # what numpy says when the reference indexes log_b_matrix[state, obs] with a float (hmm_training.py:353)
        raise IndexError("only integers, slices (`:`), ellipsis (`...`), numpy.newaxis (`None`) and integer or boolean "
                         "arrays are valid indices")
    if flat.dtype.kind == "i" and flat.size and int(flat.min()) < 0:
        raise IndexError("negative codeword index")
    if flat.size and int(flat.max()) >= M:
        raise IndexError(f"index {int(flat.max())} is out of bounds for axis 1 with size {M}")
    dt = np.uint8 if M <= 256 else (np.uint16 if M <= 65536 else np.uint32)
    return np.ascontiguousarray(flat.astype(dt, copy=False)), offsets
