"""ctypes binding of the C ABI declared in include/aware_b200.h.

There is no CPU fallback: importing this module only loads the shared library
(so the symbol table can be checked without a GPU); creating a context without a
CUDA device raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libaware_b200.so")

PREC_TF32, PREC_FP32, PREC_BF16, PREC_FP16 = 0, 1, 2, 3
OPT_THRESHOLD, OPT_EXACT_MARGIN, OPT_TC_SPECTRAL, OPT_TWO_PASS, OPT_PAIR_GEMM, OPT_BWD64_STREAM = 0, 1, 2, 3, 4, 5
STAT_DETECT_CLIPS, STAT_REEVAL_CLIPS = 0, 1
SCALE_NONE, SCALE_SIGNED_MAX = 0, 1


class AwModel(C.Structure):
    _fields_ = [("w", C.POINTER(C.c_float) * 4),
                ("mel_basis", C.POINTER(C.c_float)),
                ("window", C.POINTER(C.c_float)),
                ("band_lo_hz", C.c_float), ("band_hi_hz", C.c_float),
                ("tolerance_db", C.c_float), ("threshold", C.c_float)]


_vp, _i, _i64, _f = C.c_void_p, C.c_int, C.c_int64, C.c_float
_dp = C.POINTER(C.c_double)

COMM_F64, COMM_I64 = 0, 1
COMM_SUM, COMM_MAX = 0, 1
ALLREDUCE_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_int, C.c_int, C.c_void_p)
ALLGATHER_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_int64, C.c_int64, C.c_int64, C.c_void_p)


class AwComm(C.Structure):
    _fields_ = [("user", C.c_void_p), ("allreduce", ALLREDUCE_FN), ("allgather", ALLGATHER_FN),
                ("d_arena", C.c_void_p), ("arena_bytes", C.c_int64), ("rank", C.c_int), ("world", C.c_int)]


# name -> (restype, argtypes); must list every symbol of include/aware_b200.h
SIGNATURES = {
    "aw_last_error": (C.c_char_p, []),
    "aw_version": (C.c_char_p, []),
    "aw_ctx_create": (_i, [C.POINTER(_vp), _i, C.POINTER(AwModel)]),
    "aw_ctx_destroy": (_i, [_vp]),
    "aw_ctx_set_precision": (_i, [_vp, _i]),
    "aw_band_bins": (_i, [_vp, _i, C.POINTER(_i), C.POINTER(_i)]),
    "aw_launch_count": (_i64, [_vp]),
    "aw_ctx_set_option": (_i, [_vp, _i, C.c_double]),
    "aw_ctx_get_stat": (_i, [_vp, _i, C.POINTER(_i64)]),
    "aw_embed_status": (_i, [_vp, _vp, _i, _vp]),
    "aw_profile_enable": (_i, [_vp, _i]),
    "aw_profile_read": (_i, [_vp, _i, C.POINTER(_i), C.POINTER(_i), C.POINTER(_i), C.POINTER(_i),
                             C.POINTER(_i64), _dp]),
    "aw_profile_read_named": (_i, [_vp, _i, C.POINTER(_i), C.c_char_p, C.POINTER(_i64), _dp]),
    "aw_detect_batch": (_i, [_vp, _vp, _i, _i, _i64, _i, _vp, _vp]),
    "aw_embed_batch": (_i, [_vp, _vp, _i, _i, _i64, _i, _vp, _i, _vp, _i, _vp, _i64, _vp, _vp, _i, _vp]),
    "aw_embed_state": (_i, [_vp, _i, _vp, _i64, _vp]),
    "aw_detect_sharded": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, C.POINTER(AwComm), _vp, _vp]),
    "aw_embed_sharded": (_i, [_vp, _vp, _i, _i, _i, _i, _i, _i, _vp, _i, C.POINTER(AwComm), _vp, _i64, _vp, _vp,
                              C.POINTER(_i64), _vp]),
    "aw_decide_and_count": (_i, [_vp, _vp, _vp, _i, _vp, _vp, _vp, _vp]),
    "aw_snr_batch": (_i, [_vp, _vp, _i64, _vp, _i64, _i, _i, _vp, _vp, _vp]),
    "aw_stoi_batch": (_i, [_vp, _vp, _i64, _vp, _i64, _i, _i, _vp, _vp, C.c_double, _vp]),
    "aw_stft_band": (_i, [_vp, _vp, _i, _i, _i64, _i, _i, _vp, _vp, _vp]),
    "aw_istft_band": (_i, [_vp, _vp, _vp, _i, _i, _i, _vp, _vp]),
    "aw_stft_full": (_i, [_vp, _vp, _i, _i, _i64, _vp, _vp]),
    "aw_phase_vocoder": (_i, [_vp, _vp, _i, _i, C.c_double, _i, _vp, _vp]),
    "aw_istft_full": (_i, [_vp, _vp, _i, _i, _i, _vp, _i64, _vp]),
    "aw_gemm": (_i, [_vp, _vp, _vp, _vp, _i, _i, _i, _i, _vp]),
    "aw_attack_pcm": (_i, [_vp, _vp, _i, _i, _i64, _i, _vp, _i64, _vp]),
    "aw_attack_decimate_interp": (_i, [_vp, _vp, _i, _i, _i64, _i, _vp, _i64, _vp]),
    "aw_attack_upfirdn": (_i, [_vp, _vp, _i, _i, _i64, _vp, _i, _i, _i, _i, _i, _vp, _i64, _vp]),
    "aw_attack_lfilter": (_i, [_vp, _vp, _i, _i, _i64, _dp, _dp, _i, _i, _vp, _i64, _vp]),
    "aw_attack_filtfilt": (_i, [_vp, _vp, _i, _i, _i64, _dp, _dp, _dp, _i, _i, _vp, _i64, _vp]),
    "aw_attack_delete": (_i, [_vp, _vp, _i, _i, _i64, _vp, _i, _vp, _i64, _vp]),
    "aw_attack_suppress": (_i, [_vp, _vp, _i, _i, _i64, _vp, _i, _vp, _i64, _vp]),
    "aw_attack_cropout": (_i, [_vp, _vp, _i, _i, _i64, _i, _vp, _i64, _vp]),
    "aw_attack_affine": (_i, [_vp, _vp, _i, _i, _i64, _f, _vp, _i64, _f, _vp, _i64, _vp]),
    "aw_attack_spectral_quantize": (_i, [_vp, _vp, _i, _i, _i, _f, _f, _vp, _vp]),
    "aw_attack_convolve": (_i, [_vp, _vp, _i, _i, _i64, _vp, _i, _i, _vp, _vp, _i64, _vp]),
}

_lib = None


def lib() -> C.CDLL:
    """Load libaware_b200.so (built by __graft_entry__.build()); raise if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                "aware_b200: %s is missing -- build it with `python -c 'import __graft_entry__ as g; "
                "g.build()'`.  There is no CPU fallback." % LIB_PATH)
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)      # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        _lib = handle
    return _lib


class AwareError(RuntimeError):
    pass


def check(status: int) -> None:
    """Map a non-zero status to the exception type the reference raises for it."""
    if status == 0:
        return
    msg = lib().aw_last_error().decode("utf-8", "replace")
    if ("Unsupported PCM" in msg or "must be" in msg or "unsupported" in msg.lower()
            or "bad argument" in msg):
        raise ValueError(msg)
    raise AwareError(msg)
