"""ctypes binding of libacoss_b200.so (the C ABI declared in include/acoss_b200.h).

This is the binding a maintainer of the reference would add (INTEGRATION.md).  There is no CPU
fallback: if the shared library is missing, or no sm_100 device is usable, calls raise.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "csrc", "libacoss_b200.so")

OK, E_INVALID, E_CUDA, E_TOO_SHORT, E_NAN, E_NONBINARY, E_NOMEM = 0, -1, -2, -3, -4, -5, -6
ALIGN_QMAX, ALIGN_SW, ALIGN_DMAX, ALIGN_DMAX_PLAIN = 0, 1, 2, 3
CRP_AUTO, CRP_EXACT = 0, 1


class AcossError(RuntimeError):
    """Raised for every non-zero return code of the C ABI (code in ``.code``)."""

    def __init__(self, code, msg):
        super().__init__("acoss_b200 error %d: %s" % (code, msg))
        self.code = code


class Params(C.Structure):
    """Mirror of ``acoss_params`` (include/acoss_b200.h)."""
    _fields_ = [("m", C.c_int32), ("tau", C.c_int32), ("kappa", C.c_float), ("oti", C.c_int32),
                ("noti", C.c_int32), ("gamma_o", C.c_float), ("gamma_e", C.c_float),
                ("align", C.c_int32), ("integer_guard", C.c_int32), ("crp_path", C.c_int32),
                ("f2_strict", C.c_int32), ("f3_float_acc", C.c_int32), ("f4_keep_last", C.c_int32),
                ("f5_asymmetric", C.c_int32)]


class SimpleParams(C.Structure):
    """Mirror of ``acoss_simple_params`` (include/acoss_b200.h)."""
    _fields_ = [("m", C.c_int32), ("oti", C.c_int32), ("s2_squared", C.c_int32), ("s3_positive", C.c_int32),
                ("s4_roll_first", C.c_int32)]


_lib = None

# name -> (restype, argtypes); every symbol include/acoss_b200.h declares
_vp, _i32p, _i64p, _fp = C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p
SIGNATURES = {
    "acoss_default_params": (None, [C.POINTER(Params)]),
    "acoss_last_error": (C.c_char_p, []),
    "acoss_version": (C.c_char_p, []),
    "acoss_compiled_sm": (C.c_int, []),
    "acoss_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "acoss_destroy": (C.c_int, [_vp]),
    "acoss_set_workspace_limit": (C.c_int, [_vp, C.c_int64]),
    "acoss_set_tracks": (C.c_int, [_vp, _fp, _i64p, C.c_int32, C.c_int]),
    "acoss_set_tracks_raw": (C.c_int, [_vp, _fp, _i64p, C.c_int32, C.c_int32, _i64p]),
    "acoss_get_tracks": (C.c_int, [_vp, _fp, C.c_int64]),
    "acoss_score_pairs": (C.c_int, [_vp, _i32p, C.c_int64, C.POINTER(Params), _fp]),
    "acoss_score_pairs_device": (C.c_int, [_vp, _i32p, C.c_int64, C.POINTER(Params), _fp]),
    "acoss_score_pairs_chen": (C.c_int, [_vp, _i32p, C.c_int64, C.POINTER(Params), _fp, _fp]),
    "acoss_score_pairs_chen_device": (C.c_int, [_vp, _i32p, C.c_int64, C.POINTER(Params), _fp, _fp]),
    "acoss_sync": (C.c_int, [_vp]),
    "acoss_stream": (C.c_void_p, [_vp]),
    "acoss_oti_pairs": (C.c_int, [_vp, _i32p, C.c_int64, C.c_int32, _i32p]),
    "acoss_dump_pair": (C.c_int, [_vp, C.c_int32, C.c_int32, C.POINTER(Params), _i32p, _vp, _fp, _fp, _fp]),
    "acoss_dp_bytes": (C.c_int, [_vp, _vp, _i64p, _i32p, C.c_int64, C.c_int32, C.c_float, C.c_float, _fp]),
    "acoss_knn_sw": (C.c_int, [_vp, _vp, _i64p, _i32p, _i32p, C.c_int64, _fp, _vp]),
    "acoss_last_stats": (C.c_int, [_vp, _i64p]),
    "acoss_debug_counters": (C.c_int, [_vp, _i64p]),
    "acoss_set_profiling": (C.c_int, [_vp, C.c_int]),
    "acoss_stage_ms": (C.c_int, [_vp, _vp]),
    "acoss_kernel_ms": (C.c_int, [_vp, _vp]),
    "acoss_ef_set_tracks": (C.c_int, [_vp, _vp, C.c_int32, _vp, C.c_int32, _vp, C.c_int32, _vp, _i64p, C.c_int32, C.c_int32]),
    "acoss_ef_score_pairs": (C.c_int, [_vp, _i32p, C.c_int64, C.c_double, C.c_int32, _fp]),
    "acoss_ef_dump_pair": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_double, C.c_int32, _i32p, _vp, _vp, _fp]),
    "acoss_ef_stage_ms": (C.c_int, [_vp, _vp]),
    "acoss_ef_last_stats": (C.c_int, [_vp, _i64p]),
    "acoss_set_tracks_pooled": (C.c_int, [_vp, _fp, _i64p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, _i64p]),
    "acoss_simple_default_params": (None, [C.POINTER(SimpleParams)]),
    "acoss_simple_score_pairs": (C.c_int, [_vp, _i32p, C.c_int64, C.POINTER(SimpleParams), _fp]),
    "acoss_simple_score_pairs_device": (C.c_int, [_vp, _i32p, C.c_int64, C.POINTER(SimpleParams), _fp]),
    "acoss_simple_dump_pair": (C.c_int, [_vp, C.c_int32, C.c_int32, C.POINTER(SimpleParams), _i32p, _vp, _i32p, _fp]),
    "acoss_snf": (C.c_int, [_vp, _vp, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_int32,
                            _vp, _fp, _fp, _i32p, _fp]),
    "acoss_snf_stage_ms": (C.c_int, [_vp, _vp]),
}

SNF_MAX_K, SNF_MAX_MATS = 63, 16     # ACOSS_SNF_MAX_K, ACOSS_SNF_MAX_MATS


def load():
    """Load the shared library (once).  Raises if it has not been built: no fallback."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "%s not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(acoss_b200 has no CPU fallback)" % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int):
    if rc != OK:
        raise AcossError(rc, load().acoss_last_error().decode("utf-8", "replace"))


def default_params(**overrides) -> Params:
    p = Params()
    load().acoss_default_params(C.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise TypeError("unknown parameter %r" % k)
        setattr(p, k, v)
    return p


def simple_default_params(**overrides) -> SimpleParams:
    """acoss_simple_default_params (m = 10, oti = 1, S2 = S3 = S4 = 0) with keyword overrides."""
    p = SimpleParams()
    load().acoss_simple_default_params(C.byref(p))
    for k, v in overrides.items():
        if not hasattr(p, k):
            raise TypeError("unknown parameter %r" % k)
        setattr(p, k, int(v))
    return p
