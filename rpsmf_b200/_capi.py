# -*- coding: utf-8 -*-
"""ctypes binding of libpsmf_b200.so (include/psmf_b200.h).

The CUDA library is the product path: there is no CPU or PyTorch fallback.  A
missing library raises at first use with the build command to run.
"""

from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PSMF_B200_LIB") or os.path.join(_HERE, "libpsmf_b200.so")   # the override is for kernel experiments

F64, F32 = 0, 1
ROBUST, SIMPLIFIED, CUPDATE_VT, FIXED_LAMBDA, LL_STUDENT, NAN_MASK, RHO_VECTOR, GRAD_LINEAR = 1, 2, 4, 16, 32, 64, 128, 256
LOGLIK = 512
DYN_IDENTITY, DYN_COS, DYN_LINEAR, DYN_EXTERNAL = 0, 1, 2, 3
KERNEL_AUTO, KERNEL_DIRECT, KERNEL_STREAM, KERNEL_BATCH = 0, 1, 2, 3
XCHG_NVLINK, XCHG_EXTERNAL = 0, 1
NSCAL = 8
NSCAL_LL, SCAL_NLL, SCAL_LOGPRED = 10, 8, 9      # LOGLIK: the record gains nll_k and log p(y_obs,k | past)
NEVAL = 4
EVAL_SSE, EVAL_INSIDE, EVAL_COUNT = 0, 1, 2
MAILBOX_BLOB_BYTES = 128
SCAL_NAMES = ("a", "eta", "N", "omega", "phi", "sSe", "lam", "rho")

# every symbol include/psmf_b200.h declares (checked by tests/test_host_cpu.py: the header, this tuple and the built library must agree)
EXPORTS = (
    "psmf_create", "psmf_destroy", "psmf_last_error", "psmf_version", "psmf_set_state", "psmf_get_state",
    "psmf_run", "psmf_status", "psmf_launch_info", "psmf_launch_info2", "psmf_set_trace", "psmf_mailbox_export", "psmf_mailbox_connect",
    "psmf_stats_buffer", "psmf_run_finish", "psmf_set_linear_dynamics", "psmf_predict", "psmf_eval_full", "psmf_ingest",
    "psmf_transpose_mask", "psmf_missing_segments", "psmf_count_nan",
)


class PsmfConfig(C.Structure):
    _fields_ = [
        ("d", C.c_int64), ("d_global", C.c_int64), ("r", C.c_int32), ("n_series", C.c_int32),
        ("dtype", C.c_int32), ("flags", C.c_int32), ("dynamics", C.c_int32), ("device", C.c_int32),
        ("world_size", C.c_int32), ("rank", C.c_int32), ("ctas", C.c_int32), ("kernel", C.c_int32),
        ("alpha", C.c_double), ("beta", C.c_double), ("exchange", C.c_int32), ("reserved", C.c_int32),
    ]


class PsmfIO(C.Structure):
    _fields_ = [
        ("Y", C.c_void_p), ("ldy", C.c_int64), ("y_series_stride", C.c_int64),
        ("M", C.c_void_p), ("ldm", C.c_int64), ("m_series_stride", C.c_int64),
        ("X_out", C.c_void_p),
        ("Yrec_out", C.c_void_p), ("ldrec", C.c_int64), ("rec_series_stride", C.c_int64),
        ("scal_out", C.c_void_p),
        ("xbar_ext", C.c_void_p), ("F_ext", C.c_void_p), ("grad_out", C.c_void_p),
        ("Yorig", C.c_void_p), ("E", C.c_void_p), ("lde", C.c_int64), ("e_series_stride", C.c_int64), ("sig", C.c_double),
        ("eval_out", C.c_void_p),
    ]


class PsmfError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("psmf_b200 error %d: %s" % (code, msg))
        self.code = code


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "rpsmf_b200: %s is missing. Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "or `make -C rpsmf_b200/csrc`. There is no CPU fallback." % LIB_PATH)
    L = C.CDLL(LIB_PATH)
    vp, i64, i32 = C.c_void_p, C.c_int64, C.c_int32
    L.psmf_create.argtypes = [C.POINTER(vp), C.POINTER(PsmfConfig)]
    L.psmf_destroy.argtypes = [vp]
    L.psmf_last_error.argtypes = [vp]
    L.psmf_last_error.restype = C.c_char_p
    L.psmf_version.restype = C.c_int
    L.psmf_set_state.argtypes = [vp] + [vp] * 8 + [vp]
    L.psmf_get_state.argtypes = [vp] + [vp] * 8 + [vp]
    L.psmf_run.argtypes = [vp, C.POINTER(PsmfIO), i64, i64, vp]
    L.psmf_status.argtypes = [vp, C.POINTER(i64)]
    L.psmf_launch_info.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.psmf_launch_info2.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.psmf_set_trace.argtypes = [vp, vp, i32]
    L.psmf_mailbox_export.argtypes = [vp, vp]
    L.psmf_mailbox_connect.argtypes = [vp, vp, i32]
    L.psmf_stats_buffer.argtypes = [vp, C.POINTER(vp), C.POINTER(i32)]
    L.psmf_run_finish.argtypes = [vp, C.POINTER(PsmfIO), i64, vp]
    L.psmf_set_linear_dynamics.argtypes = [vp, vp, vp, vp]
    L.psmf_predict.argtypes = [vp, i64, i64, vp, vp, vp, i64, i64, vp]
    L.psmf_eval_full.argtypes = [vp, vp, i64, vp, i64, i64, vp, i64, i64, vp, vp]
    L.psmf_ingest.argtypes = [i32, vp, i64, i64, i32, i32, vp, i64, vp, i64, vp]
    L.psmf_transpose_mask.argtypes = [i32, vp, i64, i64, vp, i64, vp]
    L.psmf_missing_segments.argtypes = [i32, i32, vp, i64, vp, i64, i64, i64, vp, i32, vp, vp]
    L.psmf_count_nan.argtypes = [i32, i32, vp, i64, i64, i64, vp, vp]
    for name in EXPORTS:
        if name not in ("psmf_last_error",):
            getattr(L, name).restype = C.c_int
    L.psmf_last_error.restype = C.c_char_p
    _lib = L
    return L


def check(handle, rc):
    if rc != 0:
        msg = lib().psmf_last_error(handle)
        raise PsmfError(rc, msg.decode() if msg else "unknown")
