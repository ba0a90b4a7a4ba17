"""ctypes binding of libac_b200.so (the C ABI declared in include/ac_b200.h).

This is the binding a maintainer of the reference would add (INTEGRATION.md).  There is no CPU
fallback: if the library is missing, or the device is not sm_100, calls raise.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_float, c_int, c_int32, c_int64, c_size_t, c_void_p

import torch  # noqa: F401  (loads libcudart.so.12 into the process before the library is opened)

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libac_b200.so")

AC_OK = 0
AC_ERR_INVALID, AC_ERR_UNSUPPORTED, AC_ERR_DEVICE, AC_ERR_CUDA, AC_ERR_WORKSPACE = -1, -2, -3, -4, -5
AC_DT_F32, AC_DT_F16, AC_DT_BF16 = 0, 1, 2
AC_PREC_F16, AC_PREC_BF16, AC_PREC_F16X3, AC_PREC_BF16X3, AC_PREC_F32 = 0, 1, 2, 3, 4
AC_REDUCE_MEAN, AC_REDUCE_MIN = 0, 1

PRECISIONS = {"f16": AC_PREC_F16, "bf16": AC_PREC_BF16, "f16x3": AC_PREC_F16X3, "bf16x3": AC_PREC_BF16X3, "f32": AC_PREC_F32,
              # "r" modes: one tensor-core pass that also records the arg-min + exact fp32 re-evaluation (ac_refine_min_dist)
              "f16r": AC_PREC_F16, "bf16r": AC_PREC_BF16}


class AcLayer(ctypes.Structure):
    _fields_ = [
        ("ptr", c_void_p),
        ("C", c_int32),
        ("H", c_int32),
        ("W", c_int32),
        ("sb", c_int64),
        ("sc", c_int64),
        ("sh", c_int64),
        ("sw", c_int64),
    ]


class AcError(RuntimeError):
    def __init__(self, code: int, what: str):
        self.code = code
        super().__init__(what)


# name -> (restype, argtypes); every symbol of include/ac_b200.h
SIGNATURES = {
    "ac_version": (c_int, []),
    "ac_strerror": (c_char_p, [c_int]),
    "ac_device_ok": (c_int, [c_int]),
    "ac_last_cuda_error": (c_int, []),
    "ac_last_watchdog": (c_int, []),
    "ac_embed_workspace_bytes": (c_size_t, [POINTER(AcLayer), c_int, c_int, c_int, c_int, c_int, c_int]),
    "ac_embed": (
        c_int,
        [POINTER(AcLayer), c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_int,
         c_void_p, c_size_t, c_void_p],
    ),
    "ac_embed_ex": (
        c_int,
        [POINTER(AcLayer), c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_int,
         c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "ac_patchify": (c_int, [c_void_p, c_int, c_int, c_int, c_int, c_int, c_int, c_void_p, POINTER(c_int), c_void_p]),
    "ac_adaptive_pool1d": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "ac_split_operand": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int, c_void_p]),
    "ac_row_norms": (c_int, [c_void_p, c_void_p, c_int, c_int64, c_int, c_void_p, c_void_p]),
    "ac_min_dist_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int, c_int]),
    "ac_min_dist": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
         c_size_t, c_void_p],
    ),
    "ac_min_dist_sym": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
         c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "ac_min_dist_arg": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p,
         c_size_t, c_void_p],
    ),
    "ac_min_dist_sym_arg": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
         c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "ac_refine_min_dist": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p, c_int, c_int,
         c_void_p, c_int, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "ac_min_dist_sym_ex": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
         c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "ac_min_dist_ready": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p,
         c_void_p, c_int, c_void_p, c_size_t, c_void_p],
    ),
    "ac_min_dist_sym_ready": (
        c_int,
        [c_void_p, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_int, c_int,
         c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "ac_reduce_weights_sym_ex": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p]),
    "ac_reduce_weights_ex": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p, c_int, c_void_p, c_void_p]),
    "ac_reduce_weights_sym": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ac_reduce_weights": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_int, c_void_p, c_void_p]),
    "ac_alpha": (c_int, [c_void_p, c_int, c_int, POINTER(c_double), c_int, c_void_p, c_void_p, c_void_p]),
    "ac_weighted_embed": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ac_weighted_embed_multi": (c_int, [c_void_p, c_void_p, c_int, c_int, c_int, c_int, c_void_p, c_void_p]),
    "ac_weighted_embed_from_features_workspace_bytes": (c_size_t, [POINTER(AcLayer), c_int, c_int, c_int]),
    "ac_weighted_embed_from_features": (
        c_int,
        [POINTER(AcLayer), c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float, c_void_p, c_void_p, c_void_p, c_size_t,
         c_void_p],
    ),
    "ac_pairwise_l2": (c_int, [c_void_p, c_int, c_int, c_void_p, c_void_p]),
    "ac_copy_blocks": (c_int, [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
}

_lib = None


def load() -> ctypes.CDLL:
    """Opens libac_b200.so.  Raises (never falls back) when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise AcError(
            AC_ERR_INVALID,
            "libac_b200.so is not built (%s); run `python -m anomaly_clustering_b200.build`. "
            "There is no CPU / PyTorch fallback for this path." % LIB_PATH,
        )
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError here == header/library mismatch
        fn.restype = res
        fn.argtypes = args
    lib.ac_debug_launches.restype = ctypes.c_ulonglong
    lib.ac_debug_launches.argtypes = []
    lib.ac_debug_set.restype = c_int
    lib.ac_debug_set.argtypes = [c_int, c_int]
    _lib = lib
    return lib


def check(code: int, what: str = "") -> None:
    if code == AC_OK:
        return
    lib = load()
    msg = lib.ac_strerror(code).decode()
    if code == AC_ERR_CUDA:
        msg += " [cudaError %d]" % lib.ac_last_cuda_error()
        wd = lib.ac_last_watchdog()
        if wd:
            msg += " [pipeline watchdog fired in wait %d of the tensor-core kernel, see ac_last_watchdog in include/ac_b200.h]" % wd
    raise AcError(code, "%s: %s (%d)" % (what or "libac_b200", msg, code))
