"""ctypes binding of ``libdeepgrp_b200.so`` (C ABI declared in ``include/deepgrp_b200.h``).

There is no CPU fallback: if the shared library is missing, or no sm_100 GPU is visible when a
computation is requested, the call raises.  Loading the library itself needs no GPU (the CPU test
suite checks that every declared symbol is exported).
"""
from __future__ import annotations

import ctypes
import os
import threading
from typing import Dict, Optional

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# DEEPGRP_B200_LIB: an alternative build of the same library (developer builds, e.g. tools/tc_trace.py)
LIB_PATH = os.environ.get("DEEPGRP_B200_LIB") or os.path.join(_HERE, "libdeepgrp_b200.so")

OK, E_CUDA, E_ARG, E_NOGPU, E_ALLN, E_CAPACITY, E_UNSUPPORTED, E_FASTA = 0, -1, -2, -3, -4, -5, -6, -7
COMPAT_REFERENCE, COMPAT_FIXED = 0, 1
MASK_SOFT, MASK_HARD = 0, 1


class DeepgrpError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__("deepgrp_b200 error %d: %s" % (code, message))
        self.code = code


class Seg(ctypes.Structure):       # dgrp_seg_t  (msseg_t of deepgrp/_mss/mss.h:11-14)
    _fields_ = [("st", ctypes.c_int), ("en", ctypes.c_int), ("sc", ctypes.c_double)]


class Row(ctypes.Structure):       # dgrp_row_t
    _fields_ = [("start", ctypes.c_int64), ("end", ctypes.c_int64), ("label", ctypes.c_int32),
                ("record", ctypes.c_int32)]


ROW_DTYPE = np.dtype([("start", np.int64), ("end", np.int64), ("label", np.int32),
                      ("record", np.int32)])
SEG_DTYPE = np.dtype([("st", np.int32), ("en", np.int32), ("sc", np.float64)], align=True)


class Timings(ctypes.Structure):   # dgrp_timings_t
    _fields_ = [("encode_ms", ctypes.c_float), ("forward_ms", ctypes.c_float),
                ("attend_ms", ctypes.c_float), ("score_ms", ctypes.c_float),
                ("mss_ms", ctypes.c_float), ("segments_ms", ctypes.c_float),
                ("total_ms", ctypes.c_float), ("windows", ctypes.c_int64),
                ("bases", ctypes.c_int64), ("kernel_launches", ctypes.c_int64)]


_P = ctypes.c_void_p
_I = ctypes.c_int
_L = ctypes.c_int64
_D = ctypes.c_double
_F = ctypes.c_float
_PL = ctypes.POINTER(ctypes.c_int64)
_PI = ctypes.POINTER(ctypes.c_int)

# name -> (restype, argtypes); every function of include/deepgrp_b200.h
SIGNATURES = {
    "dgrp_version": (_I, []),
    "dgrp_last_error": (ctypes.c_char_p, []),
    "dgrp_device_count": (_I, [_PI]),
    "dgrp_ctx_create": (_I, [_I, ctypes.POINTER(_P)]),
    "dgrp_ctx_destroy": (_I, [_P]),
    "dgrp_ctx_synchronize": (_I, [_P]),
    "dgrp_ctx_stream": (_P, [_P]),
    "dgrp_ctx_timings": (_I, [_P, ctypes.POINTER(Timings)]),
    "dgrp_ctx_launch_count": (_L, [_P]),
    "dgrp_ctx_set_int": (_I, [_P, ctypes.c_char_p, _L]),
    "dgrp_ctx_get_int": (_I, [_P, ctypes.c_char_p, _PL]),
    "dgrp_one_hot_stage": (_I, [_P, _P, _L, _I, _PL, _PL]),
    "dgrp_one_hot_fetch": (_I, [_P, _P]),
    "dgrp_get_max": (_I, [_P, _P, _L, _P, _L, _L, _L, _L]),
    "dgrp_get_max_dev": (_I, [_P, _P, _L, _P, _L, _L, _L, _L]),
    "dgrp_get_segments": (_I, [_P, _P, _L, _L, _P]),
    "dgrp_yield_segments": (_I, [_P, _P, _L, _L, _P, _L, _PL]),
    "dgrp_mss_find_all": (_I, [_P, _I, _P, _D, _D, _P, _L, _PI]),
    "dgrp_find_mss_labels": (_I, [_P, _P, _P, _I, _I, _I, _I, _P]),
    "dgrp_model_create": (_I, [_P, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, ctypes.POINTER(_P)]),
    "dgrp_model_destroy": (_I, [_P]),
    "dgrp_forward_windows": (_I, [_P, _P, _P, _L, _P]),
    "dgrp_predict_onehot": (_I, [_P, _P, _P, _L, _I, _I, _I, _P]),
    "dgrp_apply_mss": (_I, [_P, _P, _I, _I, _I, _I, _P]),
    "dgrp_mss_scores": (_I, [_P, _P, _L, _I, _P, _P]),
    "dgrp_softmax": (_I, [_P, _P, _L, _I, _P]),
    "dgrp_predict_sequence": (_I, [_P, _P, _P, _L, _I, _I, _I, _I, _I, _I, _I, _PL, _PL, _P, _P, _L, _PL]),
    "dgrp_predict_range": (_I, [_P, _P, _P, _L, _L, _L, _L, _L, _I, _I, _I, _P, _P]),
    "dgrp_finish_record": (_I, [_P, _P, _P, _L, _I, _I, _I, _I, _L, _P, _P, _L, _PL]),
    "dgrp_predict_fasta": (_I, [_P, _P, _P, _L, _I, _I, _I, _I, _I, _I, _PL, _PL]),
    "dgrp_predict_fasta_tsv": (_I, [_P, _P, _P, _L, ctypes.c_char_p, _I, _I, _I, _I, _I, _I,
                                    ctypes.POINTER(_P), _PL, _PL, _PL]),
    "dgrp_mask_fasta": (_I, [_P, _P, _L, _P, _L, _I, _P]),
    "dgrp_mask_fasta_last": (_I, [_P, _P, _L, _I, _P]),
    "dgrp_evaluate_last": (_I, [_P, _I, _P, _P, _L, _P]),
    "dgrp_track_last": (_I, [_P, _I, _I, ctypes.POINTER(_P), _PL]),
    "dgrp_fasta_rows": (_I, [_P, _P, _L]),
    "dgrp_fasta_records": (_I, [_P, _P, _P, _P, _P, _L]),
    "dgrp_fasta_record_tsv": (_I, [_P, _P, _P, _P, _L]),
    "dgrp_fasta_index": (_I, [_P, _L, _I, _P, _P, _L, _PL]),
    "dgrp_fasta_stream_plan": (_I, [_L, _I, _I, _L, _I, _I, _P, _I, _PI]),
    "dgrp_fasta_stream_open": (_I, [_P, _P, _P, _L, ctypes.c_char_p, _I, _I, _I, _I, _I, _I, ctypes.POINTER(_P)]),
    "dgrp_fasta_stream_next": (_I, [_P, ctypes.POINTER(_P), _PL, _PL, _PL, _PL, _PI, _PI]),
    "dgrp_fasta_stream_stats": (_I, [_P, _PL, _PL, _PL, _PL, _PL, _PL, _PL, ctypes.POINTER(_D), ctypes.POINTER(_D)]),
    "dgrp_fasta_stream_waits": (_I, [_P, ctypes.POINTER(_D)]),
    "dgrp_fasta_stream_close": (_I, [_P]),
    "dgrp_predict_codes_dev": (_I, [_P, _P, _P, _L, _I, _I, _I, _I, _I, _I, _PL]),
    "dgrp_predict_codes_dev_results": (_I, [_P, _P, _L, _P, _L]),
    "dgrp_predict_range_dev": (_I, [_P, _P, _P, _L, _L, _L, _L, _L, _I, _I, _I, _P, _P]),
    "dgrp_finish_record_dev": (_I, [_P, _P, _P, _L, _I, _I, _I, _I, _PL]),
    "dgrp_filter_segments": (_I, [_P, _P, _L, _L]),
    "dgrp_confusion_matrix": (_I, [_P, _P, _P, _L, _P]),
    "dgrp_train_create": (_I, [_P, _I, _I, _I, _I, _I, _P, _P, _P, _P, _P, _P, _I, _F, _F, _F, _F, _F,
                               ctypes.POINTER(_P)]),
    "dgrp_train_set_data": (_I, [_P, _I, _P, _P, _L]),
    "dgrp_train_step": (_I, [_P, _P, _P, _L, ctypes.POINTER(_F)]),
    "dgrp_train_eval": (_I, [_P, _I, _P, _L, ctypes.POINTER(_F), _P]),
    "dgrp_train_get_weights": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "dgrp_train_get_grads": (_I, [_P, _P, _P, _P, _P, _P, _P]),
    "dgrp_train_timings": (_I, [_P, _P]),
    "dgrp_train_destroy": (_I, [_P]),
}
OPT_RMSPROP, OPT_ADAM = 0, 1

_lib: Optional[ctypes.CDLL] = None
_lock = threading.Lock()
_contexts: Dict[int, "Context"] = {}


def lib() -> ctypes.CDLL:
    """Load the shared library (raises if it has not been built)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise ImportError(
                        "deepgrp_b200: %s is missing -- build it with `make -C deepgrp_b200/csrc` "
                        "(or __graft_entry__.build()); there is no CPU fallback" % LIB_PATH)
                handle = ctypes.CDLL(LIB_PATH)
                for name, (res, args) in SIGNATURES.items():
                    fn = getattr(handle, name)
                    fn.restype = res
                    fn.argtypes = args
                _lib = handle
    return _lib


def last_error() -> str:
    return lib().dgrp_last_error().decode("utf-8", "replace")


def check(code: int) -> None:
    if code != OK:
        raise DeepgrpError(code, last_error())


def ptr(a: Optional[np.ndarray]) -> ctypes.c_void_p:
    return ctypes.c_void_p(None if a is None else a.ctypes.data)


class Context:
    """One GPU: device id, stream, workspaces (``dgrp_ctx``)."""

    def __init__(self, device: int = 0):
        handle = _P()
        check(lib().dgrp_ctx_create(device, ctypes.byref(handle)))
        self.handle = handle
        self.device = device
        # tuning knobs from the environment: DEEPGRP_KNOBS="forward_tc=0,mss_chunk=4096"
        for item in filter(None, os.environ.get("DEEPGRP_KNOBS", "").split(",")):
            key, _, value = item.partition("=")
            self.set_int(key.strip(), int(value))

    def close(self) -> None:
        if self.handle:
            lib().dgrp_ctx_destroy(self.handle)
            self.handle = None

    def timings(self) -> dict:
        t = Timings()
        check(lib().dgrp_ctx_timings(self.handle, ctypes.byref(t)))
        return {name: getattr(t, name) for name, _ in Timings._fields_}

    def launch_count(self) -> int:
        return int(lib().dgrp_ctx_launch_count(self.handle))

    def set_int(self, key: str, value: int) -> None:
        check(lib().dgrp_ctx_set_int(self.handle, key.encode(), int(value)))

    def get_int(self, key: str) -> int:
        v = ctypes.c_int64(0)
        check(lib().dgrp_ctx_get_int(self.handle, key.encode(), ctypes.byref(v)))
        return int(v.value)

    def synchronize(self) -> None:
        check(lib().dgrp_ctx_synchronize(self.handle))

    def stream(self) -> int:
        return int(lib().dgrp_ctx_stream(self.handle) or 0)


def default_device() -> int:
    for key in ("DEEPGRP_DEVICE", "LOCAL_RANK"):
        if os.environ.get(key, "") != "":
            return int(os.environ[key])
    return 0


def context(device: Optional[int] = None) -> Context:
    """The process-wide context of `device` (created on first use; raises without a B200)."""
    dev = default_device() if device is None else device
    with _lock:
        ctx = _contexts.get(dev)
    if ctx is None:
        ctx = Context(dev)
        with _lock:
            _contexts.setdefault(dev, ctx)
            ctx = _contexts[dev]
    return ctx


def device_count() -> int:
    n = ctypes.c_int(0)
    lib().dgrp_device_count(ctypes.byref(n))
    return int(n.value)
