"""ctypes binding of ``include/uml_b200.h`` (the C ABI of the CUDA library).

The library is built in-tree by :mod:`unionml_b200._build` (``unionml_b200/_lib/libuml_b200.so``).  There is no
CPU fallback: if the library is missing, or no B200 is visible, the product path raises - loudly.
"""
from __future__ import annotations

import ctypes as C
import os
from pathlib import Path

LIB_PATH = Path(__file__).resolve().parent / "_lib" / "libuml_b200.so"

UML_OK, UML_ERR_INVALID, UML_ERR_CUDA, UML_ERR_NONFINITE, UML_ERR_SHAPE = 0, 1, 2, 3, 4
UML_ERR_NOMEM, UML_ERR_UNSUPPORTED, UML_ERR_NO_DEVICE = 5, 6, 7
UML_F32, UML_F64, UML_I64, UML_I32, UML_U8 = 0, 1, 2, 3, 4
UML_STAGE_KEEP_F64, UML_STAGE_SKIP_FINITE_CHECK = 1, 2
UML_PREDICT_FAST, UML_PREDICT_EXACT = 0, 1


class Stats(C.Structure):
    _fields_ = [
        ("n_rows", C.c_int64),
        ("n_flagged", C.c_int64),
        ("n_ambiguous", C.c_int64),
        ("n_nonfinite", C.c_int64),
        ("kernel_ms", C.c_double),
        ("recheck_ms", C.c_double),
        ("total_ms", C.c_double),
        ("h2d_bytes", C.c_int64),
        ("d2h_bytes", C.c_int64),
        ("kernel_launches", C.c_int32),
        ("path", C.c_int32),
    ]

    def as_dict(self) -> dict:
        return {name: getattr(self, name) for name, _ in self._fields_}


class DeviceInfo(C.Structure):
    _fields_ = [
        ("device_id", C.c_int32),
        ("sm_count", C.c_int32),
        ("cc_major", C.c_int32),
        ("cc_minor", C.c_int32),
        ("total_mem_bytes", C.c_int64),
        ("l2_bytes", C.c_int64),
        ("sm_clock_khz", C.c_int32),
        ("mem_clock_khz", C.c_int32),
        ("name", C.c_char * 64),
    ]


# name -> (restype, argtypes); must list every symbol include/uml_b200.h declares (tests/test_abi.py checks that)
_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
SIGNATURES = {
    "uml_abi_version": (C.c_int, []),
    "uml_engine_create": (C.c_int, [_PP, C.c_int]),
    "uml_engine_destroy": (None, [_P]),
    "uml_last_error": (C.c_char_p, [_P]),
    "uml_engine_info": (C.c_int, [_P, C.POINTER(DeviceInfo)]),
    "uml_engine_set_stream": (C.c_int, [_P, _P]),
    "uml_engine_synchronize": (C.c_int, [_P]),
    "uml_host_alloc": (C.c_int, [_P, _PP, C.c_int64]),
    "uml_host_free": (C.c_int, [_P, _P]),
    "uml_device_alloc": (C.c_int, [_P, _PP, C.c_int64]),
    "uml_device_free": (C.c_int, [_P, _P]),
    "uml_linear_load": (C.c_int, [_P, _PP, _P, _P, C.c_int, C.c_int, C.c_int]),
    "uml_model_free": (None, [_P]),
    "uml_linear_set_affine": (C.c_int, [_P, _P, _P, _P]),
    "uml_stage_rows": (C.c_int, [_P, _PP, _P, C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_int, C.c_uint32]),
    "uml_batch_from_device": (C.c_int, [_P, _PP, _P, C.c_int64, C.c_int, C.c_int64]),
    "uml_batch_info": (
        C.c_int,
        [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int), C.POINTER(C.c_int64), _PP, C.POINTER(C.c_int)],
    ),
    "uml_batch_free": (None, [_P]),
    "uml_linear_predict": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.POINTER(Stats)]),
    "uml_linear_predict_peers": (C.c_int, [_P, _P, _P, _PP, C.c_int, C.c_int64, C.c_int, C.c_int, C.POINTER(Stats)]),
    "uml_labels_take": (C.c_int, [_P, _P, C.c_int, C.c_int64, _P, C.c_int, _P]),
    "uml_labels_count_equal": (C.c_int, [_P, _P, C.c_int, C.c_int64, _P, C.c_int, _P, C.POINTER(C.c_int64)]),
    "uml_labels_push": (C.c_int, [_P, _P, _PP, C.c_int, C.c_int64]),
    "uml_linear_predict_host": (
        C.c_int,
        [_P, _P, _P, C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_int, _P, C.c_int, C.c_int64, C.POINTER(Stats)],
    ),
    "uml_linear_predict_host_values": (
        C.c_int,
        [_P, _P, _P, C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_int, _P, C.c_int, _P, C.c_int, C.c_int64, C.POINTER(Stats)],
    ),
    "uml_linear_predict_host_begin": (
        C.c_int,
        [_P, _P, _P, C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_int, _P, C.c_int, C.c_int64],
    ),
    "uml_async_poll": (C.c_int, [_P, C.POINTER(C.c_int64), C.POINTER(C.c_int)]),
    "uml_async_finish": (C.c_int, [_P, C.POINTER(Stats)]),
    "uml_linear_predict_proba": (C.c_int, [_P, _P, _P, _P, C.c_int]),
    "uml_mlp_load": (C.c_int, [_P, _PP, _P, _P, _P, _P, C.c_int, C.c_int, C.c_int]),
    "uml_mlp_free": (None, [_P]),
    "uml_mlp_predict": (C.c_int, [_P, _P, _P, _P, C.c_int, C.c_int, C.POINTER(Stats)]),
    "uml_mlp_predict_host": (
        C.c_int,
        [_P, _P, _P, C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_int, _P, C.c_int, C.c_int64, C.POINTER(Stats)],
    ),
    "uml_mlp_predict_host_begin": (
        C.c_int,
        [_P, _P, _P, C.c_int64, C.c_int, C.c_int64, C.c_int64, C.c_int, _P, C.c_int, C.c_int64],
    ),
    "uml_mlp_predict_peers": (C.c_int, [_P, _P, _P, _PP, C.c_int, C.c_int64, C.c_int, C.c_int, C.POINTER(Stats)]),
    "uml_mlp_predict_proba": (C.c_int, [_P, _P, _P, _P, C.c_int, C.POINTER(Stats)]),
}

_lib = None
_pylist = None
PYLIST_PATH = Path(__file__).resolve().parent / "_lib" / "libuml_pylist.so"


def pylist():
    """The CPython list helper (``csrc_host/uml_pylist.c``), loaded with ``PyDLL`` so the GIL stays held; ``None`` when
    it has not been built (callers then fall back to ``ndarray.tolist()``)."""
    global _pylist
    if _pylist is None:
        if not PYLIST_PATH.exists():
            return None
        h = C.PyDLL(str(PYLIST_PATH))
        h.uml_list_fill_from_labels.restype = C.c_int
        h.uml_list_fill_from_labels.argtypes = [C.py_object, C.c_ssize_t, C.c_void_p, C.c_ssize_t, C.py_object]
        _pylist = h
    return _pylist


class NativeLibraryMissing(ImportError):
    pass


def lib() -> C.CDLL:
    """Load (once) and return the CUDA library; raise if it has not been built."""
    global _lib
    if _lib is None:
        path = Path(os.environ.get("UNIONML_B200_LIB", LIB_PATH))
        if not path.exists():
            raise NativeLibraryMissing(
                f"{path} not found: build it with `python -m unionml_b200._build` (needs nvcc). "
                "unionml_b200 has no CPU fallback for the predict hot path."
            )
        handle = C.CDLL(str(path))
        for name, (restype, argtypes) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = restype
            fn.argtypes = argtypes
        _lib = handle
    return _lib
