"""Python handle classes over the C ABI: :class:`Engine`, :class:`LinearModel`, :class:`Batch`.

This is the device path that ``unionml_b200.model.Model.predict``, ``unionml_b200.fastapi.serving_app`` and
``unionml_b200.services`` all call (the reference reaches its CPU arithmetic through
``self._predictor(model_object, features)``, ``/root/reference/unionml/model.py:606,642``).
"""
from __future__ import annotations

import ctypes as C
import os
import threading
import weakref
from typing import Any, Optional, Tuple

import numpy as np

from unionml_b200 import _native as N

_DTYPES = {
    np.dtype(np.float32): N.UML_F32,
    np.dtype(np.float64): N.UML_F64,
    np.dtype(np.int64): N.UML_I64,
    np.dtype(np.int32): N.UML_I32,
    np.dtype(np.uint8): N.UML_U8,
}


class EngineError(RuntimeError):
    """A failure inside the CUDA library (status code + ``uml_last_error`` text)."""

    def __init__(self, status: int, message: str):
        super().__init__(f"uml_b200 status {status}: {message}")
        self.status = status


def _raise(status: int, message: str):
    # the error contract of the drop-in boundary: what sklearn raises as ValueError stays a ValueError
    if status in (N.UML_ERR_NONFINITE, N.UML_ERR_SHAPE):
        raise ValueError(message)
    if status == N.UML_ERR_NOMEM:
        raise MemoryError(message)
    raise EngineError(status, message)


def as_feature_array(features: Any) -> np.ndarray:
    """Borrow ``features`` as a 2-D ndarray in a dtype the staging kernels take, without copying when possible.

    pandas frames are feature-major blocks (SURVEY.md hard part 6); that order is kept - the transpose happens on
    the GPU.  Mirrors the dtype rule of ``check_array(dtype="numeric")``: floats and ints pass, the rest -> float64.
    """
    if hasattr(features, "to_numpy"):
        arr = features.to_numpy()
    elif hasattr(features, "detach") and hasattr(features, "numpy"):  # torch CPU tensor
        arr = features.detach().cpu().numpy()
    else:
        arr = np.asarray(features)
    if arr.ndim == 1:
        raise ValueError(
            f"Expected 2D array, got 1D array instead:\narray={arr}.\nReshape your data either using "
            "array.reshape(-1, 1) if your data has a single feature or array.reshape(1, -1) if it contains a single sample."
        )
    if arr.ndim != 2:
        raise ValueError(f"Found array with dim {arr.ndim}. Expected 2.")
    if arr.dtype not in _DTYPES:
        arr = arr.astype(np.float64)
    if not arr.dtype.isnative:
        arr = arr.astype(arr.dtype.newbyteorder("="))
    rs, cs = arr.strides
    item = arr.itemsize
    ok = (cs == item and rs >= item * arr.shape[1] and rs % item == 0) or (
        rs == item and cs >= item * arr.shape[0] and cs % item == 0
    )
    if arr.shape[0] <= 1 or arr.shape[1] <= 1:
        ok = ok or arr.flags.c_contiguous or arr.flags.f_contiguous
    if not ok:
        arr = np.ascontiguousarray(arr)
    return arr


class LinearModel:
    """``coef_``/``intercept_`` of a linear classifier resident on the device (fp32 tile operands + fp64 copy)."""

    def __init__(self, engine: "Engine", handle: int, n_features: int, n_classes: int, classes: Optional[np.ndarray]):
        self.engine = engine
        self._h = handle
        self.n_features = n_features
        self.n_classes = n_classes
        self.classes = classes
        # numeric class labels as float64, ready for the device-side classes_.take (None for string labels)
        self.classes_f64 = None
        if classes is not None and np.asarray(classes).dtype.kind in "iufb":
            self.classes_f64 = np.ascontiguousarray(classes, dtype=np.float64)
        #: one Python float per class - the objects the `List[float]` of the predictor contract references
        self.class_table = None if self.classes_f64 is None else [float(c) for c in self.classes_f64]
        self._fin = weakref.finalize(self, N.lib().uml_model_free, handle)

    def set_affine(self, shift=None, scale=None) -> None:
        """Fold ``x' = (x - shift) * scale`` (e.g. a fitted ``StandardScaler``) into W and b."""
        sh = None if shift is None else np.ascontiguousarray(shift, dtype=np.float64)
        sc = None if scale is None else np.ascontiguousarray(scale, dtype=np.float64)
        for v in (sh, sc):
            if v is not None and v.shape != (self.n_features,):
                raise ValueError(f"affine vector must have shape ({self.n_features},)")
        with self.engine._lock:
            st = N.lib().uml_linear_set_affine(
                self.engine._h,
                self._h,
                None if sh is None else sh.ctypes.data_as(C.c_void_p),
                None if sc is None else sc.ctypes.data_as(C.c_void_p),
            )
            self.engine._check(st)


class MlpModel:
    """A 2-layer ``Linear -> ReLU -> Linear`` classifier resident on the device."""

    def __init__(self, engine: "Engine", handle: int, n_in: int, n_hidden: int, n_out: int):
        self.engine = engine
        self._h = handle
        self.n_features, self.n_hidden, self.n_classes = n_in, n_hidden, n_out
        self.class_table = [float(c) for c in range(n_out)]  # `float(x) for x in ....argmax(1)`: the class index as float
        self._fin = weakref.finalize(self, N.lib().uml_mlp_free, handle)


class Batch:
    """Feature rows resident in HBM as fp32 row-major (the staged form of ``Dataset.get_features`` output)."""

    def __init__(self, engine: "Engine", handle: int, keepalive: Any = None):
        self.engine = engine
        self._h = handle
        self._keepalive = keepalive
        n, f, ld, ptr, ll = C.c_int64(), C.c_int(), C.c_int64(), C.c_void_p(), C.c_int()
        engine._check(N.lib().uml_batch_info(handle, C.byref(n), C.byref(f), C.byref(ld), C.byref(ptr), C.byref(ll)))
        self.n_rows, self.n_features, self.ld = n.value, f.value, ld.value
        self.device_ptr = ptr.value or 0
        self.lossless = bool(ll.value)
        self._fin = weakref.finalize(self, N.lib().uml_batch_free, handle)

    def free(self) -> None:
        self._fin()


class DeviceBuffer:
    """``nbytes`` of device memory from ``uml_device_alloc``."""

    def __init__(self, engine: "Engine", ptr: int, nbytes: int):
        self.engine, self.ptr, self.nbytes = engine, ptr, nbytes
        self._fin = weakref.finalize(self, N.lib().uml_device_free, engine._h, ptr)


class Engine:
    """One CUDA device bound to this process (one process per GPU)."""

    def __init__(self, device: Optional[int] = None):
        lib = N.lib()
        if device is None:
            device = int(os.environ.get("UNIONML_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        h = C.c_void_p()
        st = lib.uml_engine_create(C.byref(h), int(device))
        if st != N.UML_OK:
            msg = (lib.uml_last_error(None) or b"").decode()
            if st == N.UML_ERR_NO_DEVICE:
                raise RuntimeError(f"unionml_b200 needs a B200 (sm_100a) and has no CPU fallback: {msg}")
            _raise(st, msg)
        self._h = h.value
        self.device = int(device)
        self._lock = threading.Lock()
        self._stream: Optional[int] = None  # caller's stream handle the engine launches on (None: its own stream)
        self._fin = weakref.finalize(self, lib.uml_engine_destroy, self._h)
        info = N.DeviceInfo()
        self._check(lib.uml_engine_info(self._h, C.byref(info)))
        self.info = {
            "device_id": info.device_id,
            "name": info.name.decode(),
            "sm_count": info.sm_count,
            "cc": f"{info.cc_major}.{info.cc_minor}",
            "total_mem_bytes": info.total_mem_bytes,
            "l2_bytes": info.l2_bytes,
            "sm_clock_khz": info.sm_clock_khz,
            "mem_clock_khz": info.mem_clock_khz,
        }

    # ------------------------------------------------------------------------------------------------------------
    def _check(self, status: int) -> None:
        if status != N.UML_OK:
            _raise(status, (N.lib().uml_last_error(self._h) or b"").decode())

    def set_stream(self, cuda_stream: Optional[int]) -> None:
        """Run on the caller's stream (e.g. ``torch.cuda.current_stream().cuda_stream``); ``None`` = engine stream."""
        self._check(N.lib().uml_engine_set_stream(self._h, C.c_void_p(cuda_stream or 0)))
        self._stream = cuda_stream or None

    @property
    def stream(self) -> Optional[int]:
        """The caller's stream handle set by :meth:`set_stream`, or ``None`` when the engine runs on its own stream."""
        return self._stream

    def synchronize(self) -> None:
        self._check(N.lib().uml_engine_synchronize(self._h))

    def pinned_empty(self, shape, dtype=np.float32) -> np.ndarray:
        """A numpy array in page-locked host memory (feature frames and label vectors of the e2e path)."""
        dtype = np.dtype(dtype)
        shape = (shape,) if isinstance(shape, int) else tuple(shape)
        nbytes = int(np.prod(shape, dtype=np.int64)) * dtype.itemsize
        p = C.c_void_p()
        self._check(N.lib().uml_host_alloc(self._h, C.byref(p), nbytes))
        buf = (C.c_char * max(nbytes, 1)).from_address(p.value)
        arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape, dtype=np.int64))).reshape(shape)
        weakref.finalize(buf, N.lib().uml_host_free, self._h, p.value)
        return arr

    def device_alloc(self, nbytes: int) -> "DeviceBuffer":
        """Plain device memory owned by a small handle object (freed when it is garbage collected)."""
        p = C.c_void_p()
        self._check(N.lib().uml_device_alloc(self._h, C.byref(p), int(nbytes)))
        return DeviceBuffer(self, p.value, int(nbytes))

    # ------------------------------------------------------------------------------------------------------------
    def load_linear(self, coef, intercept, classes=None) -> LinearModel:
        coef = np.asarray(coef)
        if coef.ndim == 1:
            coef = coef[None, :]
        intercept = np.atleast_1d(np.asarray(intercept))
        dt = np.float32 if (coef.dtype == np.float32 and intercept.dtype == np.float32) else np.float64
        coef = np.ascontiguousarray(coef, dtype=dt)
        intercept = np.ascontiguousarray(intercept, dtype=dt)
        n_classes, n_features = coef.shape
        if intercept.shape != (n_classes,):
            raise ValueError(f"intercept shape {intercept.shape} does not match coef {coef.shape}")
        h = C.c_void_p()
        with self._lock:
            st = N.lib().uml_linear_load(
                self._h,
                C.byref(h),
                coef.ctypes.data_as(C.c_void_p),
                intercept.ctypes.data_as(C.c_void_p),
                n_classes,
                n_features,
                N.UML_F32 if dt == np.float32 else N.UML_F64,
            )
            self._check(st)
        return LinearModel(self, h.value, n_features, max(n_classes, 2), None if classes is None else np.asarray(classes))

    def load_mlp(self, w1, b1, w2, b2) -> MlpModel:
        """``torch.nn.Linear`` layout: ``w1`` (hidden, in), ``b1`` (hidden), ``w2`` (out, hidden), ``b2`` (out); fp32."""
        w1, b1, w2, b2 = (np.ascontiguousarray(a, dtype=np.float32) for a in (w1, b1, w2, b2))
        n_hidden, n_in = w1.shape
        n_out = w2.shape[0]
        if b1.shape != (n_hidden,) or w2.shape != (n_out, n_hidden) or b2.shape != (n_out,):
            raise ValueError(f"inconsistent MLP shapes {w1.shape} {b1.shape} {w2.shape} {b2.shape}")
        h = C.c_void_p()
        with self._lock:
            st = N.lib().uml_mlp_load(
                self._h, C.byref(h), *(a.ctypes.data_as(C.c_void_p) for a in (w1, b1, w2, b2)), n_in, n_hidden, n_out
            )
            self._check(st)
        return MlpModel(self, h.value, n_in, n_hidden, n_out)

    def predict_mlp(self, model: MlpModel, batch: Batch, exact: bool = True, out_device_ptr: Optional[int] = None,
                    want_stats: bool = True) -> Tuple[Optional[np.ndarray], Optional[dict]]:
        """Argmax class index per row of ``softmax(W2 relu(W1 x + b1) + b2)``."""
        mode = N.UML_PREDICT_EXACT if exact else N.UML_PREDICT_FAST
        stats = N.Stats() if want_stats else None
        with self._lock:
            if out_device_ptr is not None:
                st = N.lib().uml_mlp_predict(
                    self._h, model._h, batch._h, C.c_void_p(out_device_ptr), 1, mode, C.byref(stats) if stats else None
                )
                self._check(st)
                return None, stats.as_dict() if stats else None
            out = np.empty(batch.n_rows, dtype=np.int32)
            st = N.lib().uml_mlp_predict(
                self._h, model._h, batch._h, out.ctypes.data_as(C.c_void_p), 0, mode, C.byref(stats) if stats else None
            )
            self._check(st)  # under the lock: uml_last_error is per engine, another thread's call may overwrite it
        return out, stats.as_dict() if stats else None

    def predict_mlp_proba(self, model: MlpModel, batch: Batch, out_device_ptr: Optional[int] = None
                          ) -> Tuple[Optional[np.ndarray], dict]:
        """``softmax(W2 relu(W1 x + b1) + b2)`` per row, fp32 ``(n_rows, n_out)``: what ``PytorchModel.forward``
        returns.  Host result unless ``out_device_ptr`` (16-byte aligned device memory) is given."""
        stats = N.Stats()
        with self._lock:
            if out_device_ptr is not None:
                self._check(N.lib().uml_mlp_predict_proba(self._h, model._h, batch._h, C.c_void_p(out_device_ptr), 1,
                                                          C.byref(stats)))
                return None, stats.as_dict()
            out = np.empty((batch.n_rows, model.n_classes), dtype=np.float32)
            self._check(N.lib().uml_mlp_predict_proba(self._h, model._h, batch._h, out.ctypes.data_as(C.c_void_p), 0,
                                                      C.byref(stats)))
        return out, stats.as_dict()

    def predict_mlp_peers(self, model: MlpModel, batch: Batch, peer_ptrs, row_offset: int, exact: bool = True,
                          want_stats: bool = False, label_bytes: int = 4) -> Optional[dict]:
        """Fused compute + all-gather for the MLP predictor (same contract as :meth:`predict_peers`)."""
        mode = N.UML_PREDICT_EXACT if exact else N.UML_PREDICT_FAST
        arr = (C.c_void_p * len(peer_ptrs))(*[C.c_void_p(p) for p in peer_ptrs])
        stats = N.Stats() if want_stats else None
        with self._lock:
            st = N.lib().uml_mlp_predict_peers(
                self._h, model._h, batch._h, arr, len(peer_ptrs), row_offset, label_bytes, mode, C.byref(stats) if stats else None
            )
            self._check(st)
        return stats.as_dict() if stats else None

    def stage(self, features: Any, keep_f64: bool = True, check_finite: bool = True) -> Batch:
        """Host rows (ndarray / DataFrame, any order, f32/f64/int) -> device fp32 row-major, converted on the GPU."""
        arr = as_feature_array(features)
        flags = (N.UML_STAGE_KEEP_F64 if keep_f64 else 0) | (0 if check_finite else N.UML_STAGE_SKIP_FINITE_CHECK)
        h = C.c_void_p()
        with self._lock:
            st = N.lib().uml_stage_rows(
                self._h,
                C.byref(h),
                C.c_void_p(arr.ctypes.data),
                arr.shape[0],
                arr.shape[1],
                arr.strides[0],
                arr.strides[1],
                _DTYPES[arr.dtype],
                flags,
            )
            self._check(st)
        return Batch(self, h.value)

    def wrap_device(self, device_ptr: int, n_rows: int, n_features: int, ld: Optional[int] = None, keepalive: Any = None) -> Batch:
        """Wrap fp32 row-major rows that already live in HBM (e.g. a torch CUDA tensor's ``data_ptr()``)."""
        h = C.c_void_p()
        with self._lock:
            st = N.lib().uml_batch_from_device(
                self._h, C.byref(h), C.c_void_p(device_ptr), n_rows, n_features, ld if ld is not None else n_features
            )
            self._check(st)
        return Batch(self, h.value, keepalive)

    # ------------------------------------------------------------------------------------------------------------
    def predict(
        self,
        model: LinearModel,
        batch: Batch,
        exact: bool = True,
        out_device_ptr: Optional[int] = None,
        want_stats: bool = True,
    ) -> Tuple[Optional[np.ndarray], Optional[dict]]:
        """Class *indices* per row.  Host result (int32 ndarray) unless ``out_device_ptr`` is given."""
        mode = N.UML_PREDICT_EXACT if exact else N.UML_PREDICT_FAST
        stats = N.Stats() if want_stats else None
        with self._lock:
            if out_device_ptr is not None:
                st = N.lib().uml_linear_predict(
                    self._h, model._h, batch._h, C.c_void_p(out_device_ptr), 1, mode, C.byref(stats) if stats else None
                )
                self._check(st)
                return None, stats.as_dict() if stats else None
            out = np.empty(batch.n_rows, dtype=np.int32)
            st = N.lib().uml_linear_predict(
                self._h, model._h, batch._h, out.ctypes.data_as(C.c_void_p), 0, mode, C.byref(stats) if stats else None
            )
            self._check(st)
        return out, stats.as_dict() if stats else None

    def predict_peers(self, model: LinearModel, batch: Batch, peer_ptrs, row_offset: int, exact: bool = True,
                      want_stats: bool = False, label_bytes: int = 4) -> Optional[dict]:
        """Fused compute + all-gather: labels are stored into every peer's vector from the kernel epilogue."""
        mode = N.UML_PREDICT_EXACT if exact else N.UML_PREDICT_FAST
        arr = (C.c_void_p * len(peer_ptrs))(*[C.c_void_p(p) for p in peer_ptrs])
        stats = N.Stats() if want_stats else None
        with self._lock:
            st = N.lib().uml_linear_predict_peers(
                self._h, model._h, batch._h, arr, len(peer_ptrs), row_offset, label_bytes, mode, C.byref(stats) if stats else None
            )
            self._check(st)
        return stats.as_dict() if stats else None

    def take_labels(self, labels_ptr: int, n: int, classes, label_bytes: int = 4) -> np.ndarray:
        """``classes_[idx].astype(float)`` computed on the device from a device label vector; float64 host array."""
        classes = np.ascontiguousarray(classes, dtype=np.float64)
        out = np.empty(n, dtype=np.float64)
        with self._lock:
            st = N.lib().uml_labels_take(self._h, C.c_void_p(labels_ptr), label_bytes, n,
                                         classes.ctypes.data_as(C.c_void_p), len(classes), out.ctypes.data_as(C.c_void_p))
            self._check(st)
        return out

    def count_equal(self, labels_ptr: int, n: int, classes, targets, label_bytes: int = 4) -> int:
        """Number of rows whose predicted class value equals ``targets`` (accuracy numerator), reduced on the device."""
        classes = np.ascontiguousarray(classes, dtype=np.float64)
        targets = np.ascontiguousarray(targets, dtype=np.float64)
        if targets.shape != (n,):
            raise ValueError("targets must be a vector of length n")
        cnt = C.c_int64()
        with self._lock:
            st = N.lib().uml_labels_count_equal(self._h, C.c_void_p(labels_ptr), label_bytes, n,
                                                classes.ctypes.data_as(C.c_void_p), len(classes),
                                                targets.ctypes.data_as(C.c_void_p), C.byref(cnt))
            self._check(st)
        return int(cnt.value)

    def push_labels(self, src_ptr: int, dst_ptrs, nbytes: int) -> None:
        """Copy ``nbytes`` from ``src_ptr`` (this rank's label slice) to every pointer in ``dst_ptrs`` (peer-mapped
        vectors or an NVLS multicast alias) with a thin copy kernel on the engine stream."""
        arr = (C.c_void_p * len(dst_ptrs))(*[C.c_void_p(p) for p in dst_ptrs])
        with self._lock:
            st = N.lib().uml_labels_push(self._h, C.c_void_p(src_ptr), arr, len(dst_ptrs), nbytes)
            self._check(st)

    def predict_host(
        self,
        model: LinearModel,
        features: Any,
        exact: bool = True,
        out: Optional[np.ndarray] = None,
        chunk_rows: int = 0,
    ) -> Tuple[np.ndarray, dict]:
        """Host rows -> host labels in one pipelined call (chunked H2D / convert / score / D2H)."""
        arr = as_feature_array(features)
        if out is None:
            out = np.empty(arr.shape[0], dtype=np.int32)
        elif out.dtype != np.int32 or out.shape != (arr.shape[0],) or not out.flags.c_contiguous:
            raise ValueError("out must be a C-contiguous int32 vector of length n_rows")
        stats = N.Stats()
        with self._lock:
            st = N.lib().uml_linear_predict_host(
                self._h,
                model._h,
                C.c_void_p(arr.ctypes.data),
                arr.shape[0],
                arr.shape[1],
                arr.strides[0],
                arr.strides[1],
                _DTYPES[arr.dtype],
                out.ctypes.data_as(C.c_void_p),
                N.UML_PREDICT_EXACT if exact else N.UML_PREDICT_FAST,
                chunk_rows,
                C.byref(stats),
            )
            self._check(st)
        return out, stats.as_dict()

    def predict_host_values(self, model: LinearModel, features: Any, classes, exact: bool = True,
                            chunk_rows: int = 0) -> Tuple[np.ndarray, dict]:
        """Host rows -> ``classes_[argmax]`` as a float64 host vector: the pipelined call with ``classes_.take`` and the
        float conversion of the canonical predictor (``README.md:92``) done on the device, chunk by chunk."""
        arr = as_feature_array(features)
        if not (isinstance(classes, np.ndarray) and classes.dtype == np.float64 and classes.flags.c_contiguous):
            classes = np.ascontiguousarray(classes, dtype=np.float64)
        out = np.empty(arr.shape[0], dtype=np.float64)
        stats = N.Stats()
        with self._lock:
            st = N.lib().uml_linear_predict_host_values(
                self._h,
                model._h,
                C.c_void_p(arr.ctypes.data),
                arr.shape[0],
                arr.shape[1],
                arr.strides[0],
                arr.strides[1],
                _DTYPES[arr.dtype],
                classes.ctypes.data_as(C.c_void_p),
                len(classes),
                out.ctypes.data_as(C.c_void_p),
                N.UML_PREDICT_EXACT if exact else N.UML_PREDICT_FAST,
                chunk_rows,
                C.byref(stats),
            )
            self._check(st)
        return out, stats.as_dict()

    def predict_mlp_host(self, model: MlpModel, features: Any, exact: bool = True, chunk_rows: int = 0,
                         out: Optional[np.ndarray] = None) -> Tuple[np.ndarray, dict]:
        """Host rows -> argmax class index of the 2-layer MLP per row (int32), through the chunk pipeline (pinned bounce
        buffers, GPU down-cast to fp32 as the reference predictor does, scoring kernel, fp64 re-score)."""
        arr = as_feature_array(features)
        if out is None:
            out = np.empty(arr.shape[0], dtype=np.int32)
        stats = N.Stats()
        with self._lock:
            st = N.lib().uml_mlp_predict_host(
                self._h, model._h, C.c_void_p(arr.ctypes.data), arr.shape[0], arr.shape[1], arr.strides[0], arr.strides[1],
                _DTYPES[arr.dtype], out.ctypes.data_as(C.c_void_p), N.UML_PREDICT_EXACT if exact else N.UML_PREDICT_FAST,
                chunk_rows, C.byref(stats),
            )
            self._check(st)
        return out, stats.as_dict()

    def predict_host_list(self, model, features: Any, table: list, exact: bool = True, chunk_rows: int = 0,
                          asynchronous: Optional[bool] = None) -> Tuple[list, dict]:
        """The predictor contract in one call: host rows -> ``[table[label] for label in labels]`` as a Python list.

        ``table`` holds one Python float per class (``[float(c) for c in classes_]``); the list references those
        objects (``csrc_host/uml_pylist.c``: ~2 ns per row instead of ~25 ns for a fresh float per row).  With
        ``asynchronous`` (default from 1M rows) the pipeline runs on a library thread (``uml_*_predict_host_begin``) and
        the finished prefix is filled into the list while the rest of the batch is still in flight."""
        import time

        arr = as_feature_array(features)
        is_mlp = isinstance(model, MlpModel)
        n = arr.shape[0]
        labels = np.empty(n, dtype=np.int32)
        helper = N.pylist()
        lib = N.lib()
        mode = N.UML_PREDICT_EXACT if exact else N.UML_PREDICT_FAST
        if asynchronous is None:
            asynchronous = n >= 1_000_000
        stats = N.Stats()

        def fill(out, start, count):
            if helper is not None:
                helper.uml_list_fill_from_labels(out, start, C.c_void_p(labels.ctypes.data + 4 * start), count, table)
            else:  # helper not built: numpy object take (slower, same result)
                out[start : start + count] = [table[k] for k in labels[start : start + count].tolist()]

        if not asynchronous:
            if is_mlp:
                _, d = self.predict_mlp_host(model, arr, exact=exact, chunk_rows=chunk_rows, out=labels)
            else:
                _, d = self.predict_host(model, arr, exact=exact, out=labels, chunk_rows=chunk_rows)
            out: list = [None] * n
            fill(out, 0, n)
            return out, d
        begin = lib.uml_mlp_predict_host_begin if is_mlp else lib.uml_linear_predict_host_begin
        with self._lock:
            t0 = time.perf_counter()
            st = begin(self._h, model._h, C.c_void_p(arr.ctypes.data), n, arr.shape[1], arr.strides[0], arr.strides[1],
                       _DTYPES[arr.dtype], labels.ctypes.data_as(C.c_void_p), mode, chunk_rows)
            self._check(st)
            done, rows_done, finished = 0, C.c_int64(), C.c_int()
            t_pipeline = t_list = 0.0
            try:
                # the result list is allocated while the first chunks are already in flight (10M slots: ~25 ms of page
                # faults that used to sit in front of the pipeline)
                out = [None] * n
                while True:
                    lib.uml_async_poll(self._h, C.byref(rows_done), C.byref(finished))
                    if finished.value and not t_pipeline:
                        t_pipeline = time.perf_counter() - t0
                    if rows_done.value - done >= 262_144 or (finished.value and rows_done.value > done):
                        t1 = time.perf_counter()
                        fill(out, done, rows_done.value - done)
                        t_list += time.perf_counter() - t1
                        done = rows_done.value
                    elif finished.value:
                        break
                    else:
                        time.sleep(0.0002)
            finally:
                st = lib.uml_async_finish(self._h, C.byref(stats))
            self._check(st)
        if done < n:  # not reached when the call succeeded (every chunk is flushed before it finishes)
            fill(out, done, n - done)
        d = stats.as_dict()
        # host-side view of the overlap: when the library thread finished, and how long list filling took in total
        d.update(pipeline_s=t_pipeline, list_s=t_list, total_s=time.perf_counter() - t0)
        return out, d

    def predict_proba(self, model: LinearModel, batch: Batch, out_device_ptr: Optional[int] = None) -> Optional[np.ndarray]:
        """``softmax(X @ coef_.T + intercept_)`` per row (fp32), ``(n_rows, n_classes)``; ``[1 - p, p]`` for a binary model."""
        with self._lock:
            if out_device_ptr is not None:
                self._check(N.lib().uml_linear_predict_proba(self._h, model._h, batch._h, C.c_void_p(out_device_ptr), 1))
                return None
            out = np.empty((batch.n_rows, model.n_classes), dtype=np.float32)
            self._check(N.lib().uml_linear_predict_proba(self._h, model._h, batch._h, out.ctypes.data_as(C.c_void_p), 0))
        return out


_default_engine: Optional[Engine] = None
_default_lock = threading.Lock()


def get_engine() -> Engine:
    """Process-wide engine, created on first use (never at import: uvicorn workers fork, cli.py:289)."""
    global _default_engine
    with _default_lock:
        if _default_engine is None or getattr(_default_engine, "_pid", None) != os.getpid():
            _default_engine = Engine()
            _default_engine._pid = os.getpid()
        return _default_engine
