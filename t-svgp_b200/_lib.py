"""
ctypes binding of libtsvgp.so (include/tsvgp.h).  No torch, no CPU fallback: if the shared library is missing or there is
no CUDA device, the first call raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtsvgp.so")

OK, ERR_INVALID, ERR_CUDA, ERR_NOT_PD, ERR_NONPOS_VAR, ERR_COMM, ERR_STATE = 0, -1, -2, -3, -4, -5, -6
KERNEL_SE, KERNEL_MATERN52, KERNEL_MATERN12, KERNEL_MATERN32 = 0, 1, 2, 3
LIK_GAUSSIAN, LIK_BERNOULLI_PROBIT, LIK_STUDENT_T, LIK_SOFTMAX, LIK_HETEROSKEDASTIC = 0, 1, 2, 3, 4
ABI_VERSION = 1


class TsvgpError(RuntimeError):
    """Base class of errors raised by the CUDA library."""

    def __init__(self, code, message):
        super().__init__(f"libtsvgp error {code}: {message}")
        self.code = code


class InvalidArgumentError(TsvgpError, ValueError):
    """Stands in for tf.errors.InvalidArgumentError (shape checks, failed Cholesky, non-positive variance)."""


class NotPositiveDefiniteError(InvalidArgumentError):
    def __init__(self, code, message, pivot=0):
        super().__init__(code, message)
        self.pivot = pivot


class NonPositiveVarianceError(InvalidArgumentError):
    pass


class View(C.Structure):
    _fields_ = [("data", C.c_void_p), ("shape", C.c_int64 * 3), ("ndim", C.c_int), ("device_type", C.c_int), ("device_id", C.c_int)]


_dp = C.POINTER(C.c_double)
_SIGNATURES = {
    "tsvgp_abi_version": (C.c_int, []),
    "tsvgp_create": (C.c_int, [C.POINTER(C.c_void_p), C.c_int]),
    "tsvgp_destroy": (None, [C.c_void_p]),
    "tsvgp_last_error": (C.c_char_p, [C.c_void_p]),
    "tsvgp_last_info": (C.c_int, [C.c_void_p]),
    "tsvgp_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_double]),
    "tsvgp_set_kernel": (C.c_int, [C.c_void_p, C.c_int, C.c_double, _dp, C.c_int]),
    "tsvgp_set_kernels": (C.c_int, [C.c_void_p, C.c_void_p, _dp, _dp, C.c_void_p]),
    "tsvgp_set_likelihood": (C.c_int, [C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_int, _dp, _dp]),
    "tsvgp_set_inducing": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "tsvgp_set_num_latent": (C.c_int, [C.c_void_p, C.c_int]),
    "tsvgp_num_latent": (C.c_int, [C.c_void_p]),
    "tsvgp_set_mc_epsilon": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int64, C.c_int]),
    "tsvgp_set_sites": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tsvgp_get_sites": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tsvgp_get_lambda_2": (C.c_int, [C.c_void_p, C.c_void_p]),
    "tsvgp_set_data": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "tsvgp_stage_data": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p]),
    "tsvgp_commit_staged": (C.c_int, [C.c_void_p]),
    "tsvgp_natgrad_step": (C.c_int, [C.c_void_p, C.c_double, C.c_double, C.c_double, _dp]),
    "tsvgp_elbo": (C.c_int, [C.c_void_p, C.c_double, _dp]),
    "tsvgp_prior_kl": (C.c_int, [C.c_void_p, _dp]),
    "tsvgp_elbo_grad": (C.c_int, [C.c_void_p, C.c_double, _dp, _dp, C.c_void_p, C.c_void_p, _dp]),
    "tsvgp_predict_f": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tsvgp_predict_f_full_cov": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "tsvgp_predict_f_samples": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p,
                                          C.c_void_p]),
    "tsvgp_predict_f_extra_data": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p]),
    "tsvgp_posterior": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "tsvgp_comm_unique_id": (C.c_int, [C.c_void_p]),
    "tsvgp_comm_init": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "tsvgp_comm_size": (C.c_int, [C.c_void_p]),
    "tsvgp_device": (C.c_int, [C.c_void_p]),
    "tsvgp_stream": (C.c_void_p, [C.c_void_p]),
    "tsvgp_get_timings": (C.c_int, [C.c_void_p, _dp, C.c_int]),
    "tsvgp_sync": (C.c_int, [C.c_void_p]),
    "tsvgp_get_kernel_profile": (C.c_int, [C.c_void_p, _dp, C.c_int]),
    "tsvgp_timer_start": (C.c_int, [C.c_void_p]),
    "tsvgp_timer_stop": (C.c_int, [C.c_void_p, _dp]),
    "tsvgp_device_alloc": (C.c_void_p, [C.c_void_p, C.c_size_t]),
    "tsvgp_device_free": (None, [C.c_void_p, C.c_void_p]),
    "tsvgp_memcpy": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t]),
    "tsvgp_pinned_alloc": (C.c_void_p, [C.c_size_t]),
    "tsvgp_pinned_free": (None, [C.c_void_p]),
    "tsvgp_dlpack_view": (C.c_int, [C.c_void_p, C.POINTER(View)]),
}

_lib = None


def load():
    """Load libtsvgp.so (built in-tree by `__graft_entry__.build()` / `make -C t-svgp_b200/csrc`)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `make -C t-svgp_b200/csrc` (there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
    for name, (res, args) in _SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the ABI is incomplete
        fn.restype = res
        fn.argtypes = args
    if lib.tsvgp_abi_version() != ABI_VERSION:
        raise ImportError(f"libtsvgp ABI {lib.tsvgp_abi_version()} != binding {ABI_VERSION}")
    _lib = lib
    return lib


def exported_names():
    return list(_SIGNATURES)


def raise_for(lib, ctx, code):
    if code == OK:
        return
    msg = lib.tsvgp_last_error(ctx)
    msg = msg.decode() if msg else ""
    if code == ERR_NOT_PD:
        raise NotPositiveDefiniteError(code, msg, lib.tsvgp_last_info(ctx))
    if code == ERR_NONPOS_VAR:
        raise NonPositiveVarianceError(code, msg)
    if code == ERR_INVALID:
        raise InvalidArgumentError(code, msg)
    raise TsvgpError(code, msg)


# ---- DLPack hand-over --------------------------------------------------------------------------------------------------
_PyCapsule_GetPointer = C.pythonapi.PyCapsule_GetPointer
_PyCapsule_GetPointer.restype = C.c_void_p
_PyCapsule_GetPointer.argtypes = [C.py_object, C.c_char_p]

KDL_CPU, KDL_CUDA, KDL_CUDA_HOST, KDL_CUDA_MANAGED = 1, 2, 3, 13


class Tensor:
    """A float64, C-contiguous tensor borrowed through DLPack: `.ptr`, `.shape`, `.on_device`. Keeps its owner alive."""

    __slots__ = ("ptr", "shape", "on_device", "device_id", "_keep")

    def __init__(self, ptr, shape, on_device, device_id, keep):
        self.ptr, self.shape, self.on_device, self.device_id, self._keep = ptr, tuple(shape), on_device, device_id, keep


class DeviceArray:
    """A float64 row-major array in GPU memory owned by this object (cudaMalloc through the C-ABI; no tensor library)."""

    def __init__(self, model, host_array):
        a = np.ascontiguousarray(host_array, dtype=np.float64)
        self._model, self.shape, self.nbytes = model, a.shape, a.nbytes
        self.ptr = model._lib.tsvgp_device_alloc(model._ctx, a.nbytes)
        if not self.ptr:
            raise TsvgpError(ERR_CUDA, f"cudaMalloc of {a.nbytes} bytes failed")
        raise_for(model._lib, model._ctx, model._lib.tsvgp_memcpy(model._ctx, self.ptr, a.ctypes.data, a.nbytes))

    def numpy(self):
        out = np.empty(self.shape)
        raise_for(self._model._lib, self._model._ctx, self._model._lib.tsvgp_memcpy(self._model._ctx, out.ctypes.data, self.ptr, self.nbytes))
        return out

    def free(self):
        if self.ptr and getattr(self._model, "_ctx", None):
            self._model._lib.tsvgp_device_free(self._model._ctx, self.ptr)
        self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def pinned_empty(shape):
    """A float64 NumPy array over page-locked host memory (cudaHostAlloc), for full-speed host->device copies."""
    lib = load()
    n = int(np.prod(shape))
    ptr = lib.tsvgp_pinned_alloc(max(n, 1) * 8)
    if not ptr:
        raise TsvgpError(ERR_CUDA, "cudaHostAlloc failed")
    buf = (C.c_double * max(n, 1)).from_address(ptr)
    arr = np.frombuffer(buf, dtype=np.float64, count=n).reshape(shape)
    _PINNED[arr.ctypes.data] = ptr   # freed at interpreter exit by the driver; explicit pinned_free for long runs
    return arr


_PINNED = {}


def pinned_free(arr):
    ptr = _PINNED.pop(arr.ctypes.data, None)
    if ptr:
        load().tsvgp_pinned_free(ptr)


def as_tensor(obj, name="tensor", model=None):
    """numpy arrays / anything with __dlpack__ (cupy, torch, jax ...) -> Tensor.  Host data is made float64-contiguous;
    device data must already be float64 and compact (the C side validates the DLTensor).  With `model`, a device tensor is
    requested on the context's main stream (DLPack's `stream` argument: the producer orders its pending writes before that
    stream's next work) and must live on the context's device."""
    lib = load()
    if isinstance(obj, DeviceArray):
        return Tensor(obj.ptr, obj.shape, True, 0, obj)
    if not hasattr(obj, "__dlpack__") or isinstance(obj, (list, tuple)):
        obj = np.ascontiguousarray(obj, dtype=np.float64)
    if isinstance(obj, np.ndarray):
        if obj.dtype != np.float64 or not obj.flags.c_contiguous:
            obj = np.ascontiguousarray(obj, dtype=np.float64)
        if not obj.flags.writeable:  # numpy refuses to export read-only arrays through DLPack
            return Tensor(obj.ctypes.data, obj.shape, False, 0, obj)
    cap = None
    if model is not None and not isinstance(obj, np.ndarray):
        handle = lib.tsvgp_stream(model._ctx)
        try:
            cap = obj.__dlpack__(stream=int(handle or 0) or None)
        except (TypeError, ValueError, RuntimeError, AssertionError, BufferError):   # producers without stream support / host tensors
            cap = None
    if cap is None:
        cap = obj.__dlpack__()
    dlm = _PyCapsule_GetPointer(cap, b"dltensor")
    view = View()
    rc = lib.tsvgp_dlpack_view(dlm, C.byref(view))
    if rc != OK:
        raise InvalidArgumentError(rc, f"{name}: DLPack tensor must be float64, <= 3-D and compact row-major")
    shape = [view.shape[i] for i in range(view.ndim)]
    on_device = view.device_type in (KDL_CUDA, KDL_CUDA_MANAGED)
    if view.device_type not in (KDL_CPU, KDL_CUDA, KDL_CUDA_HOST, KDL_CUDA_MANAGED):
        raise InvalidArgumentError(ERR_INVALID, f"{name}: unsupported DLPack device type {view.device_type}")
    if on_device and model is not None and view.device_type == KDL_CUDA and view.device_id != lib.tsvgp_device(model._ctx):
        raise InvalidArgumentError(ERR_INVALID, f"{name}: tensor lives on cuda:{view.device_id}, the model on cuda:{lib.tsvgp_device(model._ctx)}")
    # the capsule is only borrowed (never renamed): when it is collected it runs the producer's deleter itself
    return Tensor(view.data, shape, on_device, view.device_id, (obj, cap))
