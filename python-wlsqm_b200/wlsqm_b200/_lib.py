"""ctypes binding of ``libwlsqm_b200.so`` (the C ABI declared in ``include/wlsqm_b200.h``).

The shared library is built in-tree by ``python-wlsqm_b200/csrc/Makefile`` (``__graft_entry__.build()``).
There is no fallback of any kind: if the library is missing, importing the compute modules raises,
and if no CUDA device is present every compute call raises ``RuntimeError``.
"""
from __future__ import annotations

import ctypes as C
import os
import sys
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "libwlsqm_b200.so"

OK, E_VALUE, E_MEMORY, E_CUDA, E_NOTREADY = 0, -1, -2, -3, -4
DIFF_ALL = -1

_lib = None

_i32p = C.POINTER(C.c_int32)
_i64p = C.POINTER(C.c_int64)
_vp = C.c_void_p
_i64 = C.c_int64
_int = C.c_int

# name -> (restype, argtypes); one entry per symbol declared in include/wlsqm_b200.h
SIGNATURES = {
    "wlsqm_b200_abi_version": (_int, []),
    "wlsqm_last_error": (C.c_char_p, []),
    "wlsqm_device_count": (_int, []),
    "wlsqm_number_of_dofs": (_int, [_int, _int]),
    "wlsqm_meta_summary": (_int, [_i64, _vp, _vp, _vp, _vp, _i32p, _i32p, _i32p, _i32p]),
    "wlsqm_pinned_alloc": (_vp, [_i64]),
    "wlsqm_pinned_alloc_wc": (_vp, [_i64]),
    "wlsqm_pinned_free": (None, [_vp]),
    "wlsqm_pool_stats": (_int, [_int, _i64p, _i64p]),
    "wlsqm_pool_trim": (_int, [_int]),
    "wlsqm_solver_create": (_int, [_int, _i64, _vp, _vp, _vp, _vp, _int, _int, _int, _int, _int, C.POINTER(_vp)]),
    "wlsqm_solver_create_guest": (_int, [_vp, _int, _int, _int, C.POINTER(_vp)]),
    "wlsqm_solver_prepare_guest": (_int, [_vp]),
    "wlsqm_solver_destroy": (_int, [_vp]),
    "wlsqm_solver_set_stream": (_int, [_vp, _vp]),
    "wlsqm_solver_synchronize": (_int, [_vp]),
    "wlsqm_set_caller_stream": (_int, [_vp]),
    "wlsqm_solver_prepare": (_int, [_vp, _vp, _i64, _vp, _i64, _i64]),
    "wlsqm_solver_solve": (_int, [_vp, _vp, _i64, _i64, _vp, _i64, _vp, _i64, _i64, _i32p]),
    "wlsqm_solver_iterations": (_int, [_vp, _vp]),
    "wlsqm_solver_interpolate": (_int, [_vp, _vp, _i64, _vp, _i64, _int, _vp, _i64]),
    "wlsqm_solver_conds": (_int, [_vp, _vp]),
    "wlsqm_solver_memory": (_int, [_vp, _i64p, _i64p]),
    "wlsqm_solver_get_fi": (_int, [_vp, _vp, _i64]),
    "wlsqm_fit_many": (_int, [_int, _i64, _vp, _i64, _i64, _vp, _i64, _i64, _vp, _vp, _i64, _vp, _i64, _vp, _i64,
                              _i64, _int, _vp, _vp, _vp, _int, _int, _int, _i32p]),
    "wlsqm_interpolate_fit": (_int, [_int, _int, _vp, _vp, _vp, _i64, _i64, _int, _vp, _int]),
    "wlsqm_grid_create": (_int, [_int, _i64, _vp, _i64, _int, C.POINTER(_vp)]),
    "wlsqm_grid_destroy": (_int, [_vp]),
    "wlsqm_grid_info": (_int, [_vp, _i64p, C.POINTER(C.c_double), _i64p]),
    "wlsqm_grid_knn": (_int, [_vp, _vp, _i64, _i64, _int, _int, _vp, _vp, _vp]),
    "wlsqm_grid_ball_count": (_int, [_vp, _vp, _i64, _i64, _vp, _i64, _int, _int, _vp, _vp, _i64p]),
    "wlsqm_grid_ball_csr": (_int, [_vp, _vp, _i64, _i64, _vp, _i64, _int, _int, _int, _vp, _vp]),
    "wlsqm_gather_hoods": (_int, [_vp, _i64, _int, _i64, _vp, _i64, _i64, _int, _vp, _int, _vp]),
    "wlsqm_solver_prepare_hoods": (_int, [_vp, _vp, _i64, _i64, _vp, _i64, _vp, _i64]),
    "wlsqm_solver_solve_hoods": (_int, [_vp, _vp, _i64, _vp, _i64, _vp, _i64, _i64, _i32p]),
    "wlsqm_solver_solve_fields": (_int, [_vp, _i64, _vp, _i64, _i64, _i64, _vp, _i64, _i64, _i32p]),
    "wlsqm_solver_solve_hoods_fields": (_int, [_vp, _i64, _vp, _i64, _i64, _vp, _i64, _i64, _i32p]),
    "wlsqm_solver_stencils": (_int, [_vp, _int, _vp, _vp, _vp]),
    "wlsqm_solver_operator_nnz": (_int, [_vp, _i64, _vp]),
    "wlsqm_solver_operator_csr": (_int, [_vp, _int, _vp, _i64, _int, _vp, _vp, _vp, _vp]),
    "wlsqm_solver_interp_stencils": (_int, [_vp, _vp, _i64, _vp, _i64, _int, _vp, _vp, _vp]),
    "wlsqm_solver_interp_operator_nnz": (_int, [_vp, _vp, _i64, _i64, _vp]),
    "wlsqm_solver_interp_operator_csr": (_int, [_vp, _vp, _i64, _vp, _i64, _int, _vp, _i64, _int, _vp, _vp, _vp, _vp]),
    "wlsqm_solver_interp_continuous_count": (_int, [_vp, _vp, _i64, _i64, C.c_double, _i64, _vp, _i64p, _i64p]),
    "wlsqm_solver_interp_continuous_stencils": (_int, [_vp, _vp, _i64, _i64, C.c_double, _int, _vp, _vp, _vp, _vp, _vp]),
    "wlsqm_solver_interp_continuous_operator_csr": (_int, [_vp, _vp, _i64, _i64, C.c_double, _int, _vp, _i64, _int, _vp,
                                                           _vp, _vp, _vp, _vp, _vp]),
    "wlsqm_solver_index_models": (_int, [_vp]),
    "wlsqm_solver_nearest_models": (_int, [_vp, _vp, _i64, _i64, _vp]),
    "wlsqm_solver_interpolate_continuous": (_int, [_vp, _vp, _i64, _i64, C.c_double, _int, _vp]),
    "wlsqm_solver_interpolate_fields": (_int, [_vp, _i64, _vp, _i64, _i64, _vp, _i64, _vp, _i64, _int, _vp, _i64, _i64]),
    "wlsqm_solver_interpolate_continuous_fields": (_int, [_vp, _i64, _vp, _i64, _i64, _vp, _i64, _i64, C.c_double, _int,
                                                          _vp, _i64, _i64]),
    "wlsqm_peer_alloc": (_int, [_int, _i64, C.POINTER(_vp), _vp]),
    "wlsqm_peer_open": (_int, [_int, _vp, C.POINTER(_vp)]),
    "wlsqm_peer_close": (_int, [_vp]),
    "wlsqm_peer_free": (_int, [_vp]),
    "wlsqm_solver_keep_solution": (_int, [_vp, _int]),
    "wlsqm_solver_set_gather": (_int, [_vp, _int, C.POINTER(_vp), _i64, _i64]),
    "wlsqm_mgetrf": (_int, [_int, _i64, _vp, _vp, _int]),
    "wlsqm_mgetrs": (_int, [_int, _i64, _vp, _vp, _vp, _int]),
    "wlsqm_mgesv": (_int, [_int, _i64, _vp, _vp, _vp, _int]),
    "wlsqm_msytrf": (_int, [_int, _i64, _vp, _vp, _int]),
    "wlsqm_msytrs": (_int, [_int, _i64, _vp, _vp, _vp, _int]),
    "wlsqm_msysv": (_int, [_int, _i64, _vp, _vp, _vp, _int]),
    "wlsqm_msymmetrize": (_int, [_int, _i64, _vp, _int]),
    "wlsqm_gtsv": (_int, [_int, _vp, _vp, _vp, _vp, _int]),
    "wlsqm_mrescale": (_int, [_int, _int, _i64, _vp, _int, _vp, _vp, _vp, _int]),
}


def lib():
    """Load the native library (once).  Fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `make -C python-wlsqm_b200/csrc` "
                "(or __graft_entry__.build()).  wlsqm_b200 has no CPU fallback.")
        L = C.CDLL(str(LIB_PATH))
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def check(rc: int):
    """Map a C-ABI return code to the reference's exception surface."""
    if rc == OK:
        return
    msg = lib().wlsqm_last_error().decode("utf-8", "replace")
    if rc == E_VALUE:
        raise ValueError(msg)
    if rc == E_MEMORY:
        raise MemoryError(msg)
    raise RuntimeError(msg)


def default_device() -> int:
    """CUDA ordinal used when the caller does not name one: torch's current device if torch has
    initialised CUDA in this process, else $WLSQM_DEVICE, else 0."""
    t = sys.modules.get("torch")
    if t is not None:
        try:
            if t.cuda.is_available() and t.cuda.is_initialized():
                return int(t.cuda.current_device())
        except Exception:
            pass
    return int(os.environ.get("WLSQM_DEVICE", "0"))


def current_stream_ptr(device: int):
    """torch's current CUDA stream on `device` (so that solver work orders with torch ops), or None."""
    t = sys.modules.get("torch")
    if t is None:
        return None
    try:
        if t.cuda.is_available() and t.cuda.is_initialized():
            return int(t.cuda.current_stream(device).cuda_stream)
    except Exception:
        pass
    return None


def announce_stream(device: int):
    """Tell the library which CUDA stream the handle-less entry points (one-shot fits, interpolate_fit, search grid,
    batched dense drivers) must order their work after: torch's current stream on `device`, else the default stream."""
    lib().wlsqm_set_caller_stream(current_stream_ptr(int(device)))


def _is_torch_tensor(a) -> bool:
    t = sys.modules.get("torch")
    return t is not None and isinstance(a, t.Tensor)


class Arr:
    """A float64/int array argument resolved to (pointer, element strides); numpy or torch, host or device."""

    __slots__ = ("ptr", "shape", "strides", "is_cuda", "device", "keep", "np")

    def __init__(self, ptr, shape, strides, is_cuda, device, keep, np_view=None):
        self.ptr, self.shape, self.strides = ptr, tuple(shape), tuple(strides)
        self.is_cuda, self.device, self.keep, self.np = is_cuda, device, keep, np_view


_TORCH_DTYPES = {"float64": "float64", "int64": "int64", "int32": "int32"}


def as_arr(a, dtype, ndim, name, *, writable=False, last_contig=True, allow_copy=False) -> Arr:
    """Resolve a caller array the way the reference's typed memoryviews do: dtype and ndim must match
    exactly (ValueError otherwise); `last_contig` demands a unit stride on the last axis
    (``::view.contiguous``).  Host arrays that violate it are copied only if `allow_copy`
    (the reference's fully strided ``fk``)."""
    dtype = np.dtype(dtype)
    if _is_torch_tensor(a):
        import torch
        want = getattr(torch, _TORCH_DTYPES[dtype.name])
        if a.dtype != want:
            raise ValueError(f"{name}: dtype mismatch, expected {dtype.name} but got {a.dtype}")
        if a.dim() != ndim:
            raise ValueError(f"{name}: expected {ndim} dimensions, got {a.dim()}")
        if a.is_cuda:
            st = tuple(int(s) for s in a.stride())
            if last_contig and ndim and a.shape[-1] > 1 and st[-1] != 1:
                raise ValueError(f"{name}: last axis must be contiguous")
            return Arr(int(a.data_ptr()), a.shape, st, True, a.device.index, a)
        a = a.detach().numpy()
    if not isinstance(a, np.ndarray):
        if writable:
            # the reference's typed memoryviews refuse objects without a writable buffer; a silently copied list would
            # swallow the results
            try:
                mv = memoryview(a)
            except TypeError:
                raise TypeError(f"{name}: a writable float64 buffer is required (got {type(a).__name__})") from None
            if mv.readonly:
                raise ValueError(f"{name}: buffer source array is read-only")
        try:
            a = np.asarray(a)
        except Exception as e:  # pragma: no cover
            raise TypeError(f"{name}: cannot interpret argument as an array") from e
    if a.dtype != dtype:
        raise ValueError(f"{name}: Buffer dtype mismatch, expected '{dtype.name}' but got '{a.dtype.name}'")
    if a.ndim != ndim:
        raise ValueError(f"{name}: Buffer has wrong number of dimensions (expected {ndim}, got {a.ndim})")
    if writable and not a.flags.writeable:
        raise ValueError(f"{name}: buffer source array is read-only")
    item = a.itemsize
    bad_last = ndim and a.shape[-1] > 1 and a.strides[-1] != item
    neg = any(s < 0 for s in a.strides)
    if bad_last or neg or any(s % item for s in a.strides):
        if last_contig and bad_last and not allow_copy:
            raise ValueError(f"{name}: ndarray is not contiguous in its last dimension")
        if writable:
            raise ValueError(f"{name}: unsupported strides for an output array")
        a = np.ascontiguousarray(a)
    st = tuple(s // item for s in a.strides)
    return Arr(a.ctypes.data, a.shape, st, False, None, a, a)


def meta_array(a, dtype, name) -> np.ndarray:
    """nk / order / knowns / weighting_method: 1-D, exact dtype (int[::view.generic] etc.), host."""
    if _is_torch_tensor(a):
        a = a.detach().cpu().numpy()
    a = np.asarray(a)
    dtype = np.dtype(dtype)
    if a.dtype != dtype:
        raise ValueError(f"{name}: Buffer dtype mismatch, expected '{dtype.name}' but got '{a.dtype.name}'")
    if a.ndim != 1:
        raise ValueError(f"{name}: Buffer has wrong number of dimensions (expected 1, got {a.ndim})")
    return np.ascontiguousarray(a)


def pinned_empty(shape, dtype=np.float64, write_combined=False) -> np.ndarray:
    """Page-locked host array (fast, asynchronous H2D/D2H for the staged host-pointer path).  ``write_combined``: for
    arrays the host only writes (inputs); reading them back on the CPU is very slow."""
    dtype = np.dtype(dtype)
    n = int(np.prod(shape)) * dtype.itemsize
    p = (lib().wlsqm_pinned_alloc_wc if write_combined else lib().wlsqm_pinned_alloc)(max(n, 1))
    if not p:
        raise MemoryError(f"cudaHostAlloc({n} bytes) failed")
    buf = (C.c_char * max(n, 1)).from_address(p)
    arr = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)
    _PINNED[arr.ctypes.data] = (buf, p)
    return arr


_PINNED: dict = {}


def pinned_free(arr: np.ndarray):
    ent = _PINNED.pop(arr.ctypes.data, None)
    if ent is not None:
        lib().wlsqm_pinned_free(ent[1])


def meta_summary(nk_a, order_a, knowns_a, wm_a):
    """(max nk, min order, max order, uniform) of the metadata arrays in one C pass (``wlsqm_meta_summary``)"""
    mk, lo, hi, un = C.c_int32(0), C.c_int32(0), C.c_int32(0), C.c_int32(0)
    check(lib().wlsqm_meta_summary(nk_a.shape[0], nk_a.ctypes.data, order_a.ctypes.data, knowns_a.ctypes.data,
                                   wm_a.ctypes.data, C.byref(mk), C.byref(lo), C.byref(hi), C.byref(un)))
    return int(mk.value), int(lo.value), int(hi.value), bool(un.value)


def pool_stats(device=None):
    """(reserved, used) bytes of the library's device memory pool on ``device`` (``wlsqm_pool_stats``); (-1, -1) before
    the first allocation there."""
    r, u = C.c_int64(-1), C.c_int64(-1)
    check(lib().wlsqm_pool_stats(int(default_device() if device is None else device), C.byref(r), C.byref(u)))
    return int(r.value), int(u.value)


def pool_trim(device=None):
    """Return the cached blocks of the library's device memory pool to the driver (``wlsqm_pool_trim``)."""
    check(lib().wlsqm_pool_trim(int(default_device() if device is None else device)))
