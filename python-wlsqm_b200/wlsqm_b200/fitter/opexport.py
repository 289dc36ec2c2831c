"""Export of the prepared operators: per-case stencil weights and the global sparse operator (extension).

The reference offers the linear map from data to fitted DOFs only as ``sens`` (``impl.pyx:769-779``, d fi / d fk,
recomputed by every solve), from which its callers assemble the Jacobians of implicit steps on the host.  Here the
map that ``prepare`` stored is contracted on the device with caller-given coefficient rows (the Laplacian is
``c[i2_X2] = c[i2_Y2] = 1``) and, for ``prepare_hoods`` solvers, assembled into a CSR matrix over the point cloud.
Definitions: ``include/wlsqm_b200.h`` (``wlsqm_solver_stencils`` / ``wlsqm_solver_operator_csr``).

Both bindings of ``ExpertSolver`` (the Cython shim and the ctypes twin) call these functions.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from .. import _lib

MAXNO = 35


def _root(solver):
    """the solver whose operators and neighbour lists a guest borrows (itself if it is not a guest)"""
    while getattr(solver, "host", None) is not None and getattr(solver, "_borrows", False):
        solver = solver.host
    return solver


def coefficient_rows(coeffs, maxno):
    """-> (float64 (nops, maxno) C-contiguous, whether the nops axis is dropped from the outputs).

    ``coeffs``: an int slot (one-hot row), a 1-D array (maxno,) or a 2-D array (nops, maxno), 1 <= nops <= 35."""
    if isinstance(coeffs, (int, np.integer)) and not isinstance(coeffs, (bool, np.bool_)):
        slot = int(coeffs)
        if not 0 <= slot < maxno:
            raise ValueError("slot %d is outside [0, %d)" % (slot, maxno))
        c = np.zeros((1, maxno), dtype=np.float64)
        c[0, slot] = 1.0
        return c, True
    if _lib._is_torch_tensor(coeffs):
        coeffs = coeffs.detach().cpu().numpy()
    c = np.asarray(coeffs, dtype=np.float64)
    if c.ndim == 1:
        if c.shape[0] != maxno:
            raise ValueError("coeffs must have shape (%d,), got %s" % (maxno, c.shape))
        c, squeeze = c[None, :], True
    elif c.ndim == 2:
        if c.shape[1] != maxno or not 1 <= c.shape[0] <= MAXNO:
            raise ValueError("coeffs must have shape (nops, %d) with 1 <= nops <= %d, got %s" % (maxno, MAXNO, c.shape))
        squeeze = False
    else:
        raise ValueError("coeffs must be a slot index, a 1-D or a 2-D array")
    if not np.isfinite(c).all():
        raise ValueError("coeffs must be finite")
    return np.ascontiguousarray(c), squeeze


def _empty(shape, dtype, cuda, device):
    if cuda:
        import torch
        return torch.empty(shape, dtype={np.float64: torch.float64, np.int32: torch.int32, np.int64: torch.int64}[dtype],
                           device=torch.device("cuda", device))
    return np.empty(shape, dtype=dtype)


def _ptr(a):
    return a.data_ptr() if _lib._is_torch_tensor(a) else a.ctypes.data


def stencils(solver, coeffs):
    """(W, K): W (nops, ncases, max nk) stencil weights on fk, K (nops, ncases, max no) weights on the known values;
    the nops axis is dropped for an int slot or a 1-D coefficient row.  CUDA tensors when the solver was prepared
    from CUDA tensors, numpy arrays otherwise."""
    c, squeeze = coefficient_rows(coeffs, solver._maxno)
    root = _root(solver)
    cuda = getattr(root, "_cuda_out", False)
    nops, n = c.shape[0], solver.ncases
    W = _empty((nops, n, solver._maxnk), np.float64, cuda, solver.device)
    K = _empty((nops, n, solver._maxno), np.float64, cuda, solver.device)
    solver._use_stream()
    _lib.check(_lib.lib().wlsqm_solver_stencils(solver._handle, nops, c.ctypes.data, _ptr(W), _ptr(K)))
    return (W[0], K[0]) if squeeze else (W, K)


def operator(solver, coeffs, center=None):
    """(D, K): the global sparse operator over the points x of ``prepare_hoods`` and the known-value weights.

    D (ncases, npoints): a ``torch.sparse_csr_tensor`` on the solver's device when ``prepare_hoods`` got CUDA tensors,
    a ``scipy.sparse.csr_array`` otherwise; int32 indices when nnz < 2^31, int64 beyond.  For 2-D coeffs a list of
    nops matrices sharing one index pair.  ``center``: index in x of case 0's own point; then the weight on a known F
    (slot 0) of case i moves into column center + i of D and is 0 in K."""
    c, squeeze = coefficient_rows(coeffs, solver._maxno)
    if center is None:
        center = -1
    else:
        center = int(center)
        if center < 0:
            raise ValueError("center must be >= 0, got %d" % center)
    root = _root(solver)
    L = _lib.lib()
    solver._use_stream()
    nnz = C.c_int64(0)
    _lib.check(L.wlsqm_solver_operator_nnz(solver._handle, center, C.byref(nnz)))
    nnz = int(nnz.value)
    cuda = getattr(root, "_cuda_out", False)
    nops, n, npoints = c.shape[0], solver.ncases, int(getattr(root, "_hood_points", 0))
    bits = 32 if nnz < 2 ** 31 else 64
    it = np.int32 if bits == 32 else np.int64
    rowptr = _empty((n + 1,), it, cuda, solver.device)
    col = _empty((nnz,), it, cuda, solver.device)
    values = _empty((nops, nnz), np.float64, cuda, solver.device)
    K = _empty((nops, n, solver._maxno), np.float64, cuda, solver.device)
    _lib.check(L.wlsqm_solver_operator_csr(solver._handle, nops, c.ctypes.data, center, bits, _ptr(rowptr), _ptr(col),
                                           _ptr(values), _ptr(K)))
    if cuda:
        import torch
        mats = [torch.sparse_csr_tensor(rowptr, col, values[o], size=(n, npoints)) for o in range(nops)]
    else:
        import scipy.sparse as sp
        mats = [sp.csr_array((values[o], col, rowptr), shape=(n, npoints)) for o in range(nops)]
    return (mats[0], K[0]) if squeeze else (mats, K)
