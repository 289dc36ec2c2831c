"""Export of the prepared operators: per-case stencil weights and the global sparse operator (extension).

The reference offers the linear map from data to fitted DOFs only as ``sens`` (``impl.pyx:769-779``, d fi / d fk,
recomputed by every solve), from which its callers assemble the Jacobians of implicit steps on the host.  Here the
map that ``prepare`` stored is contracted on the device with caller-given coefficient rows (the Laplacian is
``c[i2_X2] = c[i2_Y2] = 1``) and, for ``prepare_hoods`` solvers, assembled into a CSR matrix over the point cloud.
Definitions: ``include/wlsqm_b200.h`` (``wlsqm_solver_stencils`` / ``wlsqm_solver_operator_csr``).

The interpolation operators do the same at arbitrary query points: the map from the data to
``interpolate(x, mode='nearest', diff)`` (``expert.pyx:687-781``), whose row for query q is the operator of its model
I[q] contracted with the Taylor terms of the offset x[q] - xi[I[q]] (``wlsqm_solver_interp_stencils`` /
``wlsqm_solver_interp_operator_csr``).  For fixed queries one CSR product replaces a solve followed by an interpolate;
mesh-to-mesh transfer, boundary conditions at points that are not fit origins and observation operators are such maps.
With ``mode='continuous'`` they export the map to ``interpolate(x, mode='continuous', r, diff)``, the weighted average of
every model within r: one row per (query, model) pair, each the nearest-mode row of that model scaled by the pair's
normalised weight, and a CSR row per query that merges its pairs (``wlsqm_solver_interp_continuous_*``).  The transpose
of either matrix is the adjoint of the fit-and-interpolate map.

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


def _csr_matrices(rowptr, col, values, shape, cuda):
    if cuda:
        import torch
        return [torch.sparse_csr_tensor(rowptr, col, values[o], size=shape) for o in range(values.shape[0])]
    import scipy.sparse as sp
    return [sp.csr_array((values[o], col, rowptr), shape=shape) for o in range(values.shape[0])]


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
    mats = _csr_matrices(rowptr, col, values, (n, npoints), cuda)
    return (mats[0], K[0]) if squeeze else (mats, K)


def _points(solver, x):
    """-> (x Arr, row stride, nx): the query points for the C ABI"""
    dim = solver.dimension
    x_a = _lib.as_arr(x, np.float64, 2 if dim >= 2 else 1, "x", last_contig=dim >= 2)
    nx = x_a.shape[0]
    if dim >= 2 and x_a.shape[1] < dim:
        raise ValueError("x must have %d coordinates on its last axis" % dim)
    x_s0 = x_a.strides[0] if nx > 1 or dim >= 2 else dim
    if not x_a.is_cuda and dim == 1 and nx > 1 and x_s0 != 1:
        x_a = _lib.as_arr(np.ascontiguousarray(x_a.np), np.float64, 1, "x", last_contig=False)
        x_s0 = 1
    return x_a, x_s0, nx


def _queries(solver, x, I):
    """-> (x Arr, row stride, nx, int64 index array for the C ABI, I_out): the query points and their models, resolved
    as ``interpolate(x, mode='nearest', I=I)`` resolves them (``solver._nearest_models``)."""
    x_a, x_s0, nx = _points(solver, x)
    if I is None and solver.tree is None:
        raise RuntimeError("Points xi have not been indexed; prep_interpolate() must be called before the nearest models "
                           "can be found (or pass I)")
    if I is not None and len(I) != nx:
        raise ValueError("When 'I' is specified, 'I' must have the same length as x; got len(I) = %d, len(x) = %d."
                         % (len(I), nx))
    solver._use_stream()
    I_use, I_out = solver._nearest_models(x, x_a.ptr, x_s0, nx, x_a.is_cuda, I)
    if _lib._is_torch_tensor(I_use) and I_use.is_cuda:
        import torch
        if I_use.dtype != torch.int64 or I_use.dim() != 1 or (nx > 1 and I_use.stride(0) != 1):
            raise ValueError("I: a contiguous int64 tensor of shape (nx,) is required")
        I_c = I_use
    else:
        if _lib._is_torch_tensor(I_use):
            I_use = I_use.detach().cpu().numpy()
        I_c = np.ascontiguousarray(I_use, dtype=np.int64)
        if I_c.ndim != 1:
            raise ValueError("I must be one-dimensional")
    if not (x_a.is_cuda and _lib._is_torch_tensor(I_out)):
        I_out = np.asanyarray(I_out)
    return x_a, x_s0, nx, I_c, I_out


def _mode_args(solver, mode, r, I):
    """-> float r in mode='continuous' (None in nearest mode), after interpolate()'s argument checks"""
    if mode not in ['nearest', 'continuous']:
        raise ValueError("mode must be one of 'nearest', 'continuous'; got '%s'" % mode)
    if mode == 'nearest':
        return None
    if r is None:
        raise ValueError("r must be specified in mode='continuous'")
    if I is not None:
        raise ValueError("I cannot be given in mode='continuous': the models of a query are every origin within r")
    r = float(r)
    if not r > 0.0:
        raise ValueError("r must be positive, got %r" % r)
    if solver.tree is None:
        raise RuntimeError("Points xi have not been indexed; prep_interpolate() must be called before interpolate()")
    return r


def _pairs(solver, x_a, x_s0, nx, r, cuda, center=None):
    """-> (pair_ptr (nx + 1,) int64, npairs, nnz): the count call of the continuous-mode operators; nnz of the CSR
    with that center (-1: no folding) is counted when center is given, else it is None"""
    pair_ptr = _empty((nx + 1,), np.int64, cuda, solver.device)
    npairs, nnz = C.c_int64(0), C.c_int64(0)
    solver._use_stream()
    _lib.check(_lib.lib().wlsqm_solver_interp_continuous_count(solver._handle, x_a.ptr, x_s0, nx, r,
                                                               -1 if center is None else center, _ptr(pair_ptr),
                                                               C.byref(npairs), None if center is None else C.byref(nnz)))
    return pair_ptr, int(npairs.value), (None if center is None else int(nnz.value))


def _center_arg(center):
    if center is None:
        return -1
    center = int(center)
    if center < 0:
        raise ValueError("center must be >= 0, got %d" % center)
    return center


def interp_stencils(solver, x, coeffs=0, I=None, mode='nearest', r=None):
    """(W, K, I_out): the interpolation operators at the query points x as per-query weights.

    W (nops, nx, max nk) weights on the data of model I[q]'s neighbours, K (nops, nx, max no) on its known values, so
    that for an ALGO_BASIC solve  sum_D coeffs[D] d^D f(x[q]) = W[q] . fk[I[q]] + K[q] . fi[I[q]]  with d^D f the value
    interpolate(x, mode='nearest', diff=D) returns.  The nops axis is dropped for an int slot or a 1-D row.  I=None: the
    nearest models, found as interpolate() finds them (I_out returns them); a query without a model (I outside
    [0, ncases)) has W row 0 and K row NaN.  CUDA tensors when the solver was prepared from CUDA tensors.

    mode='continuous' (r required, I refused): the map to interpolate(x, mode='continuous', r), returned as
    (W, K, (pair_ptr, J)).  The pairs (q, J[p]) for p in [pair_ptr[q], pair_ptr[q+1]) are the models within r of x[q] in
    ascending order; W (nops, npairs, max nk) and K (nops, npairs, max no) are their rows, the nearest-mode rows of
    model J[p] at x[q] scaled by the normalised weight of the pair, so that
    sum_D coeffs[D] d^D f(x[q]) = sum over the pairs p of q of W[p] . fk[J[p]] + K[p] . fi[J[p]].  A query without a
    model has an empty pair range."""
    r = _mode_args(solver, mode, r, I)
    c, squeeze = coefficient_rows(coeffs, solver._maxno)
    if r is not None:
        return _continuous_stencils(solver, x, c, squeeze, r)
    x_a, x_s0, nx, I_c, I_out = _queries(solver, x, I)
    root = _root(solver)
    cuda = getattr(root, "_cuda_out", False)
    nops = c.shape[0]
    W = _empty((nops, nx, solver._maxnk), np.float64, cuda, solver.device)
    K = _empty((nops, nx, solver._maxno), np.float64, cuda, solver.device)
    _lib.check(_lib.lib().wlsqm_solver_interp_stencils(solver._handle, x_a.ptr, x_s0, _ptr(I_c), nx, nops, c.ctypes.data,
                                                       _ptr(W), _ptr(K)))
    return (W[0], K[0], I_out) if squeeze else (W, K, I_out)


def _continuous_stencils(solver, x, c, squeeze, r):
    x_a, x_s0, nx = _points(solver, x)
    cuda = getattr(_root(solver), "_cuda_out", False)
    pair_ptr, npairs, _ = _pairs(solver, x_a, x_s0, nx, r, cuda)
    nops = c.shape[0]
    J = _empty((npairs,), np.int64, cuda, solver.device)
    W = _empty((nops, npairs, solver._maxnk), np.float64, cuda, solver.device)
    K = _empty((nops, npairs, solver._maxno), np.float64, cuda, solver.device)
    _lib.check(_lib.lib().wlsqm_solver_interp_continuous_stencils(solver._handle, x_a.ptr, x_s0, nx, r, nops, c.ctypes.data,
                                                                  _ptr(pair_ptr), _ptr(J), _ptr(W), _ptr(K)))
    return (W[0], K[0], (pair_ptr, J)) if squeeze else (W, K, (pair_ptr, J))


def interp_operator(solver, x, coeffs=0, I=None, center=None, mode='nearest', r=None):
    """(E, K, I_out): the interpolation operators as a sparse matrix over the points of ``prepare_hoods``.

    E (nx, npoints), rows in the order of x: a ``torch.sparse_csr_tensor`` or a ``scipy.sparse.csr_array`` by the rule
    of ``operator()`` (a list of nops matrices sharing one index pair for 2-D coeffs), so that
    sum_D coeffs[D] d^D f(x[q]) = (E @ f)[q] + K[q] . fi[I[q]].  ``center``: index in x of case 0's own point; the weight
    on a known F of model I[q] then moves into column center + I[q] and is 0 in K.  A query without a model has an
    empty row and a NaN K row.

    mode='continuous' (r required, I refused): (E, K, (pair_ptr, J)) for interpolate(x, mode='continuous', r), with K per
    pair as in interp_stencils, so that sum_D coeffs[D] d^D f(x[q]) = (E @ f)[q] + sum over the pairs p of q of
    K[p] . fi[J[p]]; with ``center`` the known-F weight of each pair moves into column center + J[p].  A query without a
    model has an empty row."""
    r = _mode_args(solver, mode, r, I)
    c, squeeze = coefficient_rows(coeffs, solver._maxno)
    center = _center_arg(center)
    if r is not None:
        return _continuous_operator(solver, x, c, squeeze, r, center)
    x_a, x_s0, nx, I_c, I_out = _queries(solver, x, I)
    root = _root(solver)
    L = _lib.lib()
    nnz = C.c_int64(0)
    _lib.check(L.wlsqm_solver_interp_operator_nnz(solver._handle, _ptr(I_c), nx, center, C.byref(nnz)))
    nnz = int(nnz.value)
    cuda = getattr(root, "_cuda_out", False)
    nops, npoints = c.shape[0], int(getattr(root, "_hood_points", 0))
    bits = 32 if nnz < 2 ** 31 else 64
    it = np.int32 if bits == 32 else np.int64
    rowptr = _empty((nx + 1,), it, cuda, solver.device)
    col = _empty((nnz,), it, cuda, solver.device)
    values = _empty((nops, nnz), np.float64, cuda, solver.device)
    K = _empty((nops, nx, solver._maxno), np.float64, cuda, solver.device)
    _lib.check(L.wlsqm_solver_interp_operator_csr(solver._handle, x_a.ptr, x_s0, _ptr(I_c), nx, nops, c.ctypes.data,
                                                  center, bits, _ptr(rowptr), _ptr(col), _ptr(values), _ptr(K)))
    mats = _csr_matrices(rowptr, col, values, (nx, npoints), cuda)
    return (mats[0], K[0], I_out) if squeeze else (mats, K, I_out)


def _continuous_operator(solver, x, c, squeeze, r, center):
    x_a, x_s0, nx = _points(solver, x)
    root = _root(solver)
    cuda = getattr(root, "_cuda_out", False)
    pair_ptr, npairs, nnz = _pairs(solver, x_a, x_s0, nx, r, cuda, center=center)
    nops, npoints = c.shape[0], int(getattr(root, "_hood_points", 0))
    bits = 32 if nnz < 2 ** 31 else 64
    it = np.int32 if bits == 32 else np.int64
    J = _empty((npairs,), np.int64, cuda, solver.device)
    rowptr = _empty((nx + 1,), it, cuda, solver.device)
    col = _empty((nnz,), it, cuda, solver.device)
    values = _empty((nops, nnz), np.float64, cuda, solver.device)
    K = _empty((nops, npairs, solver._maxno), np.float64, cuda, solver.device)
    _lib.check(_lib.lib().wlsqm_solver_interp_continuous_operator_csr(
        solver._handle, x_a.ptr, x_s0, nx, r, nops, c.ctypes.data, center, bits, _ptr(pair_ptr), _ptr(J), _ptr(rowptr),
        _ptr(col), _ptr(values), _ptr(K)))
    mats = _csr_matrices(rowptr, col, values, (nx, npoints), cuda)
    return (mats[0], K[0], (pair_ptr, J)) if squeeze else (mats, K, (pair_ptr, J))
