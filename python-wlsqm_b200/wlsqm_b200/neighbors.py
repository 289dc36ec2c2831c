"""Neighbourhood construction and nearest-point search on the GPU (extension; SURVEY.md 8f items 1-2).

The reference leaves these steps to the caller and to ``scipy.spatial.cKDTree`` on the host:

    tree  = scipy.spatial.cKDTree(x)
    hoods = tree.query(x, k + 1)[1][:, 1:]           # examples/expertsolver_example.py:59-66
    xk, fk = x[hoods], f[hoods]

At a million points the kd-tree query costs seconds while the fit costs milliseconds, so the same searches are
offered on the device (uniform grid, exact k nearest neighbours ordered by (distance, index); identical to
cKDTree wherever distances are distinct):

    grid  = wlsqm_b200.PointGrid(x)                  # x: numpy array or CUDA tensor, (n, dim) or (n,)
    hoods = grid.knn(k)                              # (n, k) int32, self excluded
    d, I  = grid.query(xq, k=1)                      # like cKDTree.query
    rowptr, col = grid.ball(r)                       # fixed-radius lists (CSR), like cKDTree.query_ball_point
    hoods, nk = wlsqm_b200.ball_hoods(x, r)          # ragged radius neighbourhoods for ExpertSolver(nk=nk)

``ExpertSolver.prepare_hoods(x, hoods)`` / ``solve_hoods(f, fi)`` take the index lists directly.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib

__all__ = ["PointGrid", "knn_hoods", "ball_hoods", "gather"]

_BALL_ORDER = {"index": 0, "distance": 1}


def _points(x, name="x"):
    """(n, dim) or (n,) float64, numpy or CUDA tensor -> (Arr, n, dim, row stride)"""
    nd = x.dim() if _lib._is_torch_tensor(x) else np.ndim(x)
    if nd == 1:
        a = _lib.as_arr(x, np.float64, 1, name, last_contig=False)
        return a, a.shape[0], 1, (a.strides[0] if a.shape[0] > 1 else 1)
    a = _lib.as_arr(x, np.float64, 2, name)
    if a.shape[1] not in (1, 2, 3):
        raise ValueError(f"{name}: points must have 1, 2 or 3 coordinates, got {a.shape[1]}")
    return a, a.shape[0], a.shape[1], a.strides[0]


class PointGrid:
    """Uniform search grid over a point cloud, resident on one GPU."""

    def __init__(self, x, device=None):
        a, n, dim, s0 = _points(x)
        if device is None:
            device = a.device if a.is_cuda else _lib.default_device()
        self.device, self.n, self.dimension = int(device), n, dim
        self._on_device = a.is_cuda
        self._torch_device = x.device if a.is_cuda else None
        h = C.c_void_p()
        _lib.announce_stream(self.device)
        _lib.check(_lib.lib().wlsqm_grid_create(dim, n, a.ptr, s0, self.device, C.byref(h)))
        self._handle = h

    def close(self):
        h, self._handle = getattr(self, "_handle", None), None
        if h is not None and h.value:
            _lib.lib().wlsqm_grid_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def info(self):
        """(number of cells, cell edge length, device bytes)"""
        nc, hh, nb = C.c_int64(), C.c_double(), C.c_int64()
        _lib.check(_lib.lib().wlsqm_grid_info(self._handle, C.byref(nc), C.byref(hh), C.byref(nb)))
        return nc.value, hh.value, nb.value

    def _out(self, shape, np_dtype, on_device):
        if on_device:
            import torch
            t = torch.empty(shape, dtype=getattr(torch, np.dtype(np_dtype).name), device=self._torch_device or f"cuda:{self.device}")
            return t, int(t.data_ptr())
        a = np.empty(shape, dtype=np_dtype)
        return a, a.ctypes.data

    def knn(self, k, exclude_self=True, return_distance=False):
        """The k nearest neighbours of every point of the cloud: (n, k) int32, nearest first; with
        ``exclude_self`` the point itself is left out (``tree.query(x, k+1)[1][:, 1:]``)."""
        k = int(k)
        idx, ip = self._out((self.n, k), np.int32, self._on_device)
        d2, dp = (self._out((self.n, k), np.float64, self._on_device) if return_distance else (None, None))
        _lib.announce_stream(self.device)
        _lib.check(_lib.lib().wlsqm_grid_knn(self._handle, None, 0, self.n, k, 1 if exclude_self else 0, ip, None, dp))
        if return_distance:
            return (d2.sqrt() if self._on_device else np.sqrt(d2)), idx
        return idx

    def query(self, xq, k=1):
        """``cKDTree.query(xq, k)``: (distances, indices); indices are int64 (``np.int_``), missing neighbours n."""
        a, nq, dim, s0 = _points(xq, "xq")
        if dim != self.dimension:
            raise ValueError("xq has %d coordinates, the grid has %d" % (dim, self.dimension))
        k = int(k)
        idx, ip = self._out((nq, k), np.int64, a.is_cuda)
        d2, dp = self._out((nq, k), np.float64, a.is_cuda)
        if nq:
            _lib.announce_stream(self.device)
            _lib.check(_lib.lib().wlsqm_grid_knn(self._handle, a.ptr, s0, nq, k, 0, None, ip, dp))
        d = d2.sqrt() if a.is_cuda else np.sqrt(d2)
        if k == 1:
            return d[:, 0], idx[:, 0]
        return d, idx

    def ball(self, r, xq=None, *, exclude_self=None, max_k=None, order="index"):
        """Fixed-radius neighbourhoods as CSR lists: ``(rowptr int64 (nq+1,), col int32 (nnz,))``; row q holds the
        grid points within ``r`` of query q (``d2 <= r*r``, the exact rule is in ``include/wlsqm_b200.h``).

        ``xq=None``: the queries are the grid's own points and ``exclude_self`` (default True) leaves each point out of
        its own row (coincident points stay).  ``r``: a scalar or one radius per query (numpy or CUDA tensor), >= 0,
        ``inf`` allowed.  ``order='index'`` sorts each row by index (``query_ball_point``'s order), ``'distance'`` by
        (distance, index).  ``max_k`` (1..128) keeps the ``max_k`` nearest members of each row.  Points with non-finite
        coordinates are never members; a query with a NaN or infinite coordinate gets an empty row.  The outputs are
        CUDA tensors when the queries are (for ``xq=None``: when the grid was built from a CUDA tensor), else numpy."""
        if max_k is None:
            max_k = 0
        else:
            max_k = int(max_k)
            if not 1 <= max_k <= 128:
                raise ValueError("max_k must be between 1 and 128, got %d" % max_k)
        if order not in _BALL_ORDER:
            raise ValueError("order must be 'index' or 'distance', got %r" % (order,))
        empty = False
        if xq is None:
            nq, on_device, xq_ptr, s0 = self.n, self._on_device, None, 0
            exclude_self = True if exclude_self is None else bool(exclude_self)
        else:
            if exclude_self:
                raise ValueError("exclude_self applies to the grid's own points only (xq=None)")
            exclude_self = False
            if np.ndim(xq) >= 1 and len(xq) == 0:         # no queries: an empty CSR, after the checks below
                if np.ndim(xq) == 2 and xq.shape[1] != self.dimension:
                    raise ValueError("xq has %d coordinates, the grid has %d" % (xq.shape[1], self.dimension))
                nq, on_device, empty = 0, _lib._is_torch_tensor(xq) and xq.is_cuda, True
            else:
                a, nq, dim, s0 = _points(xq, "xq")
                if dim != self.dimension:
                    raise ValueError("xq has %d coordinates, the grid has %d" % (dim, self.dimension))
                on_device, xq_ptr = a.is_cuda, a.ptr
        r_keep, r_ptr, r_s0 = self._radii(r, nq)
        if empty:
            return self._out((1,), np.int64, on_device)[0] * 0, self._out((0,), np.int32, on_device)[0]
        rowptr, rp = self._out((nq + 1,), np.int64, on_device)
        nnz = C.c_int64(0)
        L = _lib.lib()
        _lib.announce_stream(self.device)
        _lib.check(L.wlsqm_grid_ball_count(self._handle, xq_ptr, s0, nq, r_ptr, r_s0, int(exclude_self), max_k, rp, None,
                                           C.byref(nnz)))
        col, cp = self._out((nnz.value,), np.int32, on_device)
        _lib.announce_stream(self.device)
        _lib.check(L.wlsqm_grid_ball_csr(self._handle, xq_ptr, s0, nq, r_ptr, r_s0, int(exclude_self), max_k,
                                         _BALL_ORDER[order], rp, cp))
        del r_keep
        return rowptr, col

    @staticmethod
    def _radii(r, nq):
        """r -> (object keeping the buffer alive, pointer, stride); validated: length nq or scalar, >= 0, not NaN"""
        if _lib._is_torch_tensor(r) and r.dim() == 0:
            if not r.is_cuda:
                r = float(r)
            else:                                           # one radius in device memory (stride 0)
                import torch
                r = r.to(torch.float64).reshape(1)
                if not bool((r >= 0).all()):
                    raise ValueError("r must be >= 0 and not NaN")
                return r, int(r.data_ptr()), 0
        if _lib._is_torch_tensor(r):
            a = _lib.as_arr(r, np.float64, 1, "r", last_contig=False)
            if a.shape[0] != nq:
                raise ValueError("r has %d entries for %d queries" % (a.shape[0], nq))
            if a.is_cuda:
                if nq and not bool((r >= 0).all()):        # (False for NaN too)
                    raise ValueError("r must be >= 0 and not NaN")
                return r, a.ptr, a.strides[0]
            r = a.np
        ra = np.asarray(r, dtype=np.float64) if not isinstance(r, np.ndarray) else r
        if ra.ndim == 0:
            ra = np.array([float(ra)])
            s0 = 0
        else:
            if ra.dtype != np.float64:
                ra = ra.astype(np.float64)
            if ra.ndim != 1 or ra.shape[0] != nq:
                raise ValueError("r must be a scalar or have one entry per query (%d), got shape %s" % (nq, ra.shape))
            ra = np.ascontiguousarray(ra)
            s0 = 1
        if not (ra >= 0).all():
            raise ValueError("r must be >= 0 and not NaN")
        return ra, ra.ctypes.data, s0

    def query_ball_point(self, x, r, return_sorted=None, return_length=False):
        """``cKDTree.query_ball_point(x, r)`` for host arrays: an object array of index lists (a list for a single
        point), or their lengths with ``return_length``.  The lists are always sorted by index (``return_sorted`` is
        accepted for compatibility) and include a query's own point.  CUDA tensors: use ``ball``."""
        if _lib._is_torch_tensor(x) and x.is_cuda:
            raise ValueError("query_ball_point takes host arrays; for CUDA tensors use PointGrid.ball (CSR on the device)")
        x = np.asarray(x, dtype=np.float64)
        single = x.ndim == 1 and self.dimension > 1 or x.ndim == 0
        xq = x.reshape(1, -1) if single else x
        rowptr, col = self.ball(r if np.ndim(r) == 0 else np.asarray(r, dtype=np.float64).reshape(-1), xq)
        counts = np.diff(rowptr)
        if return_length:
            return int(counts[0]) if single else counts.astype(np.intp)
        lists = np.split(col.astype(np.intp), rowptr[1:-1])
        if single:
            return lists[0].tolist()
        out = np.empty(len(lists), dtype=object)
        for i, l in enumerate(lists):
            out[i] = l.tolist()
        return out


def knn_hoods(x, k, device=None):
    """hoods = cKDTree(x).query(x, k+1)[1][:, 1:] on the GPU: (n, k) int32."""
    g = PointGrid(x, device=device)
    try:
        return g.knn(k)
    finally:
        g.close()


def ball_hoods(x, r, max_k=None, device=None):
    """Radius neighbourhoods of every point, self excluded, for ``ExpertSolver(dim, nk, ...)`` and
    ``prepare_hoods(x, hoods)``: ``(hoods (n, width) int32, nk (n,) int32)`` with ``width = max(nk)`` (at least 1),
    each row ascending by index and padded with ``n``.  Row i is ``cKDTree(x).query_ball_point(x[i], r)`` without i;
    with ``max_k`` only its ``max_k`` nearest points.  CUDA tensors in, CUDA tensors out."""
    g = PointGrid(x, device=device)
    try:
        rowptr, col = g.ball(r, max_k=max_k)
    finally:
        g.close()
    n = g.n
    if _lib._is_torch_tensor(rowptr):
        import torch
        nk = (rowptr[1:] - rowptr[:-1]).to(torch.int32)
        width = max(int(nk.max()) if n else 0, 1)
        hoods = torch.full((n, width), n, dtype=torch.int32, device=rowptr.device)
        rows = torch.repeat_interleave(torch.arange(n, device=rowptr.device), nk.long())
        pos = torch.arange(col.shape[0], device=rowptr.device) - rowptr[:-1][rows]
        hoods[rows, pos] = col
        return hoods, nk
    nk = np.diff(rowptr).astype(np.int32)
    width = max(int(nk.max()) if n else 0, 1)
    hoods = np.full((n, width), n, dtype=np.int32)
    rows = np.repeat(np.arange(n), nk)
    hoods[rows, np.arange(col.shape[0]) - rowptr[:-1][rows]] = col
    return hoods, nk


def gather(src, hoods):
    """``src[hoods]`` on the device: src (npoints,) or (npoints, w) float64 CUDA tensor, hoods (n, k) int32 CUDA
    tensor -> (n, k) or (n, k, w)."""
    import torch
    if not (_lib._is_torch_tensor(src) and src.is_cuda and _lib._is_torch_tensor(hoods) and hoods.is_cuda):
        raise ValueError("gather() works on CUDA tensors (numpy arrays: use src[hoods])")
    if hoods.dtype != torch.int32 or hoods.dim() != 2 or hoods.stride(1) != 1:
        raise ValueError("hoods must be a (n, k) int32 tensor with contiguous rows")
    if src.dtype != torch.float64:
        raise ValueError("src must be float64")
    w = 1 if src.dim() == 1 else src.shape[1]
    if src.dim() == 2 and src.stride(1) != 1:
        src = src.contiguous()
    n, k = hoods.shape
    out = torch.empty((n, k) if src.dim() == 1 else (n, k, w), dtype=torch.float64, device=src.device)
    sp = _lib.current_stream_ptr(src.device.index)
    _lib.check(_lib.lib().wlsqm_gather_hoods(int(src.data_ptr()), src.stride(0), w, src.shape[0], int(hoods.data_ptr()),
                                             hoods.stride(0), n, k, int(out.data_ptr()), src.device.index, sp))
    return out
