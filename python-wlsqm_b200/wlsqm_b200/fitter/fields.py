"""Several fields on one geometry in one pass (extension): ``solve_fields`` / ``solve_hoods_fields``.

A multi-field time step fits several fields (velocity components, temperature, concentration) on the same
neighbourhoods.  The reference does that with one ``solve`` per field, or with guest solvers sharing the host's
matrices (``expert.pyx:243-263``); either way every field streams the whole stored operator again.  These entry points
stream each operator block once per pass for all fields of the pass (``wlsqm_solver_solve_fields`` /
``wlsqm_solver_solve_hoods_fields`` in ``include/wlsqm_b200.h``), and the unknown slots of every field are bit for bit
what a single ``solve`` of that field writes.

Both bindings of ``ExpertSolver`` (the Cython shim and the ctypes twin) call these functions, so that the shape and
stride rules below exist once.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from .. import _lib
from . import opexport


def fi_layout_ok(nf, ncases, maxno, fi_sf, fi_s0):
    """whether the (field, case, slot) -> element map of an fi with these element strides is injective in one of the two
    accepted layouts: fields-outer rows (fi_sf >= (ncases-1)*fi_s0 + max no) or fields-inner rows (fi_sf >= max no,
    fi_s0 >= (nf-1)*fi_sf + max no).  Strides of an axis of length 1 do not matter."""
    if fi_sf < 0 or fi_s0 < 0:
        return False
    outer = (nf <= 1 or fi_sf >= (ncases - 1) * fi_s0 + maxno) and (ncases <= 1 or fi_s0 >= maxno)
    inner = (nf <= 1 or fi_sf >= maxno) and (ncases <= 1 or fi_s0 >= (nf - 1) * fi_sf + maxno)
    return outer or inner


def _no_fields(a, ndim):
    """whether `a` is a float64 array of `ndim` dimensions holding no field (numpy gives such arrays zero strides)"""
    shape, dtype = tuple(getattr(a, "shape", ())), str(getattr(a, "dtype", ""))
    return len(shape) == ndim and shape[0] == 0 and dtype.endswith("float64")


def resolve_fi(fi, ncases, maxno):
    """fi (nf, >= ncases, >= max no) float64, in/out, contiguous last axis -> (Arr, nf, fi_sf, fi_s0)"""
    if _no_fields(fi, 3):
        return None, 0, 0, 0
    a = _lib.as_arr(fi, np.float64, 3, "fi", writable=True)
    nf = a.shape[0]
    if nf and ncases and (a.shape[1] < ncases or a.shape[2] < maxno):
        raise ValueError("fi must have shape (nf, >= ncases = %d, >= max no = %d), got %s" % (ncases, maxno, a.shape))
    fi_sf, fi_s0 = a.strides[0], a.strides[1]
    if nf and ncases and not fi_layout_ok(nf, ncases, maxno, fi_sf, fi_s0):
        raise ValueError("fi: element strides (%d, %d) map two (field, case, slot) entries to one element; use "
                         "fields-outer rows (nf, ncases, no) or fields-inner rows (ncases, nf, no)" % (fi_sf, fi_s0))
    return a, nf, fi_sf, fi_s0


def resolve_fk(fk, nf, ncases, maxnk):
    """fk (nf, >= ncases, >= max nk) float64, any strides (host arrays get a unit last stride) -> (Arr, sf, s0, s1)"""
    a = _lib.as_arr(fk, np.float64, 3, "fk", last_contig=False, allow_copy=True)
    if a.shape[0] != nf:
        raise ValueError("fk holds %d fields, fi %d" % (a.shape[0], nf))
    if nf and ncases and (a.shape[1] < ncases or a.shape[2] < maxnk):
        raise ValueError("fk must have shape (nf, >= ncases = %d, >= max nk = %d), got %s" % (ncases, maxnk, a.shape))
    if not a.is_cuda and maxnk > 1 and a.strides[2] != 1:
        a = _lib.as_arr(np.ascontiguousarray(a.np), np.float64, 3, "fk")
    return a, a.strides[0], a.strides[1], a.strides[2]


def resolve_f(f, nf, npoints):
    """f (nf, >= npoints) float64, any strides (f.T of a (npoints, nf) array is fine) -> (Arr, f_sf, f_s0)"""
    a = _lib.as_arr(f, np.float64, 2, "f", last_contig=False, allow_copy=True)
    if a.shape[0] != nf:
        raise ValueError("f holds %d fields, fi %d" % (a.shape[0], nf))
    if nf and a.shape[1] < npoints:
        raise ValueError("f must hold one value per point of the x given to prepare_hoods() (%d), got %d"
                         % (npoints, a.shape[1]))
    return a, a.strides[0], a.strides[1]


def _ready(solver):
    if not solver.ready:
        raise RuntimeError("Solver is not in the ready state; prepare() must be called before solve()")


def solve_fields(solver, fk, fi):
    """Fit nf fields on the prepared geometry in one pass over the operators.  fk (nf, >= ncases, >= max nk); fi
    (nf, >= ncases, >= max no) in/out.  Returns the maximum of the per-field solve() return values."""
    _ready(solver)
    fi_a, nf, fi_sf, fi_s0 = resolve_fi(fi, solver.ncases, solver._maxno)
    if nf == 0 and _no_fields(fk, 3):
        return 0
    fk_a, fk_sf, fk_s0, fk_s1 = resolve_fk(fk, nf, solver.ncases, solver._maxnk)
    solver._use_stream()
    it = C.c_int32(0)
    _lib.check(_lib.lib().wlsqm_solver_solve_fields(solver._handle, nf, fk_a.ptr, fk_sf, fk_s0, fk_s1, fi_a.ptr, fi_sf,
                                                    fi_s0, C.byref(it)))
    return int(it.value)


def solve_hoods_fields(solver, f, fi):
    """solve_fields with the data per point, f (nf, >= npoints) -- fk[j] = f[j][hoods] gathered on the device (needs
    prepare_hoods)."""
    _ready(solver)
    fi_a, nf, fi_sf, fi_s0 = resolve_fi(fi, solver.ncases, solver._maxno)
    if nf == 0 and _no_fields(f, 2):
        return 0
    f_a, f_sf, f_s0 = resolve_f(f, nf, int(getattr(solver, "_hood_points", 0)))
    solver._use_stream()
    it = C.c_int32(0)
    _lib.check(_lib.lib().wlsqm_solver_solve_hoods_fields(solver._handle, nf, f_a.ptr, f_sf, f_s0, fi_a.ptr, fi_sf, fi_s0,
                                                          C.byref(it)))
    return int(it.value)


def resolve_fi_read(fi, ncases, maxno):
    """fi (nf, >= ncases, >= max no) float64, read only, contiguous last axis -> (Arr, nf, fi_sf, fi_s0); any
    non-negative strides"""
    if _no_fields(fi, 3):
        return None, 0, 0, 0
    a = _lib.as_arr(fi, np.float64, 3, "fi")
    nf = a.shape[0]
    if nf and (a.shape[1] < ncases or a.shape[2] < maxno):
        raise ValueError("fi must have shape (nf, >= ncases = %d, >= max no = %d), got %s" % (ncases, maxno, a.shape))
    return a, nf, a.strides[0], a.strides[1]


def interpolate_fields(solver, x, fi, mode='nearest', r=None, diff=0, I=None):
    """interpolate() for nf caller-held solutions fi (nf, >= ncases, >= max no) -- the fi of solve_fields, say -- in one
    pass over the queries.  Returns (out, I_out): out (nf, nx), or (nf, nx, max no) for diff='all', a CUDA tensor when x
    is one, else numpy; out[j] is bit for bit interpolate(x, mode, r, diff, I)[0] of a solver whose last solve() produced
    fi[j].  Models and I_out are found as interpolate() finds them; the solver's own solution copy is not used."""
    if mode not in ['nearest', 'continuous']:
        raise ValueError("mode must be one of 'nearest', 'continuous'; got '%s'" % mode)
    if mode == 'continuous' and r is None:
        raise ValueError("r must be specified in mode='continuous'")
    if diff is None:
        raise ValueError("diff cannot be None")
    if solver.tree is None:
        raise RuntimeError("Points xi have not been indexed; prep_interpolate() must be called before interpolate()")
    if I is not None and len(I) != len(x):
        raise ValueError("When 'I' is specified, 'I' must have the same length as x; got len(I) = %d, len(x) = %d."
                         % (len(I), len(x)))
    all_diffs = isinstance(diff, str) and diff == 'all'
    if mode == 'continuous' and all_diffs:
        raise ValueError("diff='all' is not available in mode='continuous'")
    cdiff = _lib.DIFF_ALL if all_diffs else int(diff)
    fi_a, nf, fi_sf, fi_s0 = resolve_fi_read(fi, solver.ncases, solver._maxno)
    fi_p = fi_a.ptr if nf else None
    if mode == 'continuous':
        x_a, x_s0, nx = opexport._points(solver, x)
        I_c, I_out = None, np.asanyarray(None)
    else:
        x_a, x_s0, nx, I_c, I_out = opexport._queries(solver, x, I)
    width = solver._maxno if all_diffs else 1
    shape = (nf, nx, width) if all_diffs else (nf, nx)
    if x_a.is_cuda:
        import torch
        out = torch.empty(shape, dtype=torch.float64, device=x_a.keep.device)
        out_p = int(out.data_ptr())
    else:
        out = np.empty(shape, dtype=np.float64)
        out_p = out.ctypes.data
    out_sf, out_sq = nx * width, width
    if mode == 'continuous':
        solver._use_stream()                      # (opexport._queries sets it in nearest mode)
        _lib.check(_lib.lib().wlsqm_solver_interpolate_continuous_fields(solver._handle, nf, fi_p, fi_sf, fi_s0,
                                                                         x_a.ptr, x_s0, nx, float(r), cdiff, out_p,
                                                                         out_sf, out_sq))
        return out, I_out
    # a query that found no neighbour (NaN coordinates) poisons the whole output (expert.pyx:862-870)
    I_cuda = _lib._is_torch_tensor(I_c) and I_c.is_cuda
    if not I_cuda and nx and (I_c == solver.ncases).any():
        out[...] = np.nan
        return out, I_out
    I_p = int(I_c.data_ptr()) if I_cuda else I_c.ctypes.data
    _lib.check(_lib.lib().wlsqm_solver_interpolate_fields(solver._handle, nf, fi_p, fi_sf, fi_s0, x_a.ptr, x_s0, I_p,
                                                          nx, cdiff, out_p, out_sf, out_sq))
    return out, I_out
