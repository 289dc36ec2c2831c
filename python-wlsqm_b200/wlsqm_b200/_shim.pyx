# cython: language_level=3
# cython: boundscheck=False
# cython: wraparound=False
# cython: cdivision=True
"""The Cython C-ABI shim: ``ExpertSolver``, ``number_of_dofs`` and the 18 ``fit_*`` functions bound directly to
``libwlsqm_b200.so`` (``cdef extern from "wlsqm_b200.h"``).

The reference's own Python layer is Cython (``wlsqm/fitter/expert.pyx``, ``simple.pyx``); this is its counterpart over
the B200 library, with the reference's typed signatures: integer arguments are C ``int`` (``None`` -> Cython's
``TypeError: an integer is required``, as from the compiled reference), host arrays are coerced to the reference's
memoryview layouts (``expert.pyx:92-93, 309, 467, 687``; ``simple.pyx:131-163, 379-398``), so dtype / ndim / layout
errors are Cython's own ``ValueError`` / ``TypeError``, and the C calls run ``with nogil``.  CUDA ``torch.Tensor``
arguments (an extension: zero copy, asynchronous on torch's current stream) carry no buffer protocol and take a
pointer path instead.  ``wlsqm_b200.fitter.expert`` / ``.simple`` fall back to their ctypes twins when this module has
not been built (``WLSQM_BINDING=ctypes`` forces that).
"""
import ctypes as _C
import sys as _sys

import numpy as np

from cython cimport view
from libc.stdint cimport int32_t, int64_t, uintptr_t

from .fitter import defs
from . import _lib
from .fitter import opexport as _opexport
from .fitter import fields as _fields

cdef extern from "wlsqm_b200.h" nogil:
    ctypedef struct wlsqm_solver_t:
        pass
    const char* wlsqm_last_error()
    int wlsqm_device_count()
    int wlsqm_meta_summary(int64_t ncases, const int32_t* nk, const int32_t* order, const int64_t* knowns, const int32_t* wm,
                           int32_t* max_nk, int32_t* min_order, int32_t* max_order, int32_t* uniform)
    int wlsqm_solver_create(int dimension, int64_t ncases, const int32_t* nk, const int32_t* order, const int64_t* knowns,
                            const int32_t* wm, int algorithm, int do_sens, int max_iter, int debug, int device,
                            wlsqm_solver_t** out)
    int wlsqm_solver_create_guest(wlsqm_solver_t* host, int algorithm, int do_sens, int max_iter, wlsqm_solver_t** out)
    int wlsqm_solver_prepare_guest(wlsqm_solver_t* s)
    int wlsqm_solver_destroy(wlsqm_solver_t* s)
    int wlsqm_solver_set_stream(wlsqm_solver_t* s, void* cuda_stream)
    int wlsqm_solver_keep_solution(wlsqm_solver_t* s, int keep)
    int wlsqm_solver_synchronize(wlsqm_solver_t* s)
    int wlsqm_set_caller_stream(void* cuda_stream)
    int wlsqm_solver_prepare(wlsqm_solver_t* s, const double* xi, int64_t xi_s0, const double* xk, int64_t xk_s0, int64_t xk_s1)
    int wlsqm_solver_solve(wlsqm_solver_t* s, const double* fk, int64_t fk_s0, int64_t fk_s1, double* fi, int64_t fi_s0,
                           double* sens, int64_t sens_s0, int64_t sens_s1, int32_t* iters_out)
    int wlsqm_solver_iterations(wlsqm_solver_t* s, int32_t* out)
    int wlsqm_solver_interpolate(wlsqm_solver_t* s, const double* x, int64_t x_s0, const int64_t* I, int64_t nx, int diff,
                                 double* out, int64_t out_s0)
    int wlsqm_solver_conds(wlsqm_solver_t* s, double* out)
    int wlsqm_solver_memory(wlsqm_solver_t* s, int64_t* used, int64_t* total)
    int wlsqm_fit_many(int dimension, int64_t ncases, const double* xk, int64_t xk_s0, int64_t xk_s1, const double* fk,
                       int64_t fk_s0, int64_t fk_s1, const int32_t* nk, const double* xi, int64_t xi_s0, double* fi,
                       int64_t fi_s0, double* sens, int64_t sens_s0, int64_t sens_s1, int do_sens, const int32_t* order,
                       const int64_t* knowns, const int32_t* wm, int algorithm, int max_iter, int device, int32_t* iters_out)
    int wlsqm_solver_prepare_hoods(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t npoints, const int32_t* hoods,
                                   int64_t hoods_s0, const double* xi, int64_t xi_s0)
    int wlsqm_solver_solve_hoods(wlsqm_solver_t* s, const double* f, int64_t f_s0, double* fi, int64_t fi_s0, double* sens,
                                 int64_t sens_s0, int64_t sens_s1, int32_t* iters_out)
    int wlsqm_solver_stencils(wlsqm_solver_t* s, int nops, const double* coeffs, double* W, double* K)
    int wlsqm_solver_operator_nnz(wlsqm_solver_t* s, int64_t center, int64_t* nnz)
    int wlsqm_solver_operator_csr(wlsqm_solver_t* s, int nops, const double* coeffs, int64_t center, int index_bits,
                                  void* rowptr, void* col, double* values, double* K)
    int wlsqm_solver_index_models(wlsqm_solver_t* s)
    int wlsqm_solver_nearest_models(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, int64_t* I_out)
    int wlsqm_solver_interpolate_continuous(wlsqm_solver_t* s, const double* x, int64_t x_s0, int64_t nx, double r, int diff,
                                            double* out)

DEF E_VALUE = -1
DEF E_MEMORY = -2
DEF DIFF_ALL = -1

BINDING = "cython"

__all__ = ["number_of_dofs", "ExpertSolver"] + [f"fit_{d}D{it}{many}" for d in (1, 2, 3) for it in ("", "_iterative")
                                                for many in ("", "_many", "_many_parallel")]


cdef int _check(int rc) except -1:
    """map a C-ABI return code to the reference's exception surface (expert.pyx:131-189, 493-494, 673-674, 742-743)"""
    if rc == 0:
        return 0
    msg = (<bytes>wlsqm_last_error()).decode("utf-8", "replace")
    if rc == E_VALUE:
        raise ValueError(msg)
    if rc == E_MEMORY:
        raise MemoryError(msg)
    raise RuntimeError(msg)


# ---- array arguments ---------------------------------------------------------------------------------------------------
cdef struct Arr:
    double* p
    Py_ssize_t n0, n1, n2
    Py_ssize_t s0, s1, s2        # element strides
    bint cuda
    int device

cdef object _torch = None


cdef inline bint _is_tensor(object a):
    global _torch
    if _torch is None:
        _torch = _sys.modules.get("torch")
        if _torch is None:
            return False
    return isinstance(a, _torch.Tensor)


cdef int _tensor(object a, int ndim, str name, Arr* out, bint last_contig, list keep) except -1:
    """a CUDA torch.Tensor: pointer and element strides (no buffer protocol there); dtype / ndim are checked like the
    memoryview coercion checks them"""
    if a.dtype != _torch.float64:
        raise ValueError("%s: Buffer dtype mismatch, expected 'double' but got '%s'" % (name, a.dtype))
    if a.dim() != ndim:
        raise ValueError("%s: Buffer has wrong number of dimensions (expected %d, got %d)" % (name, ndim, a.dim()))
    shp, st = a.shape, a.stride()
    out.n0 = shp[0]; out.s0 = st[0]
    out.n1 = shp[1] if ndim > 1 else 1
    out.s1 = st[1] if ndim > 1 else 1
    out.n2 = shp[2] if ndim > 2 else 1
    out.s2 = st[2] if ndim > 2 else 1
    if last_contig and ndim > 0 and shp[ndim - 1] > 1 and st[ndim - 1] != 1:
        raise ValueError("%s: last axis must be contiguous" % name)
    out.p = <double*><uintptr_t>a.data_ptr()
    out.cuda = True
    out.device = a.device.index
    keep.append(a)
    return 0


cdef int _arr1(object a, str name, Arr* out, list keep) except -1:
    """double[::view.generic]"""
    cdef double[::view.generic] v
    if _is_tensor(a):
        if a.is_cuda:
            return _tensor(a, 1, name, out, False, keep)
        a = a.detach().numpy()
    v = a
    out.n0 = v.shape[0]; out.n1 = 1; out.n2 = 1
    out.s0 = v.strides[0] // 8; out.s1 = 1; out.s2 = 1
    out.p = &v[0] if v.shape[0] > 0 else NULL
    out.cuda = False; out.device = -1
    keep.append(v)
    return 0


cdef int _arr2(object a, str name, Arr* out, bint last_contig, list keep) except -1:
    """double[::view.generic, ::view.contiguous] (last_contig) or double[::view.generic, ::view.generic]"""
    cdef double[::view.generic, ::view.contiguous] vc
    cdef double[::view.generic, ::view.generic] vg
    if _is_tensor(a):
        if a.is_cuda:
            return _tensor(a, 2, name, out, last_contig, keep)
        a = a.detach().numpy()
    out.n2 = 1; out.s2 = 1
    out.cuda = False; out.device = -1
    if last_contig:
        vc = a
        out.n0 = vc.shape[0]; out.n1 = vc.shape[1]
        out.s0 = vc.strides[0] // 8; out.s1 = 1
        out.p = &vc[0, 0] if (vc.shape[0] > 0 and vc.shape[1] > 0) else NULL
        keep.append(vc)
    else:
        vg = a
        out.n0 = vg.shape[0]; out.n1 = vg.shape[1]
        out.s0 = vg.strides[0] // 8; out.s1 = vg.strides[1] // 8
        out.p = &vg[0, 0] if (vg.shape[0] > 0 and vg.shape[1] > 0) else NULL
        keep.append(vg)
    return 0


cdef int _arr3(object a, str name, Arr* out, list keep) except -1:
    """double[::view.generic, ::view.generic, ::view.contiguous]"""
    cdef double[::view.generic, ::view.generic, ::view.contiguous] v
    if _is_tensor(a):
        if a.is_cuda:
            return _tensor(a, 3, name, out, True, keep)
        a = a.detach().numpy()
    v = a
    out.n0 = v.shape[0]; out.n1 = v.shape[1]; out.n2 = v.shape[2]
    out.s0 = v.strides[0] // 8; out.s1 = v.strides[1] // 8; out.s2 = 1
    out.p = &v[0, 0, 0] if (v.shape[0] > 0 and v.shape[1] > 0 and v.shape[2] > 0) else NULL
    out.cuda = False; out.device = -1
    keep.append(v)
    return 0


cdef object _dense_host_fk(object fk, Arr* a, list keep):
    """the library wants a unit stride on the last axis of HOST arrays; the reference's fk is fully strided"""
    if (not a.cuda) and a.n1 > 1 and a.s1 != 1:
        fk = np.ascontiguousarray(fk)
        _arr2(fk, "fk", a, True, keep)
    return fk


cdef void* _stream_ptr(int device):
    sp = _lib.current_stream_ptr(device)
    return <void*><uintptr_t>(sp if sp is not None else 0)


def number_of_dofs(int dimension, int order):
    """Number of DOFs for given dimension (1,2,3) and order (0..4); -1 / -2 for a bad dimension / order
    (``expert.pyx:57-63`` -> ``infra.pyx:67-112``; no exception, like the reference)."""
    if dimension not in (1, 2, 3):
        return -1
    if order not in (0, 1, 2, 3, 4):
        return -2
    return defs.NUMBER_OF_DOFS[dimension][order]


# ---- the simple API: wlsqm/fitter/simple.pyx:60-604 ----------------------------------------------------------------------
cdef int _fit_many(int dim, object xk, object fk, int[::view.generic] nk, object xi, object fi, object sens, int do_sens,
                   int[::view.generic] order, long long[::view.generic] knowns, int[::view.generic] weighting_method,
                   int algorithm, int max_iter, object device) except -1:
    cdef Arr axk, afk, axi, afi, asn
    cdef list keep = []
    cdef int[::1] nk_c = np.ascontiguousarray(nk)
    cdef int[::1] od_c = np.ascontiguousarray(order)
    cdef long long[::1] kn_c = np.ascontiguousarray(knowns)
    cdef int[::1] wm_c = np.ascontiguousarray(weighting_method)
    cdef Py_ssize_t ncases = nk_c.shape[0]
    cdef int32_t maxnk = 0, lo = 0, hi = 0, uni = 0
    cdef int maxno, dev, rc
    cdef int32_t it = 0
    cdef double* sens_p = NULL
    cdef int64_t sn0 = 0, sn1 = 0
    if od_c.shape[0] != ncases or kn_c.shape[0] != ncases or wm_c.shape[0] != ncases:
        raise ValueError("nk, order, knowns and weighting_method must have the same length")
    if ncases < 1:         # CaseManager_new (infra.pyx:308-360) refuses an empty batch
        raise ValueError("Must specify max_cases > 0 when creating a CaseManager.")
    if dim >= 2:
        _arr3(xk, "xk", &axk, keep)
        _arr2(xi, "xi", &axi, True, keep)
        if axi.n1 < dim or axk.n2 < dim:
            raise ValueError("xi and xk must have %d coordinates on their last axis" % dim)
        if (not axk.cuda) and axk.n1 > 1 and (axk.s1 != dim or axk.n2 != dim):
            # dense neighbour rows of exactly `dim` coordinates from host memory (the reference reads the first dim columns)
            xk = np.ascontiguousarray(np.asarray(xk)[:, :, :dim])
            _arr3(xk, "xk", &axk, keep)
    else:
        _arr2(xk, "xk", &axk, False, keep)
        _arr1(xi, "xi", &axi, keep)
        if (not axk.cuda) and axk.n1 > 1 and axk.s1 != 1:
            xk = np.ascontiguousarray(xk)
            _arr2(xk, "xk", &axk, False, keep)
    _arr2(fk, "fk", &afk, False, keep)
    fk = _dense_host_fk(fk, &afk, keep)
    _arr2(fi, "fi", &afi, True, keep)
    _check(wlsqm_meta_summary(ncases, <const int32_t*>&nk_c[0], <const int32_t*>&od_c[0], <const int64_t*>&kn_c[0],
                              <const int32_t*>&wm_c[0], &maxnk, &lo, &hi, &uni))
    if lo < 0 or hi > 4:
        raise ValueError("order must be 0, 1, 2, 3 or 4")
    maxno = defs.NUMBER_OF_DOFS[dim][hi]
    if axk.n0 < ncases or afk.n0 < ncases or axi.n0 < ncases or afi.n0 < ncases:
        raise ValueError("xk, fk, xi and fi must have at least ncases = %d rows" % ncases)
    if axk.n1 < maxnk or afk.n1 < maxnk or afi.n1 < maxno:
        raise ValueError("xk/fk need >= max(nk) = %d columns and fi >= %d columns" % (maxnk, maxno))
    if do_sens:
        if sens is None:
            raise ValueError("sens must be given when do_sens is set")
        _arr3(sens, "sens", &asn, keep)
        if asn.n0 < ncases or asn.n1 < maxnk or asn.n2 < maxno:
            raise ValueError("sens must have shape (>= ncases, >= max nk, >= max no)")
        sens_p = asn.p; sn0 = asn.s0; sn1 = asn.s1
    if device is None:
        dev = axk.device if axk.cuda else (afk.device if afk.cuda else (afi.device if afi.cuda else _lib.default_device()))
    else:
        dev = device
    wlsqm_set_caller_stream(_stream_ptr(dev))
    with nogil:
        rc = wlsqm_fit_many(dim, ncases, axk.p, axk.s0, axk.s1, afk.p, afk.s0, afk.s1, <const int32_t*>&nk_c[0], axi.p, axi.s0,
                            afi.p, afi.s0, sens_p, sn0, sn1, do_sens, <const int32_t*>&od_c[0], <const int64_t*>&kn_c[0],
                            <const int32_t*>&wm_c[0], algorithm, max_iter, dev, &it)
    _check(rc)
    return it


cdef object _expand_single(object a):
    """view of a single-case array as a batch of one (no copy, so in-place updates reach the caller)"""
    if _is_tensor(a):
        return a.unsqueeze(0)
    return np.asarray(a)[np.newaxis, ...]


cdef int _fit_one(int dim, object xk, object fk, object xi, object fi, object sens, int do_sens, int order, long long knowns,
                  int weighting_method, int algorithm, int max_iter, object device) except -1:
    cdef Arr t, tk
    cdef list keep = []
    if dim >= 2:
        _arr2(xk, "xk", &tk, True, keep)
        _arr1(xi, "xi", &t, keep)
        xi_b = _expand_single(xi)
    else:
        _arr1(xk, "xk", &tk, keep)
        xi_b = np.array([float(xi)], dtype=np.float64)
    nk = np.array([tk.n0], dtype=np.int32)
    _arr1(fk, "fk", &t, keep)
    _arr1(fi, "fi", &t, keep)
    sens_b = None
    if do_sens:
        if sens is None:
            raise ValueError("sens must be given when do_sens is set")
        _arr2(sens, "sens", &t, True, keep)
        sens_b = _expand_single(sens)
    return _fit_many(dim, _expand_single(xk), _expand_single(fk), nk, xi_b, _expand_single(fi), sens_b, do_sens,
                     np.array([order], dtype=np.int32), np.array([knowns], dtype=np.int64),
                     np.array([weighting_method], dtype=np.int32), algorithm, max_iter, device)


def _make(int dim):
    cdef long long bF = 1  # b{1,2,3}_F
    cdef int ALGO_BASIC = defs.ALGO_BASIC, ALGO_ITERATIVE = defs.ALGO_ITERATIVE, WC = defs.WEIGHT_CENTER

    def fit(xk, fk, xi, fi, sens, int do_sens=0, int order=2, long long knowns=bF, int weighting_method=WC, int debug=0,
            device=None):
        return _fit_one(dim, xk, fk, xi, fi, sens, do_sens, order, knowns, weighting_method, ALGO_BASIC, 0, device)

    def fit_iterative(xk, fk, xi, fi, sens, int do_sens=0, int order=2, long long knowns=bF, int weighting_method=WC,
                      int max_iter=10, int debug=0, device=None):
        return _fit_one(dim, xk, fk, xi, fi, sens, do_sens, order, knowns, weighting_method, ALGO_ITERATIVE, max_iter, device)

    def fit_many(xk, fk, int[::view.generic] nk, xi, fi, sens, int do_sens, int[::view.generic] order,
                 long long[::view.generic] knowns, int[::view.generic] weighting_method, int debug=0, device=None):
        return _fit_many(dim, xk, fk, nk, xi, fi, sens, do_sens, order, knowns, weighting_method, ALGO_BASIC, 0, device)

    def fit_iterative_many(xk, fk, int[::view.generic] nk, xi, fi, sens, int do_sens, int[::view.generic] order,
                           long long[::view.generic] knowns, int[::view.generic] weighting_method, int max_iter=10,
                           int debug=0, device=None):
        return _fit_many(dim, xk, fk, nk, xi, fi, sens, do_sens, order, knowns, weighting_method, ALGO_ITERATIVE, max_iter,
                         device)

    def fit_many_parallel(xk, fk, int[::view.generic] nk, xi, fi, sens, int do_sens, int[::view.generic] order,
                          long long[::view.generic] knowns, int[::view.generic] weighting_method, int ntasks=8, int debug=0,
                          device=None):
        return _fit_many(dim, xk, fk, nk, xi, fi, sens, do_sens, order, knowns, weighting_method, ALGO_BASIC, 0, device)

    def fit_iterative_many_parallel(xk, fk, int[::view.generic] nk, xi, fi, sens, int do_sens, int[::view.generic] order,
                                    long long[::view.generic] knowns, int[::view.generic] weighting_method, int max_iter=10,
                                    int ntasks=8, int debug=0, device=None):
        return _fit_many(dim, xk, fk, nk, xi, fi, sens, do_sens, order, knowns, weighting_method, ALGO_ITERATIVE, max_iter,
                         device)

    lines = {1: ("simple.pyx:429-478", "481-498", "501-537", "540-559", "562-581", "584-604"),
             2: ("simple.pyx:241-290", "293-310", "318-354", "357-376", "379-398", "401-421"),
             3: ("simple.pyx:60-109", "111-128", "131-167", "170-189", "192-211", "214-234")}[dim]
    out = {}
    for f, suffix, ln, what in (
            (fit, "", lines[0], "Fit one local model"),
            (fit_iterative, "_iterative", lines[1], "Fit one local model, with iterative refinement"),
            (fit_many, "_many", lines[2], "Fit many local models"),
            (fit_iterative_many, "_iterative_many", lines[3], "Fit many local models, with iterative refinement"),
            (fit_many_parallel, "_many_parallel", lines[4], "Fit many local models (one GPU launch; ntasks ignored)"),
            (fit_iterative_many_parallel, "_iterative_many_parallel", lines[5],
             "Fit many local models with iterative refinement (one GPU launch; ntasks ignored)")):
        name = "fit_%dD%s" % (dim, suffix)
        try:
            f.__name__ = f.__qualname__ = name
            f.__doc__ = ("%s to %dD scalar data (reference: wlsqm/fitter/%s).\n\n"
                         "fi is updated in place (knowns untouched, unknowns overwritten); sens[k, j] = d fi[j] / d fk[k],\n"
                         "NaN for known j.  Returns the number of refinement iterations taken (0 without _iterative)."
                         % (what, dim, ln))
        except (AttributeError, TypeError):
            pass
        out[name] = f
    return out


for _d in (1, 2, 3):
    globals().update(_make(_d))


# ---- ExpertSolver: wlsqm/fitter/expert.pyx:66-781 -------------------------------------------------------------------------
cdef inline wlsqm_solver_t* _h(object self):
    return <wlsqm_solver_t*><uintptr_t>self._hptr


class ExpertSolver:
    """Advanced API / "expert mode" with separate prepare and solve stages (``expert.pyx:66-88``).

    s = ExpertSolver(...); s.prepare(xi, xk); s.solve(fk, fi[, sens]) -- repeat solve() with new data.
    State lives in device memory (no 2 GiB arena limit); ``ntasks`` is accepted and validated but has no meaning; every
    array argument may also be a CUDA ``torch.Tensor``; ``device=`` selects the GPU and ``interpolate(..., diff='all')``
    returns every derivative slot in one pass (extensions)."""

    def __init__(self, int dimension, int[::view.generic] nk, int[::view.generic] order, long long[::view.generic] knowns,
                 int[::view.generic] weighting_method, int algorithm=defs.ALGO_BASIC, int do_sens=False, int max_iter=10,
                 int ntasks=1, int debug=False, host=None, device=None):
        cdef int[::1] nk_c = np.ascontiguousarray(nk)
        cdef int[::1] od_c = np.ascontiguousarray(order)
        cdef long long[::1] kn_c = np.ascontiguousarray(knowns)
        cdef int[::1] wm_c = np.ascontiguousarray(weighting_method)
        cdef Py_ssize_t ncases = nk_c.shape[0]
        cdef int32_t maxnk = 0, lo = 0, hi = 0, uni = 0
        cdef wlsqm_solver_t* h = NULL
        cdef int dev, rc
        self._hptr = 0
        self._handle = None
        # sanity checks, in the reference's order (expert.pyx:130-159)
        if od_c.shape[0] != ncases or kn_c.shape[0] != ncases or wm_c.shape[0] != ncases:
            raise ValueError("nk, order, knowns and weighting method must have the same length; currently, "
                             "len(nk)=%d, len(order)=%d, len(knowns)=%d, len(weighting_method)=%d"
                             % (nk_c.shape[0], od_c.shape[0], kn_c.shape[0], wm_c.shape[0]))
        if dimension not in (1, 2, 3):
            raise ValueError("Dimension must be 1, 2 or 3, got %d" % dimension)
        if algorithm not in (defs.ALGO_BASIC, defs.ALGO_ITERATIVE):
            raise ValueError("Unknown algorithm specifier %d; see wlsqm.fitter.defs for valid specifiers ALGO_*" % algorithm)
        if ntasks < 1:
            raise ValueError("ntasks must be >= 1, got %d" % ntasks)
        if ncases < 1:     # CaseManager_new (infra.pyx:308-360) refuses an empty batch
            raise ValueError("Must specify max_cases > 0 when creating a CaseManager.")
        nk_a, order_a, knowns_a, wm_a = np.asarray(nk_c), np.asarray(od_c), np.asarray(kn_c), np.asarray(wm_c)
        # guest mode sanity checks (expert.pyx:163-189)
        if host is not None:
            if not host.ready:
                raise RuntimeError("In guest mode, host must be in the ready state (host.prepare() must have been "
                                   "called before creating another ExpertSolver instance in guest mode).")
            if host.ncases != ncases:
                raise RuntimeError("In guest mode, number of cases (number of elements in nk) must match; got %d, "
                                   "host has %d" % (ncases, host.ncases))
            if host.dimension != dimension:
                raise ValueError("In guest mode, dimension must match; got %d, host has %d" % (dimension, host.dimension))
            if bool(host.debug) != bool(debug):
                raise ValueError("In guest mode, debug flag must match; got %s, host has %s" % (bool(debug), bool(host.debug)))
            if (np.asanyarray(host.nk) != nk_a).any():
                raise ValueError("In guest mode, 'nk' must match element-by-element.")
            if (np.asanyarray(host.order) != order_a).any():
                raise ValueError("In guest mode, 'order' must match element-by-element.")
            if (np.asanyarray(host.knowns) != knowns_a).any():
                raise ValueError("In guest mode, 'knowns' must match element-by-element.")
            if (np.asanyarray(host.weighting_method) != wm_a).any():
                raise ValueError("In guest mode, 'weighting_method' must match element-by-element.")
        self.host = host
        self.ready = False
        self.dimension = dimension
        self.algorithm = algorithm
        self.max_iter = max_iter
        self.ncases = ncases
        self.do_sens = do_sens
        self.ntasks = ntasks
        self.debug = debug
        self.xk = None
        self.xi = None
        self.tree = None
        self.nk = nk_a
        self.order = order_a
        self.knowns = knowns_a
        self.weighting_method = wm_a
        if device is None:
            device = host.device if host is not None else _lib.default_device()
        dev = device
        self.device = dev
        # metadata is validated ONCE here; solve() / prepare() only compare shapes against the cached sizes
        _check(wlsqm_meta_summary(ncases, <const int32_t*>&nk_c[0], <const int32_t*>&od_c[0], <const int64_t*>&kn_c[0],
                                  <const int32_t*>&wm_c[0], &maxnk, &lo, &hi, &uni))
        if lo < 0 or hi > 4:
            raise ValueError("order must be 0, 1, 2, 3 or 4")
        self._maxnk = maxnk
        self._maxno = defs.NUMBER_OF_DOFS[dimension][hi]
        self._stream = -1
        self._hood_points = 0
        # guest mode: borrow the host's operators (one set of operators for several fields on one geometry);
        # an iterative guest of a non-iterative host needs the geometry itself and prepares on its own
        self._borrows = (host is not None and getattr(host, "_hptr", 0) != 0
                         and (algorithm != defs.ALGO_ITERATIVE or host.algorithm == defs.ALGO_ITERATIVE))
        if self._borrows:
            _check(wlsqm_solver_create_guest(_h(host), algorithm, do_sens, max_iter, &h))
        else:
            with nogil:
                rc = wlsqm_solver_create(dimension, ncases, <const int32_t*>&nk_c[0], <const int32_t*>&od_c[0],
                                         <const int64_t*>&kn_c[0], <const int32_t*>&wm_c[0], algorithm, do_sens, max_iter,
                                         debug, dev, &h)
            _check(rc)
        self._hptr = <uintptr_t>h
        self._handle = _C.c_void_p(<uintptr_t>h)      # (wlsqm_b200.parallel and the ctypes helpers take the handle this way)
        self.manager_pw = self._handle                # the reference keeps its CaseManager pointer under this name (expert.pyx:257-260)
        if host is not None:
            self.tree = host.tree

    # -- lifetime -----------------------------------------------------------------------------------
    def close(self):
        """Free the device state now (guests of this solver must be closed first)."""
        cdef uintptr_t h = getattr(self, "_hptr", 0)
        self._hptr = 0
        self._handle = None
        if h:
            wlsqm_solver_destroy(<wlsqm_solver_t*>h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _use_stream(self):
        sp = _lib.current_stream_ptr(self.device)
        if sp is not None and sp != self._stream:
            _check(wlsqm_solver_set_stream(_h(self), <void*><uintptr_t>sp))
            self._stream = sp

    def keep_solution(self, keep=True):
        """Extension: keep=False drops the solver's own copy of the solution (the reference's Case_set_fi, infra.pyx:780-786)
        for solve() calls with a CUDA-tensor fi: 8*no bytes per case less traffic; interpolate() then raises until a
        solve() with the copy enabled."""
        _check(wlsqm_solver_keep_solution(_h(self), 1 if keep else 0))

    def synchronize(self):
        """Wait for everything enqueued by this solver (only needed with CUDA-tensor arguments)."""
        cdef int rc
        cdef wlsqm_solver_t* h = _h(self)
        with nogil:
            rc = wlsqm_solver_synchronize(h)
        _check(rc)

    def memory_used(self):
        """(bytes of solver state on the device, state + staging buffers) -- ``expert.pyx:289-306``."""
        cdef int64_t used = 0, total = 0
        _check(wlsqm_solver_memory(_h(self), &used, &total))
        return (used, total)

    # -- prepare --------------------------------------------------------------------------------------
    def prepare(self, xi, xk):
        """Generate, scale and factor the problem matrices and store the solution operators
        (``expert.pyx:309-426``).  xi: (ncases, dim) [1D: (ncases,)], xk: (ncases, >=max nk, dim)
        [1D: (ncases, >=max nk)], float64."""
        cdef Arr axi, axk
        cdef list keep = []
        cdef int dim = self.dimension, rc
        cdef Py_ssize_t ncases = self.ncases, maxnk = self._maxnk
        cdef wlsqm_solver_t* h = _h(self)
        self.ready = False
        if self.host is not None:
            # guest mode: geometry (and operators) are the host's (expert.pyx:348-385)
            self.xk, self.xi = self.host.xk, self.host.xi
            xi, xk = self.xi, self.xk
            if self._borrows:
                _check(wlsqm_solver_prepare_guest(h))
                self.ready = True
                return
        if dim >= 2:
            _arr2(xi, "xi", &axi, True, keep)
            _arr3(xk, "xk", &axk, keep)
            if axi.n1 < dim or axk.n2 < dim:
                raise ValueError("xi and xk must have %d coordinates on their last axis" % dim)
            if (not axk.cuda) and maxnk > 1 and (axk.s1 != dim or axk.n2 != dim):
                # host rows must be dense with exactly `dim` coordinates; the reference's double[:,:,::contiguous] view also
                # accepts pitched rows / a longer last axis and reads only the first dim columns
                xk_d = np.ascontiguousarray(np.asarray(xk)[:, :, :dim])
                _arr3(xk_d, "xk", &axk, keep)
        else:
            _arr1(xi, "xi", &axi, keep)
            _arr2(xk, "xk", &axk, False, keep)
            if (not axk.cuda) and maxnk > 1 and axk.s1 != 1:
                xk_d = np.ascontiguousarray(xk)
                _arr2(xk_d, "xk", &axk, False, keep)
        if axi.n0 < ncases or axk.n0 < ncases:
            raise ValueError("xi and xk must have at least ncases = %d rows" % ncases)
        if axk.n1 < maxnk:
            raise ValueError("xk must hold at least max(nk) = %d neighbours per case" % maxnk)
        self._use_stream()
        if self.host is None:
            self.xk, self.xi, self.tree = xk, xi, None
        with nogil:
            rc = wlsqm_solver_prepare(h, axi.p, axi.s0, axk.p, axk.s0, axk.s1)
        _check(rc)
        self._cuda_out = bool(axk.cuda)
        self.ready = True

    def conds(self):
        """2-norm condition number of the scaled problem matrix of every case (needs debug=True;
        ``expert.pyx:429-464``)."""
        cdef double[::1] out
        if not self.ready:
            raise RuntimeError("Solver is not in the ready state; prepare() must be called before conds()")
        if not self.debug:
            raise RuntimeError("Not in debug mode; condition number data has not been computed")
        out = np.empty((self.ncases,), dtype=np.float64)
        _check(wlsqm_solver_conds(_h(self), &out[0]))
        return np.asarray(out)

    # -- neighbourhoods as index lists (extension) ----------------------------------------------------
    def prepare_hoods(self, x, hoods, xi=None):
        """``prepare(xi, x[hoods])`` with the gather done on the device (extension).

        x: (npoints, dim) [1D: (npoints,)] float64; hoods: (ncases, >= max nk) int32 indices into x (numpy or
        CUDA tensor, e.g. from ``PointGrid.knn``); xi: the origins, default ``x[:ncases]``."""
        self.ready = False
        from . import neighbors
        xa, npts, dim, x_s0 = neighbors._points(x)
        if dim != self.dimension:
            raise ValueError("x has %d coordinates, the solver has dimension %d" % (dim, self.dimension))
        ha = _lib.as_arr(hoods, np.int32, 2, "hoods")
        if ha.shape[0] < self.ncases or (self.ncases and ha.shape[1] < self._maxnk):
            raise ValueError("hoods must have shape (>= ncases, >= max nk)")
        cdef uintptr_t xi_p = 0
        cdef int64_t xi_s0 = 0
        if xi is not None:
            xia, nxi, dimi, xs0 = neighbors._points(xi, "xi")
            if dimi != dim or nxi < self.ncases:
                raise ValueError("xi must hold one origin per case")
            xi_p = xia.ptr
            xi_s0 = xs0
        elif npts < self.ncases:
            raise ValueError("without xi, x must hold one point per case")
        self._use_stream()
        cdef uintptr_t xp = xa.ptr, hp = ha.ptr
        cdef int64_t xs = x_s0, np_ = npts, hs = ha.strides[0]
        cdef int rc
        cdef wlsqm_solver_t* h = _h(self)
        with nogil:
            rc = wlsqm_solver_prepare_hoods(h, <const double*>xp, xs, np_, <const int32_t*>hp, hs, <const double*>xi_p, xi_s0)
        _check(rc)
        self.xi = xi if xi is not None else x[:self.ncases]
        self.xk, self.tree = None, None
        self._hood_points = npts
        self._cuda_out = bool(ha.is_cuda)
        self.ready = True

    # -- export of the prepared operators (extension; wlsqm_b200/fitter/opexport.py) ------------------------------------
    def stencils(self, coeffs):
        """(W, K): the prepared operators contracted with coefficient rows -- W (nops, ncases, max nk) weights on fk,
        K (nops, ncases, max no) weights on the known values, so that sum_s c[s] fi[i, s] = W[i] . fk[i] + K[i] . fi[i]
        for an ALGO_BASIC solve.  coeffs: an int slot, a (max no,) row or a (nops, max no) array (the nops axis is dropped
        for the first two).  The d fi / d fk of the reference's sens (impl.pyx:769-779); an ALGO_ITERATIVE solver exports
        the same operator (the refinement corrections are not part of it)."""
        return _opexport.stencils(self, coeffs)

    def operator(self, coeffs, center=None):
        """(D, K): the global sparse operator (ncases, npoints) over the points of prepare_hoods (torch CSR on the
        device for CUDA hoods, scipy csr_array otherwise; a list for 2-D coeffs) and the known-value weights.
        center: index in x of case 0's own point -- the weight on a known F of case i then goes to column center + i.
        See wlsqm_b200.fitter.opexport.operator."""
        return _opexport.operator(self, coeffs, center)

    def solve_hoods(self, f, fi, sens=None):
        """``solve(f[hoods], fi, sens)`` with the gather done on the device (extension; needs prepare_hoods).
        f: (npoints,) float64 -- one value per point instead of one per (point, neighbour)."""
        cdef Arr af, afi, asn
        cdef list keep = []
        cdef double* sens_p = NULL
        cdef int64_t sn0 = 0, sn1 = 0
        cdef int32_t it = 0
        cdef int rc
        cdef wlsqm_solver_t* h = _h(self)
        if not self.ready:
            raise RuntimeError("Solver is not in the ready state; prepare() must be called before solve()")
        _arr1(f, "f", &af, keep)
        if af.n0 < self._hood_points:
            raise ValueError("f must hold one value per point of the x given to prepare_hoods()")
        _arr2(fi, "fi", &afi, True, keep)
        if afi.n0 < self.ncases or afi.n1 < self._maxno:
            raise ValueError("fi must have shape (>= ncases, >= %d)" % self._maxno)
        if self.do_sens:
            if sens is None:
                raise ValueError("sens must be given when do_sens is set")
            _arr3(sens, "sens", &asn, keep)
            sens_p = asn.p; sn0 = asn.s0; sn1 = asn.s1
        self._use_stream()
        with nogil:
            rc = wlsqm_solver_solve_hoods(h, af.p, af.s0 if af.n0 > 1 else 1, afi.p, afi.s0, sens_p, sn0, sn1, &it)
        _check(rc)
        return it

    # -- solve ------------------------------------------------------------------------------------------
    def solve(self, fk, fi, sens=None):
        """Fit the model to the data fk using the prepared geometry (``expert.pyx:467-655``).

        fk (ncases, >=max nk); fi (ncases, >=max no) in/out: knowns are read, unknowns written in place;
        sens (ncases, >=max nk, >=max no) out, needed iff do_sens.  Returns the maximum number of
        refinement iterations taken (0 for ALGO_BASIC)."""
        cdef Arr afk, afi, asn
        cdef list keep = []
        cdef double* sens_p = NULL
        cdef int64_t sn0 = 0, sn1 = 0
        cdef int32_t it = 0
        cdef int rc
        cdef Py_ssize_t ncases = self.ncases, maxnk = self._maxnk, maxno = self._maxno
        cdef wlsqm_solver_t* h = _h(self)
        if not self.ready:
            raise RuntimeError("Solver is not in the ready state; prepare() must be called before solve()")
        _arr2(fk, "fk", &afk, False, keep)
        _arr2(fi, "fi", &afi, True, keep)
        if afk.n0 < ncases or afi.n0 < ncases:
            raise ValueError("fk and fi must have at least ncases = %d rows" % ncases)
        if afk.n1 < maxnk or afi.n1 < maxno:
            raise ValueError("fk needs >= %d columns and fi >= %d columns" % (maxnk, maxno))
        fk = _dense_host_fk(fk, &afk, keep)
        if self.do_sens:
            if sens is None:
                raise ValueError("sens must be given when do_sens is set")
            _arr3(sens, "sens", &asn, keep)
            if asn.n0 < ncases or asn.n1 < maxnk or asn.n2 < maxno:
                raise ValueError("sens must have shape (>= ncases, >= max nk, >= max no)")
            sens_p = asn.p; sn0 = asn.s0; sn1 = asn.s1
        self._use_stream()
        with nogil:
            rc = wlsqm_solver_solve(h, afk.p, afk.s0, afk.s1, afi.p, afi.s0, sens_p, sn0, sn1, &it)
        _check(rc)
        return it

    def solve_fields(self, fk, fi):
        """Fit nf fields on the prepared geometry in one pass over the stored operators (extension).

        fk (nf, >= ncases, >= max nk); fi (nf, >= ncases, >= max no) in/out, fields-outer or fields-inner rows (e.g.
        ``fi_all.transpose(1, 0, 2)`` of an (ncases, nf, no) array).  Field j's unknown slots are bit for bit what
        ``solve(fk[j], fi[j])`` writes; returns the maximum of those solves' return values, and iterations() gives the
        per-case maximum.  The solver's own solution copy is not written (interpolate() raises until the next solve());
        sens is not produced.  See wlsqm_b200.fitter.fields."""
        return _fields.solve_fields(self, fk, fi)

    def solve_hoods_fields(self, f, fi):
        """solve_fields with the data per point (extension; needs prepare_hoods): f (nf, >= npoints), any strides --
        ``f_all.T`` of an (npoints, nf) array is fine.  Field j equals ``solve_hoods(f[j], fi[j])`` bit for bit."""
        return _fields.solve_hoods_fields(self, f, fi)

    def iterations(self):
        """Per-case refinement iteration counts of the last solve (extension; zeros for ALGO_BASIC)."""
        cdef int[::1] out = np.zeros((self.ncases,), dtype=np.int32)
        _check(wlsqm_solver_iterations(_h(self), <int32_t*>&out[0]))
        return np.asarray(out)

    # -- interpolate ----------------------------------------------------------------------------------
    def _xi_host(self):
        xi = self.xi
        if _is_tensor(xi):
            xi = xi.detach().cpu().numpy()
        return np.asarray(xi)

    def prep_interpolate(self, search=None):
        """Index the model origins xi for the nearest-model search (``expert.pyx:658-681``).

        search='scipy' (default for host arrays): SciPy's cKDTree on the host, so that the index I is the
        reference's by construction.  search='gpu' (default when xi is a CUDA tensor; extension): a uniform
        grid on the device -- the same nearest model wherever distances are distinct, without the 1.8 us per
        query host step.  mode='continuous' always searches on the device."""
        if not self.ready:
            raise RuntimeError("Solver is not in the ready state; prepare() must be called before prep_interpolate()")
        if search is None:
            search = 'gpu' if _is_tensor(self.xi) and self.xi.is_cuda else 'scipy'
        if search not in ('scipy', 'gpu'):
            raise ValueError("search must be 'scipy' or 'gpu'; got %r" % (search,))
        self._use_stream()
        _lib.announce_stream(self.device)
        _check(wlsqm_solver_index_models(_h(self)))
        if self.host is not None and self.host.tree is not None:
            self.tree = self.host.tree
        elif search == 'gpu':
            self.tree = _DeviceModelIndex(self)
        else:
            import scipy.spatial
            xi = self._xi_host()
            xi_rank2 = xi if self.dimension >= 2 else np.atleast_2d(xi).T
            self.tree = scipy.spatial.cKDTree(data=xi_rank2)

    def _nearest_models(self, x, uintptr_t xp, int64_t x_s0, Py_ssize_t nx, bint x_cuda, I):
        """(I_use, I_out): the model of every query in mode='nearest' -- I itself when given, else the nearest origin
        by self.tree (the device grid for CUDA queries or search='gpu', I then stays where x lives; cKDTree otherwise).
        interpolate() and the interpolation operators (fitter/opexport.py) resolve their models here."""
        cdef uintptr_t ip
        if I is not None:
            return I, I
        if isinstance(self.tree, _DeviceModelIndex) or x_cuda:
            # nearest model by the device-side grid (extension); I stays where x lives
            if x_cuda:
                I_out = _torch.empty((nx,), dtype=_torch.int64, device=x.device)
                ip = I_out.data_ptr()
            else:
                I_out = np.empty((nx,), dtype=np.int_)
                ip = I_out.ctypes.data
            _lib.announce_stream(self.device)
            _check(wlsqm_solver_nearest_models(_h(self), <const double*>xp, x_s0, nx, <int64_t*>ip))
            return I_out, I_out
        xh = np.asarray(x)
        xq = xh if self.dimension >= 2 else np.atleast_2d(xh).T
        _d, I_h = self.tree.query(xq, k=1)
        I_out = np.ascontiguousarray(I_h, dtype=np.int_)
        return I_out, I_out

    # -- interpolation operators (extension; wlsqm_b200/fitter/opexport.py) -------------------------------------------
    def interp_stencils(self, x, coeffs=0, I=None, mode='nearest', r=None):
        """(W, K, I_out): the map from the data to interpolate(x, mode='nearest') as per-query weights -- W (nops, nx,
        max nk) on fk[I[q]], K (nops, nx, max no) on the known values of model I[q], for the coefficient rows coeffs over
        the derivative slots (an int slot, a (max no,) row or a (nops, max no) array).  I=None: the nearest models, found
        as interpolate() finds them.  mode='continuous' (needs r, refuses I): one row per (query, model) pair of the
        models within r, returned as (W, K, (pair_ptr, J)).  See wlsqm_b200.fitter.opexport.interp_stencils."""
        return _opexport.interp_stencils(self, x, coeffs, I, mode, r)

    def interp_operator(self, x, coeffs=0, I=None, center=None, mode='nearest', r=None):
        """(E, K, I_out): the same map as a sparse matrix (nx, npoints) over the points of prepare_hoods, like operator().
        mode='continuous': (E, K, (pair_ptr, J)) with K per pair.  See wlsqm_b200.fitter.opexport.interp_operator."""
        return _opexport.interp_operator(self, x, coeffs, I, center, mode, r)

    def interpolate(self, x, mode='nearest', r=None, diff=0, I=None):
        """Interpolate the global patched model or one derivative of it (``expert.pyx:687-781``).

        Returns (out, I_out).  ``diff='all'`` (extension, mode='nearest') returns out of shape
        (nx, max no): every derivative slot in one pass."""
        cdef Arr ax
        cdef list keep = []
        cdef int dim = self.dimension, cdiff, rc
        cdef Py_ssize_t nx, width
        cdef int64_t x_s0
        cdef uintptr_t ip, op
        cdef long[::1] I_v
        cdef wlsqm_solver_t* h = _h(self)
        if mode not in ['nearest', 'continuous']:
            raise ValueError("mode must be one of 'nearest', 'continuous'; got '%s'" % mode)
        if mode == 'continuous' and r is None:
            raise ValueError("r must be specified in mode='continuous'")
        if diff is None:
            raise ValueError("diff cannot be None")
        if self.tree is None:
            raise RuntimeError("Points xi have not been indexed; prep_interpolate() must be called before interpolate()")
        if I is not None and len(I) != len(x):
            raise ValueError("When 'I' is specified, 'I' must have the same length as x; got len(I) = %d, len(x) = %d."
                             % (len(I), len(x)))
        all_diffs = isinstance(diff, str) and diff == 'all'
        cdiff = DIFF_ALL if all_diffs else diff
        if dim >= 2:
            _arr2(x, "x", &ax, True, keep)
        else:
            _arr1(x, "x", &ax, keep)
            if (not ax.cuda) and ax.n0 > 1 and ax.s0 != 1:
                x_c = np.ascontiguousarray(x)
                _arr1(x_c, "x", &ax, keep)
        nx = ax.n0
        x_s0 = ax.s0
        self._use_stream()
        if mode == 'continuous':
            return self._interpolate_continuous(x, <uintptr_t>ax.p, x_s0, nx, ax.cuda, float(r), cdiff), np.asanyarray(None)

        I_use, I_out = self._nearest_models(x, <uintptr_t>ax.p, x_s0, nx, ax.cuda, I)
        i_cuda = _is_tensor(I_use) and I_use.is_cuda
        if i_cuda:
            if I_use.dtype != _torch.int64 or I_use.dim() != 1 or (nx > 1 and I_use.stride(0) != 1):
                raise ValueError("I: a contiguous int64 tensor of shape (nx,) is required")
            ip = I_use.data_ptr()
        else:
            I_v = I_use.detach().numpy() if _is_tensor(I_use) else I_use       # long[::1], like the reference (expert.pyx:830)
            ip = <uintptr_t>&I_v[0] if nx > 0 else 0
        width = self._maxno if all_diffs else 1
        oshape = [nx, width] if all_diffs else [nx]
        if ax.cuda:
            out = _torch.empty(oshape, dtype=_torch.float64, device=x.device)
            op = out.data_ptr()
        else:
            out = np.empty(oshape, dtype=np.float64)
            op = out.ctypes.data
        # a query that found no neighbour (NaN coordinates) poisons the whole output (expert.pyx:862-870)
        if (not i_cuda) and nx and (np.asarray(I_v) == self.ncases).any():
            out[...] = np.nan
            return out, np.asanyarray(I_out)
        with nogil:
            rc = wlsqm_solver_interpolate(h, ax.p, x_s0, <const int64_t*>ip, nx, cdiff, <double*>op, width)
        _check(rc)
        return out, (I_out if ax.cuda and _is_tensor(I_out) else np.asanyarray(I_out))

    def interpolate_fields(self, x, fi, mode='nearest', r=None, diff=0, I=None):
        """interpolate() for nf caller-held solutions at once (extension): fi (nf, >= ncases, >= max no), e.g. the fi of
        solve_fields (fi[None] for one field).  Returns (out, I_out) with out (nf, nx), or (nf, nx, max no) for
        diff='all'; out[j] is bit for bit what interpolate() returns on a solver whose last solve() produced fi[j].  The
        solver's own solution copy is not used, so this works after solve_fields and keep_solution(False).  See
        wlsqm_b200.fitter.fields.interpolate_fields."""
        return _fields.interpolate_fields(self, x, fi, mode, r, diff, I)

    def _interpolate_continuous(self, x, uintptr_t xp, int64_t x_s0, Py_ssize_t nx, bint cuda, double r, int cdiff):
        """mode='continuous' (``expert_interpolate_continuous``, ``expert.pyx:898-985``): weighted average
        over every local model whose origin lies within r; weights (1 - sqrt(d2/r2))^2.  One kernel: each query
        walks the cells of the model-origin grid that meet its ball and evaluates the models on the fly."""
        cdef uintptr_t op
        cdef int rc
        cdef wlsqm_solver_t* h = _h(self)
        if cdiff < 0:
            raise ValueError("diff='all' is not available in mode='continuous'")
        if cuda:
            out = _torch.empty((nx,), dtype=_torch.float64, device=x.device)
            op = out.data_ptr()
        else:
            out = np.empty((nx,), dtype=np.float64)
            op = out.ctypes.data
        with nogil:
            rc = wlsqm_solver_interpolate_continuous(h, <const double*>xp, x_s0, nx, r, cdiff, <double*>op)
        _check(rc)
        return out


class _DeviceModelIndex:
    """Stands where the reference keeps its cKDTree (``ExpertSolver.tree``) when the nearest-model search runs
    on the device; ``query(x, k=1)`` answers like ``cKDTree.query``."""

    def __init__(self, solver):
        import weakref
        self._solver = weakref.ref(solver)

    def query(self, x, k=1):
        s = self._solver()
        if k != 1:
            raise ValueError("the model index answers k=1 queries")
        from . import neighbors
        xa, nx, dim, x_s0 = neighbors._points(x)
        _lib.announce_stream(s.device)
        if xa.is_cuda:
            It = _torch.empty((nx,), dtype=_torch.int64, device=x.device)
            _lib.check(_lib.lib().wlsqm_solver_nearest_models(s._handle, xa.ptr, x_s0, nx, int(It.data_ptr())))
            return None, It
        I = np.empty((nx,), dtype=np.int_)
        _lib.check(_lib.lib().wlsqm_solver_nearest_models(s._handle, xa.ptr, x_s0, nx, I.ctypes.data))
        return None, I
