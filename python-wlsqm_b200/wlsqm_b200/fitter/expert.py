"""``ExpertSolver``: prepare once, solve many times -- the reference's advanced API on one B200.

Host-side mirror of ``wlsqm/fitter/expert.pyx`` (class ``ExpertSolver``, :66-781, and
``number_of_dofs``, :57-63): same constructor arguments, attributes, exceptions, in-place semantics
and return values, over the C ABI of ``include/wlsqm_b200.h``.  What differs by design:

* state lives in device memory (the reference's CaseManager arena, ``infra.pyx:308-471``, is gone and
  with it the 2 GiB ``int`` size limit); ``ntasks`` is accepted and validated but has no meaning;
* ``prepare`` stores one dense solution operator per case instead of (c, w, LU, ipiv, scales), so
  ``solve`` is a single streaming pass over HBM;
* every array argument may also be a CUDA ``torch.Tensor`` (zero copy, asynchronous on torch's
  current stream); numpy arrays are staged through the device and are complete on return;
* ``device=`` selects the GPU (extension); ``interpolate(..., diff='all')`` returns every derivative
  slot in one pass (extension).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import defs, fields, opexport
from .. import _lib

__all__ = ["number_of_dofs", "ExpertSolver"]

BINDING = "ctypes"


def number_of_dofs(dimension, order):
    """Number of DOFs for given dimension (1,2,3) and order (0..4); -1 / -2 for a bad dimension / order
    (``expert.pyx:57-63`` -> ``infra.pyx:67-112``; no exception, like the reference)."""
    dimension, order = int(dimension), int(order)
    if dimension not in (1, 2, 3):
        return -1
    if order not in (0, 1, 2, 3, 4):
        return -2
    return defs.NUMBER_OF_DOFS[dimension][order]


def _as_c_int(v, name):
    """typed `int` arguments of the reference (expert.pyx:92-93): Cython refuses None with TypeError"""
    if v is None:
        raise TypeError(f"{name}: an integer is required")
    return int(v)


class ExpertSolver:
    """Advanced API / "expert mode" with separate prepare and solve stages (``expert.pyx:66-88``).

    s = ExpertSolver(...); s.prepare(xi, xk); s.solve(fk, fi[, sens]) -- repeat solve() with new data.
    """

    def __init__(self, dimension, nk, order, knowns, weighting_method, algorithm=defs.ALGO_BASIC,
                 do_sens=False, max_iter=10, ntasks=1, debug=False, host=None, device=None):
        dimension = int(dimension)
        nk_a = _lib.meta_array(nk, np.int32, "nk")
        order_a = _lib.meta_array(order, np.int32, "order")
        knowns_a = _lib.meta_array(knowns, np.int64, "knowns")
        wm_a = _lib.meta_array(weighting_method, np.int32, "weighting_method")
        ncases = nk_a.shape[0]
        # sanity checks, in the reference's order (expert.pyx:130-159)
        if order_a.shape[0] != ncases or knowns_a.shape[0] != ncases or wm_a.shape[0] != ncases:
            raise ValueError("nk, order, knowns and weighting method must have the same length; currently, "
                             "len(nk)=%d, len(order)=%d, len(knowns)=%d, len(weighting_method)=%d"
                             % (nk_a.shape[0], order_a.shape[0], knowns_a.shape[0], wm_a.shape[0]))
        if dimension not in (1, 2, 3):
            raise ValueError("Dimension must be 1, 2 or 3, got %d" % dimension)
        algorithm = _as_c_int(algorithm, "algorithm")
        do_sens = _as_c_int(do_sens, "do_sens")
        max_iter = _as_c_int(max_iter, "max_iter")
        ntasks = _as_c_int(ntasks, "ntasks")
        debug = _as_c_int(debug, "debug")
        if algorithm not in (defs.ALGO_BASIC, defs.ALGO_ITERATIVE):
            raise ValueError("Unknown algorithm specifier %d; see wlsqm.fitter.defs for valid specifiers ALGO_*"
                             % algorithm)
        if ntasks < 1:
            raise ValueError("ntasks must be >= 1, got %d" % ntasks)
        if ncases < 1:     # CaseManager_new (infra.pyx:308-360) refuses an empty batch
            raise ValueError("Must specify max_cases > 0 when creating a CaseManager.")

        # guest mode sanity checks (expert.pyx:163-189)
        if host is not None:
            if not host.ready:
                raise RuntimeError("In guest mode, host must be in the ready state (host.prepare() must have been "
                                   "called before creating another ExpertSolver instance in guest mode).")
            if host.ncases != ncases:
                raise RuntimeError("In guest mode, number of cases (number of elements in nk) must match; got %d, "
                                   "host has %d" % (ncases, host.ncases))
            if host.dimension != dimension:
                raise ValueError("In guest mode, dimension must match; got %d, host has %d"
                                 % (dimension, host.dimension))
            if bool(host.debug) != bool(debug):
                raise ValueError("In guest mode, debug flag must match; got %s, host has %s"
                                 % (bool(debug), bool(host.debug)))
            if (np.asanyarray(host.nk) != nk_a).any():
                raise ValueError("In guest mode, 'nk' must match element-by-element.")
            if (np.asanyarray(host.order) != order_a).any():
                raise ValueError("In guest mode, 'order' must match element-by-element.")
            if (np.asanyarray(host.knowns) != knowns_a).any():
                raise ValueError("In guest mode, 'knowns' must match element-by-element.")
            if (np.asanyarray(host.weighting_method) != wm_a).any():
                raise ValueError("In guest mode, 'weighting_method' must match element-by-element.")

        self._handle = None
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
        self.device = int(device)
        self._maxnk, min_order, max_order, _ = _lib.meta_summary(nk_a, order_a, knowns_a, wm_a)
        if ncases and (min_order < 0 or max_order > 4):
            raise ValueError("order must be 0, 1, 2, 3 or 4")
        self._maxno = number_of_dofs(dimension, max_order) if ncases else 1

        h = C.c_void_p()
        # guest mode: borrow the host's operators (one set of operators for several fields on one geometry);
        # an iterative guest of a non-iterative host needs the geometry itself and prepares on its own
        self._borrows = (host is not None and getattr(host, "_handle", None) is not None
                         and (algorithm != defs.ALGO_ITERATIVE or host.algorithm == defs.ALGO_ITERATIVE))
        if self._borrows:
            _lib.check(_lib.lib().wlsqm_solver_create_guest(host._handle, algorithm, do_sens, max_iter, C.byref(h)))
        else:
            _lib.check(_lib.lib().wlsqm_solver_create(
                dimension, ncases, nk_a.ctypes.data, order_a.ctypes.data, knowns_a.ctypes.data, wm_a.ctypes.data,
                algorithm, do_sens, max_iter, debug, self.device, C.byref(h)))
        self._handle = h
        self.manager_pw = h   # the reference keeps its CaseManager pointer under this name (expert.pyx:257-260)
        if host is not None:
            self.tree = host.tree

    # -- lifetime -----------------------------------------------------------------------------------
    def close(self):
        """Free the device state now (guests of this solver must be closed first)."""
        h, self._handle = getattr(self, "_handle", None), None
        if h is not None and h.value:
            _lib.lib().wlsqm_solver_destroy(h)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _use_stream(self):
        sp = _lib.current_stream_ptr(self.device)
        if sp is not None and sp != getattr(self, "_stream", -1):
            _lib.check(_lib.lib().wlsqm_solver_set_stream(self._handle, sp))
            self._stream = sp

    def keep_solution(self, keep=True):
        """Extension: keep=False drops the solver's own copy of the solution (the reference's Case_set_fi, infra.pyx:780-786)
        for solve() calls with a CUDA-tensor fi: 8*no bytes per case less traffic; interpolate() then raises until a
        solve() with the copy enabled."""
        _lib.check(_lib.lib().wlsqm_solver_keep_solution(self._handle, 1 if keep else 0))

    def synchronize(self):
        """Wait for everything enqueued by this solver (only needed with CUDA-tensor arguments)."""
        _lib.check(_lib.lib().wlsqm_solver_synchronize(self._handle))

    def memory_used(self):
        """(bytes of solver state on the device, state + staging buffers) -- ``expert.pyx:289-306``."""
        used, total = C.c_int64(), C.c_int64()
        _lib.check(_lib.lib().wlsqm_solver_memory(self._handle, C.byref(used), C.byref(total)))
        return (used.value, total.value)

    # -- prepare --------------------------------------------------------------------------------------
    def prepare(self, xi, xk):
        """Generate, scale and factor the problem matrices and store the solution operators
        (``expert.pyx:309-426``).  xi: (ncases, dim) [1D: (ncases,)], xk: (ncases, >=max nk, dim)
        [1D: (ncases, >=max nk)], float64."""
        self.ready = False
        if self.host is not None:
            # guest mode: geometry (and operators) are the host's (expert.pyx:348-385)
            self.xk, self.xi = self.host.xk, self.host.xi
            xi, xk = self.xi, self.xk
            if self._borrows:
                _lib.check(_lib.lib().wlsqm_solver_prepare_guest(self._handle))
                self.ready = True
                return
        dim = self.dimension
        if dim >= 2:
            xi_a = _lib.as_arr(xi, np.float64, 2, "xi")
            xk_a = _lib.as_arr(xk, np.float64, 3, "xk")
            if xi_a.shape[1] < dim or xk_a.shape[2] < dim:
                raise ValueError("xi and xk must have %d coordinates on their last axis" % dim)
            xi_s0, xk_s0, xk_s1 = xi_a.strides[0], xk_a.strides[0], xk_a.strides[1]
        else:
            xi_a = _lib.as_arr(xi, np.float64, 1, "xi", last_contig=False)
            xk_a = _lib.as_arr(xk, np.float64, 2, "xk", last_contig=False, allow_copy=True)
            xi_s0, xk_s0, xk_s1 = xi_a.strides[0], xk_a.strides[0], xk_a.strides[1]
        if xi_a.shape[0] < self.ncases or xk_a.shape[0] < self.ncases:
            raise ValueError("xi and xk must have at least ncases = %d rows" % self.ncases)
        if self.ncases and xk_a.shape[1] < self._maxnk:
            raise ValueError("xk must hold at least max(nk) = %d neighbours per case" % self._maxnk)
        if not xk_a.is_cuda and dim >= 2 and self._maxnk > 1 and (xk_s1 != dim or xk_a.shape[2] != dim):
            # host rows must be dense with exactly `dim` coordinates; the reference's double[:,:,::contiguous] view also
            # accepts pitched rows / a longer last axis and reads only the first dim columns
            xk_a = _lib.as_arr(np.ascontiguousarray(xk_a.np[:, :, :dim]), np.float64, 3, "xk")
            xk_s0, xk_s1 = xk_a.strides[0], xk_a.strides[1]
        if not xk_a.is_cuda and dim == 1 and self._maxnk > 1 and xk_s1 != 1:
            xk_a = _lib.as_arr(np.ascontiguousarray(xk_a.np), np.float64, 2, "xk", last_contig=False)
            xk_s0, xk_s1 = xk_a.strides[0], xk_a.strides[1]
        self._use_stream()
        if self.host is None:
            self.xk, self.xi, self.tree = xk, xi, None
        _lib.check(_lib.lib().wlsqm_solver_prepare(self._handle, xi_a.ptr, xi_s0, xk_a.ptr, xk_s0, xk_s1))
        self._cuda_out = bool(xk_a.is_cuda)
        self.ready = True

    def conds(self):
        """2-norm condition number of the scaled problem matrix of every case (needs debug=True;
        ``expert.pyx:429-464``)."""
        if not self.ready:
            raise RuntimeError("Solver is not in the ready state; prepare() must be called before conds()")
        if not self.debug:
            raise RuntimeError("Not in debug mode; condition number data has not been computed")
        out = np.empty((self.ncases,), dtype=np.float64)
        _lib.check(_lib.lib().wlsqm_solver_conds(self._handle, out.ctypes.data))
        return out

    # -- neighbourhoods as index lists (extension) ----------------------------------------------------
    def prepare_hoods(self, x, hoods, xi=None):
        """``prepare(xi, x[hoods])`` with the gather done on the device (extension).

        x: (npoints, dim) [1D: (npoints,)] float64; hoods: (ncases, >= max nk) int32 indices into x (numpy or
        CUDA tensor, e.g. from ``PointGrid.knn``); xi: the origins, default ``x[:ncases]``."""
        self.ready = False
        from .. import neighbors
        xa, npts, dim, x_s0 = neighbors._points(x)
        if dim != self.dimension:
            raise ValueError("x has %d coordinates, the solver has dimension %d" % (dim, self.dimension))
        ha = _lib.as_arr(hoods, np.int32, 2, "hoods")
        if ha.shape[0] < self.ncases or (self.ncases and ha.shape[1] < self._maxnk):
            raise ValueError("hoods must have shape (>= ncases, >= max nk)")
        xi_p, xi_s0 = None, 0
        if xi is not None:
            xia, nxi, dimi, xi_s0 = neighbors._points(xi, "xi")
            if dimi != dim or nxi < self.ncases:
                raise ValueError("xi must hold one origin per case")
            xi_p = xia.ptr
        elif npts < self.ncases:
            raise ValueError("without xi, x must hold one point per case")
        self._use_stream()
        _lib.check(_lib.lib().wlsqm_solver_prepare_hoods(self._handle, xa.ptr, x_s0, npts, ha.ptr, ha.strides[0], xi_p, xi_s0))
        self.xi = xi if xi is not None else x[:self.ncases]
        self.xk, self.tree = None, None
        self._hood_points = npts
        self._cuda_out = bool(ha.is_cuda)
        self.ready = True

    # -- export of the prepared operators (extension; opexport.py) --------------------------------------------------------
    def stencils(self, coeffs):
        """(W, K): the prepared operators contracted with coefficient rows -- W (nops, ncases, max nk) weights on fk,
        K (nops, ncases, max no) weights on the known values, so that sum_s c[s] fi[i, s] = W[i] . fk[i] + K[i] . fi[i]
        for an ALGO_BASIC solve.  coeffs: an int slot, a (max no,) row or a (nops, max no) array (the nops axis is dropped
        for the first two).  The d fi / d fk of the reference's sens (impl.pyx:769-779); an ALGO_ITERATIVE solver exports
        the same operator (the refinement corrections are not part of it)."""
        return opexport.stencils(self, coeffs)

    def operator(self, coeffs, center=None):
        """(D, K): the global sparse operator (ncases, npoints) over the points of prepare_hoods (torch CSR on the
        device for CUDA hoods, scipy csr_array otherwise; a list for 2-D coeffs) and the known-value weights.
        center: index in x of case 0's own point -- the weight on a known F of case i then goes to column center + i.
        See wlsqm_b200.fitter.opexport.operator."""
        return opexport.operator(self, coeffs, center)

    def solve_hoods(self, f, fi, sens=None):
        """``solve(f[hoods], fi, sens)`` with the gather done on the device (extension; needs prepare_hoods).
        f: (npoints,) float64 -- one value per point instead of one per (point, neighbour)."""
        if not self.ready:
            raise RuntimeError("Solver is not in the ready state; prepare() must be called before solve()")
        fa = _lib.as_arr(f, np.float64, 1, "f", last_contig=False)
        if fa.shape[0] < getattr(self, "_hood_points", 0):
            raise ValueError("f must hold one value per point of the x given to prepare_hoods()")
        fi_a = _lib.as_arr(fi, np.float64, 2, "fi", writable=True)
        if fi_a.shape[0] < self.ncases or (self.ncases and fi_a.shape[1] < self._maxno):
            raise ValueError("fi must have shape (>= ncases, >= %d)" % self._maxno)
        sens_p, s0, s1 = None, 0, 0
        if self.do_sens:
            if sens is None:
                raise ValueError("sens must be given when do_sens is set")
            sens_a = _lib.as_arr(sens, np.float64, 3, "sens", writable=True)
            sens_p, s0, s1 = sens_a.ptr, sens_a.strides[0], sens_a.strides[1]
        self._use_stream()
        it = C.c_int32(0)
        _lib.check(_lib.lib().wlsqm_solver_solve_hoods(self._handle, fa.ptr, fa.strides[0] if fa.shape[0] > 1 else 1,
                                                       fi_a.ptr, fi_a.strides[0], sens_p, s0, s1, C.byref(it)))
        return int(it.value)

    # -- solve ------------------------------------------------------------------------------------------
    def solve(self, fk, fi, sens=None):
        """Fit the model to the data fk using the prepared geometry (``expert.pyx:467-655``).

        fk (ncases, >=max nk); fi (ncases, >=max no) in/out: knowns are read, unknowns written in place;
        sens (ncases, >=max nk, >=max no) out, needed iff do_sens.  Returns the maximum number of
        refinement iterations taken (0 for ALGO_BASIC)."""
        if not self.ready:
            raise RuntimeError("Solver is not in the ready state; prepare() must be called before solve()")
        fk_a = _lib.as_arr(fk, np.float64, 2, "fk", last_contig=False, allow_copy=True)
        fi_a = _lib.as_arr(fi, np.float64, 2, "fi", writable=True)
        if fk_a.shape[0] < self.ncases or fi_a.shape[0] < self.ncases:
            raise ValueError("fk and fi must have at least ncases = %d rows" % self.ncases)
        if self.ncases and (fk_a.shape[1] < self._maxnk or fi_a.shape[1] < self._maxno):
            raise ValueError("fk needs >= %d columns and fi >= %d columns" % (self._maxnk, self._maxno))
        if not fk_a.is_cuda and self._maxnk > 1 and fk_a.strides[1] != 1:
            fk_a = _lib.as_arr(np.ascontiguousarray(fk_a.np), np.float64, 2, "fk")
        sens_p, s0, s1 = None, 0, 0
        if self.do_sens:
            if sens is None:
                raise ValueError("sens must be given when do_sens is set")
            sens_a = _lib.as_arr(sens, np.float64, 3, "sens", writable=True)
            if sens_a.shape[0] < self.ncases or (self.ncases and (sens_a.shape[1] < self._maxnk
                                                                  or sens_a.shape[2] < self._maxno)):
                raise ValueError("sens must have shape (>= ncases, >= max nk, >= max no)")
            sens_p, s0, s1 = sens_a.ptr, sens_a.strides[0], sens_a.strides[1]
        self._use_stream()
        it = C.c_int32(0)
        _lib.check(_lib.lib().wlsqm_solver_solve(self._handle, fk_a.ptr, fk_a.strides[0], fk_a.strides[1],
                                                 fi_a.ptr, fi_a.strides[0], sens_p, s0, s1, C.byref(it)))
        return int(it.value)

    def solve_fields(self, fk, fi):
        """Fit nf fields on the prepared geometry in one pass over the stored operators (extension).

        fk (nf, >= ncases, >= max nk); fi (nf, >= ncases, >= max no) in/out, fields-outer or fields-inner rows (e.g.
        ``fi_all.transpose(1, 0, 2)`` of an (ncases, nf, no) array).  Field j's unknown slots are bit for bit what
        ``solve(fk[j], fi[j])`` writes; returns the maximum of those solves' return values, and iterations() gives the
        per-case maximum.  The solver's own solution copy is not written (interpolate() raises until the next solve());
        sens is not produced.  See wlsqm_b200.fitter.fields."""
        return fields.solve_fields(self, fk, fi)

    def solve_hoods_fields(self, f, fi):
        """solve_fields with the data per point (extension; needs prepare_hoods): f (nf, >= npoints), any strides --
        ``f_all.T`` of an (npoints, nf) array is fine.  Field j equals ``solve_hoods(f[j], fi[j])`` bit for bit."""
        return fields.solve_hoods_fields(self, f, fi)

    def iterations(self):
        """Per-case refinement iteration counts of the last solve (extension; zeros for ALGO_BASIC)."""
        out = np.zeros((self.ncases,), dtype=np.int32)
        _lib.check(_lib.lib().wlsqm_solver_iterations(self._handle, out.ctypes.data))
        return out

    # -- interpolate ----------------------------------------------------------------------------------
    def _xi_host(self):
        xi = self.xi
        if _lib._is_torch_tensor(xi):
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
            search = 'gpu' if _lib._is_torch_tensor(self.xi) and self.xi.is_cuda else 'scipy'
        if search not in ('scipy', 'gpu'):
            raise ValueError("search must be 'scipy' or 'gpu'; got %r" % (search,))
        self._use_stream()
        _lib.check(_lib.lib().wlsqm_solver_index_models(self._handle))
        if self.host is not None and self.host.tree is not None:
            self.tree = self.host.tree
        elif search == 'gpu':
            self.tree = _DeviceModelIndex(self)
        else:
            import scipy.spatial
            xi = self._xi_host()
            xi_rank2 = xi if self.dimension >= 2 else np.atleast_2d(xi).T
            self.tree = scipy.spatial.cKDTree(data=xi_rank2)

    def _nearest_models(self, x, xp, x_s0, nx, x_cuda, I):
        """(I_use, I_out): the model of every query in mode='nearest' -- I itself when given, else the nearest origin
        by self.tree (the device grid for CUDA queries or search='gpu', I then stays where x lives; cKDTree otherwise).
        interpolate() and the interpolation operators (opexport.py) resolve their models here."""
        if I is not None:
            return I, I
        if isinstance(self.tree, _DeviceModelIndex) or x_cuda:
            # nearest model by the device-side grid (extension); I stays where x lives
            if x_cuda:
                import torch
                I_out = torch.empty((nx,), dtype=torch.int64, device=x.device)
                ip = int(I_out.data_ptr())
            else:
                I_out = np.empty((nx,), dtype=np.int_)
                ip = I_out.ctypes.data
            _lib.check(_lib.lib().wlsqm_solver_nearest_models(self._handle, xp, x_s0, nx, ip))
            return I_out, I_out
        xh = np.asarray(x)
        xq = xh if self.dimension >= 2 else np.atleast_2d(xh).T
        _d, I_h = self.tree.query(xq, k=1)
        I_out = np.ascontiguousarray(I_h, dtype=np.int_)
        return I_out, I_out

    # -- interpolation operators (extension; opexport.py) -----------------------------------------------------------------
    def interp_stencils(self, x, coeffs=0, I=None, mode='nearest', r=None):
        """(W, K, I_out): the map from the data to interpolate(x, mode='nearest') as per-query weights -- W (nops, nx,
        max nk) on fk[I[q]], K (nops, nx, max no) on the known values of model I[q], for the coefficient rows coeffs over
        the derivative slots (an int slot, a (max no,) row or a (nops, max no) array).  I=None: the nearest models, found
        as interpolate() finds them.  mode='continuous' (needs r, refuses I): one row per (query, model) pair of the
        models within r, returned as (W, K, (pair_ptr, J)).  See wlsqm_b200.fitter.opexport.interp_stencils."""
        return opexport.interp_stencils(self, x, coeffs, I, mode, r)

    def interp_operator(self, x, coeffs=0, I=None, center=None, mode='nearest', r=None):
        """(E, K, I_out): the same map as a sparse matrix (nx, npoints) over the points of prepare_hoods, like operator().
        mode='continuous': (E, K, (pair_ptr, J)) with K per pair.  See wlsqm_b200.fitter.opexport.interp_operator."""
        return opexport.interp_operator(self, x, coeffs, I, center, mode, r)

    def interpolate(self, x, mode='nearest', r=None, diff=0, I=None):
        """Interpolate the global patched model or one derivative of it (``expert.pyx:687-781``).

        Returns (out, I_out).  ``diff='all'`` (extension, mode='nearest') returns out of shape
        (nx, max no): every derivative slot in one pass."""
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
        cdiff = _lib.DIFF_ALL if all_diffs else int(diff)
        dim = self.dimension
        x_a = _lib.as_arr(x, np.float64, 2 if dim >= 2 else 1, "x", last_contig=dim >= 2)
        nx = x_a.shape[0]
        x_s0 = x_a.strides[0]
        if not x_a.is_cuda and dim == 1 and nx > 1 and x_s0 != 1:
            x_a = _lib.as_arr(np.ascontiguousarray(x_a.np), np.float64, 1, "x", last_contig=False)
            x_s0 = 1
        self._use_stream()
        if mode == 'continuous':
            return self._interpolate_continuous(x_a, x_s0, float(r), cdiff), np.asanyarray(None)

        I_use, I_out = self._nearest_models(x, x_a.ptr, x_s0, nx, x_a.is_cuda, I)
        I_a = _lib.as_arr(I_use, np.int64, 1, "I")
        if not I_a.is_cuda and I_a.strides[0] != 1 and nx > 1:
            raise ValueError("I: ndarray is not C-contiguous")
        width = self._maxno if all_diffs else 1
        if x_a.is_cuda:
            import torch
            out = torch.empty((nx, width) if all_diffs else (nx,), dtype=torch.float64, device=x.device)
            out_p = int(out.data_ptr())
        else:
            out = np.empty((nx, width) if all_diffs else (nx,), dtype=np.float64)
            out_p = out.ctypes.data
        # a query that found no neighbour (NaN coordinates) poisons the whole output (expert.pyx:862-870)
        if not I_a.is_cuda and nx and (I_a.np == self.ncases).any():
            out[...] = np.nan
            return out, np.asanyarray(I_out)
        _lib.check(_lib.lib().wlsqm_solver_interpolate(self._handle, x_a.ptr, x_s0, I_a.ptr, nx, cdiff, out_p, width))
        return out, (I_out if x_a.is_cuda and _lib._is_torch_tensor(I_out) else np.asanyarray(I_out))

    def interpolate_fields(self, x, fi, mode='nearest', r=None, diff=0, I=None):
        """interpolate() for nf caller-held solutions at once (extension): fi (nf, >= ncases, >= max no), e.g. the fi of
        solve_fields (fi[None] for one field).  Returns (out, I_out) with out (nf, nx), or (nf, nx, max no) for
        diff='all'; out[j] is bit for bit what interpolate() returns on a solver whose last solve() produced fi[j].  The
        solver's own solution copy is not used, so this works after solve_fields and keep_solution(False).  See
        wlsqm_b200.fitter.fields.interpolate_fields."""
        return fields.interpolate_fields(self, x, fi, mode, r, diff, I)

    def _interpolate_continuous(self, x_a, x_s0, r, cdiff):
        """mode='continuous' (``expert_interpolate_continuous``, ``expert.pyx:898-985``): weighted average
        over every local model whose origin lies within r; weights (1 - sqrt(d2/r2))^2.  One kernel: each query
        walks the cells of the model-origin grid that meet its ball and evaluates the models on the fly."""
        if cdiff < 0:
            raise ValueError("diff='all' is not available in mode='continuous'")
        nx = x_a.shape[0]
        if x_a.is_cuda:
            import torch
            out = torch.empty((nx,), dtype=torch.float64, device=x_a.keep.device)
            op = int(out.data_ptr())
        else:
            out = np.empty((nx,), dtype=np.float64)
            op = out.ctypes.data
        _lib.check(_lib.lib().wlsqm_solver_interpolate_continuous(self._handle, x_a.ptr, x_s0, nx, r, cdiff, op))
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
        from .. import neighbors
        xa, nx, dim, x_s0 = neighbors._points(x)
        I = np.empty((nx,), dtype=np.int_)
        if xa.is_cuda:
            import torch
            It = torch.empty((nx,), dtype=torch.int64, device=x.device)
            _lib.check(_lib.lib().wlsqm_solver_nearest_models(s._handle, xa.ptr, x_s0, nx, int(It.data_ptr())))
            return None, It
        _lib.check(_lib.lib().wlsqm_solver_nearest_models(s._handle, xa.ptr, x_s0, nx, I.ctypes.data))
        return None, I


# ---- the shipped binding is the Cython shim (wlsqm_b200/_shim.pyx); this module's ctypes twin above is the fallback ------
import os as _os

if _os.environ.get("WLSQM_BINDING", "cython") != "ctypes":
    try:
        from .._shim import ExpertSolver, number_of_dofs, _DeviceModelIndex, BINDING     # noqa: F401,F811
    except ImportError:      # the shim has not been built (python-wlsqm_b200/build_shim.py): ctypes serves the same API
        pass
