"""GPU tests of the continuous-mode interpolation operators: ExpertSolver.interp_stencils / .interp_operator with
mode='continuous' (csrc/wlsqm_operator.cu, include/wlsqm_b200.h).

The pairs (query, model within r) must be the sorted cKDTree.query_ball_point rows and the ball rule restated in numpy
(tests/interp_continuous_reference.py); a pair's rows must equal stencils(alpha * c_q)[J[p]] bit for bit with alpha and
c_q formed on the host; the CSR must equal the host merge of the same rows.  Against solve_hoods + interpolate(mode=
'continuous') the rows are held to the identity bound of the nearest-mode operators, summed over the pairs, plus the
rounding of the weighted average.  Clouds and offsets are dyadic.
"""
import ctypes as C
import math

import numpy as np
import pytest
from scipy.spatial import cKDTree

import wlsqm_b200 as w
from wlsqm_b200 import _lib
from wlsqm_b200.fitter import defs
import interp_operator_reference as iref
import interp_continuous_reference as cref
from test_interp_operator_reference import IDENTITY_CONST
from test_gpu_interp_operator import _batch, _solver, _np, _eq, _csr_parts, _x

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

EPS = np.finfo(np.float64).eps


def _spacing(xi):
    d, _ = cKDTree(xi).query(xi, 2)
    return float(np.median(d[:, 1]))


def _near(b, nq, seed, frac=0.25):
    """dyadic queries within frac * spacing of an origin per axis: every query has a model well inside r >= spacing"""
    rng = np.random.default_rng(seed)
    n, dim = len(b["nk"]), b["dim"]
    h = _spacing(b["xi"])
    step = 2.0 ** math.floor(math.log2(frac * h))
    return b["xi"][rng.integers(0, n, nq)] + rng.integers(-8, 9, size=(nq, dim)) / 8.0 * step


def _lattice_solver(dim, xi, k=None, order=1):
    k = k or {1: 4, 2: 8, 3: 12}[dim]
    n = len(xi)
    _, hoods = cKDTree(xi).query(xi, k)
    s = w.ExpertSolver(dim, np.full(n, k, np.int32), np.full(n, order, np.int32), np.zeros(n, np.int64),
                       np.ones(n, np.int32))
    s.prepare_hoods(xi if dim > 1 else xi[:, 0], hoods.astype(np.int32))
    s.prep_interpolate(search="gpu")
    return s


def _kdtree_rows(xi, xq, r):
    ok = np.isfinite(xq).all(1)
    rows = [[] for _ in range(len(xq))]
    if ok.any():
        for q, row in zip(np.flatnonzero(ok), cKDTree(xi).query_ball_point(xq[ok], r)):
            rows[q] = sorted(row)
    ptr = np.concatenate([[0], np.cumsum([len(t) for t in rows])]).astype(np.int64)
    return ptr, np.array([m for t in rows for m in t], np.int64)


def _clouds(dim, layout, rng):
    if layout == "uniform":
        xi = rng.integers(0, 2 ** 20, size=(300, dim)) / 2.0 ** 20
        r = 2.0 * _spacing(xi)
    elif layout == "clustered":
        centres = rng.integers(0, 2 ** 20, size=(6, dim)) / 2.0 ** 20
        xi = centres[rng.integers(0, 6, 300)] + rng.integers(-2 ** 14, 2 ** 14, size=(300, dim)) / 2.0 ** 20
        r = 3.0 * _spacing(xi)
    else:                                          # dyadic lattice: queries on the half-lattice, origins at exactly r
        g = {1: 64, 2: 12, 3: 6}[dim]
        axes = np.meshgrid(*[np.arange(g) / 16.0] * dim, indexing="ij")
        xi = np.stack([a.ravel() for a in axes], 1)
        r = 1.0 / 16.0
    lo, hi = xi.min(0) - 3 * r, xi.max(0) + 3 * r
    xq = lo + rng.integers(0, 2 ** 16, size=(400, dim)) / 2.0 ** 16 * (hi - lo)
    if layout == "lattice":
        xq = np.round(xq * 32.0) / 32.0
    xq[[3, 77]] = np.nan
    xq[5, 0] = np.inf
    return xi, xq, r


@pytest.mark.parametrize("layout", ["uniform", "clustered", "lattice"])
@pytest.mark.parametrize("dim", [1, 2, 3])
def test_pairs_equal_ckdtree(dim, layout):
    rng = np.random.default_rng(dim * 7 + len(layout))
    xi, xq, r = _clouds(dim, layout, rng)
    s = _lattice_solver(dim, xi)
    _, _, (pp, J) = s.interp_stencils(_x(dict(dim=dim), xq), 0, mode="continuous", r=r)
    want_p, want_J = _kdtree_rows(xi, xq, r)
    assert np.array_equal(pp, want_p) and np.array_equal(J, want_J)
    rp, rJ, _ = cref.pairs(xi, xq, r)
    assert np.array_equal(pp, rp) and np.array_equal(J, rJ)
    assert (np.diff(pp)[[3, 5, 77]] == 0).all() and J.dtype == np.int64
    if layout == "lattice":                        # members at exactly r are present
        d2 = np.concatenate([cref.ball_d2(xi[J[pp[q]:pp[q + 1]]], xq[q]) for q in range(len(xq))])
        assert (d2 == r * r).sum() >= 20


@pytest.mark.parametrize("knowns_mode", [0, "F", "rand"])
@pytest.mark.parametrize("dim,orders,k", [(1, [3], 8), (2, [4], 20), (3, [4], 40), (2, [2, 3, 4], 20), (3, [0, 2, 4], 40)])
def test_pair_rows_equal_stencils_of_host_rows(dim, orders, k, knowns_mode):
    b = _batch(dim, orders, k, knowns_mode, hetero_nk=len(orders) > 1, seed=dim * 10 + k + 3)
    s = _solver(b)
    s.prep_interpolate(search="gpu")
    maxno = s._maxno
    r = 2.5 * _spacing(b["xi"])
    xq = _near(b, 120, seed=k, frac=1.0)
    rng = np.random.default_rng(k)
    cs = [np.eye(maxno)[[0]], rng.standard_normal((3, maxno))]
    if maxno == 35:
        cs.append(np.vstack([np.eye(35)[:33], rng.standard_normal((2, 35))]))     # 35 coefficient rows
    for c in cs:
        W, K, (pp, J) = s.interp_stencils(_x(b, xq), c, mode="continuous", r=r)
        rp, rJ, d2 = cref.pairs(b["xi"], xq, r)
        assert np.array_equal(pp, rp) and np.array_equal(J, rJ)
        alpha, _, _ = cref.weights(pp, d2, r)
        assert W.shape == (len(c), len(J), s._maxnk) and K.shape == (len(c), len(J), maxno)
        sample = rng.choice(len(J), min(len(J), 40), replace=False)
        q_of = np.searchsorted(pp, np.arange(len(J)), side="right") - 1
        per = max(1, 35 // len(c))
        for j0 in range(0, len(sample), per):
            ps = sample[j0:j0 + per]
            cqm = np.concatenate([cref.pair_rows(dim, c, xq[[q_of[p]]], b["xi"], np.array([0, 1]), J[[p]], alpha[[p]])
                                  for p in ps])                                   # (len(ps), nops, maxno)
            Ws, Ks = s.stencils(cqm.reshape(-1, maxno))
            for t, p in enumerate(ps):
                rows = slice(t * len(c), (t + 1) * len(c))
                assert _eq(W[:, p], Ws[rows, J[p]]), p
                assert _eq(K[:, p], Ks[rows, J[p]]), p


def test_one_model_reduces_to_nearest_rows():
    b = _batch(2, [2, 3, 4], 20, "rand", center=5, hetero_nk=True, seed=41)
    s = _solver(b)
    s.prep_interpolate(search="gpu")
    h = _spacing(b["xi"])
    xq = _near(b, 300, seed=2, frac=0.05)
    c = np.random.default_rng(1).standard_normal((3, 15))
    r = 0.4 * h
    W, K, (pp, J) = s.interp_stencils(xq, c, mode="continuous", r=r)
    E, Ke, (pp2, J2) = s.interp_operator(xq, c, mode="continuous", r=r, center=5)
    assert np.array_equal(pp, pp2) and np.array_equal(J, J2)
    one = np.flatnonzero(np.diff(pp) == 1)
    assert len(one) > 100
    I = J[pp[one]]
    Wn, Kn, _ = s.interp_stencils(xq[one], c, I)
    assert _eq(W[:, pp[one]], Wn) and _eq(K[:, pp[one]], Kn)
    En, Ken, _ = s.interp_operator(xq[one], c, I, center=5)
    assert _eq(Ke[:, pp[one]], Ken)
    for (r0, c0, v0), (r1, c1, v1) in zip(_csr_parts(E), _csr_parts(En)):
        m = iref.opref.sp.csr_array((v0, c0, r0), shape=(len(xq), len(b["x"])))[one]
        assert np.array_equal(m.indptr, r1) and np.array_equal(m.indices, c1) and _eq(m.data, v1)


def _c_abi_csr(s, xq, r, c, center, bits):
    L = _lib.lib()
    xq = np.ascontiguousarray(xq)
    x_s0 = xq.shape[1] if xq.ndim > 1 else 1
    npairs, nnz = C.c_int64(), C.c_int64()
    pp = np.zeros(len(xq) + 1, np.int64)
    _lib.check(L.wlsqm_solver_interp_continuous_count(s._handle, xq.ctypes.data, x_s0, len(xq), r, center, pp.ctypes.data,
                                                      C.byref(npairs), C.byref(nnz)))
    it = np.int32 if bits == 32 else np.int64
    J = np.zeros(npairs.value, np.int64)
    rowptr, col = np.zeros(len(xq) + 1, it), np.zeros(nnz.value, it)
    values = np.zeros((c.shape[0], nnz.value))
    K = np.zeros((c.shape[0], npairs.value, s._maxno))
    _lib.check(L.wlsqm_solver_interp_continuous_operator_csr(s._handle, xq.ctypes.data, x_s0, len(xq), r, c.shape[0],
                                                             c.ctypes.data, center, bits, pp.ctypes.data, J.ctypes.data,
                                                             rowptr.ctypes.data, col.ctypes.data, values.ctypes.data,
                                                             K.ctypes.data))
    return pp, J, rowptr, col, values, K


@pytest.mark.parametrize("knowns_mode,center,rmul,nq", [(0, None, 2.5, 300), ("F", 0, 2.5, 300), ("F", 23, 1.5, 300),
                                                        ("rand", 23, 2.5, 300), ("F", 23, 12.0, 12)])
@pytest.mark.parametrize("dim,orders,k", [(2, [4], 20), (3, [2, 3, 4], 40), (1, [2], 8)])
def test_csr_equals_host_merge(dim, orders, k, knowns_mode, center, rmul, nq):
    """duplicate neighbours in hoods (_batch), centre folding, and with rmul = 12 rows of thousands of candidates"""
    b = _batch(dim, orders, k, knowns_mode, center=center or 0, hetero_nk=True, seed=7 + k)
    s = _solver(b)
    s.prep_interpolate(search="gpu")
    maxno, npoints = s._maxno, len(b["x"])
    r = rmul * _spacing(b["xi"])
    xq = _near(b, nq, seed=k, frac=2.0)
    c = np.vstack([np.eye(maxno)[:3], np.random.default_rng(k).standard_normal((2, maxno))])
    W, K, (pp, J) = s.interp_stencils(_x(b, xq), c, mode="continuous", r=r)
    rp, col, vals, Kf = cref.csr(W, K, b["hoods"], b["nk"], b["knowns"], pp, J, center=center)
    E, Ke, (pp2, J2) = s.interp_operator(_x(b, xq), c, center=center, mode="continuous", r=r)
    assert np.array_equal(pp, pp2) and np.array_equal(J, J2) and len(E) == len(c)
    for o in range(len(c)):
        assert E[o].shape == (len(xq), npoints) and E[o].indices.dtype == np.int32
        assert np.array_equal(E[o].indptr, rp) and np.array_equal(E[o].indices, col)
        assert _eq(E[o].data, vals[o]), o
    assert _eq(Ke, Kf)
    if rmul > 10 and dim > 1:
        assert (np.diff(pp) * (s._maxnk + 1)).max() > 2000          # candidates of one row
    cen = -1 if center is None else center
    r32 = _c_abi_csr(s, xq, r, c, cen, 32)
    r64 = _c_abi_csr(s, xq, r, c, cen, 64)
    assert r64[2].dtype == np.int64 and np.array_equal(r32[2], r64[2]) and np.array_equal(r32[3], r64[3])
    assert np.array_equal(r32[0], pp) and np.array_equal(r32[1], J) and np.array_equal(r32[2], rp)
    assert _eq(r32[4], vals) and _eq(r64[4], vals) and _eq(r32[5], Kf) and _eq(r64[5], Kf)


@pytest.mark.parametrize("cap,chunk", [(None, None), ("0", None), ("0", "2000"), ("128", "3000"), ("64", "700")])
def test_row_merge_and_sort_route_across_chunks(monkeypatch, cap, chunk):
    """rows of at most WLSQM_CONT_ROW_CAP candidate slots are merged by one warp in shared memory, longer ones by the sort
    route over chunks of at most WLSQM_CONT_CHUNK_SLOTS slots (a longer row is a chunk of its own): every split gives
    the host merge bit for bit, with short and long rows mixed in one call"""
    for name, val in (("WLSQM_CONT_ROW_CAP", cap), ("WLSQM_CONT_CHUNK_SLOTS", chunk)):
        if val is None:
            monkeypatch.delenv(name, raising=False)
        else:
            monkeypatch.setenv(name, val)
    b = _batch(2, [2, 3, 4], 20, "F", center=23, hetero_nk=True, seed=27)
    s = _solver(b)
    s.prep_interpolate(search="gpu")
    r = 2.5 * _spacing(b["xi"])
    xq = _near(b, 200, seed=5, frac=2.0)
    xq[[10, 11]] = [[7.0, 7.0], [np.nan, 0.5]]                   # empty rows among them
    c = np.vstack([np.eye(15)[[0, 3]], np.random.default_rng(5).standard_normal((1, 15))])
    W, K, (pp, J) = s.interp_stencils(xq, c, mode="continuous", r=r)
    slots = np.diff(pp) * (s._maxnk + 1)
    assert (slots[slots > 0] <= 128).any() and (slots > 128).any()
    rp, col, vals, Kf = cref.csr(W, K, b["hoods"], b["nk"], b["knowns"], pp, J, center=23)
    E, Ke, _ = s.interp_operator(xq, c, center=23, mode="continuous", r=r)
    for o in range(len(c)):
        assert np.array_equal(E[o].indptr, rp) and np.array_equal(E[o].indices, col) and _eq(E[o].data, vals[o])
    assert _eq(Ke, Kf)
    r64 = _c_abi_csr(s, xq, r, c, 23, 64)
    assert np.array_equal(r64[2], rp) and np.array_equal(r64[3], col) and _eq(r64[4], vals)


def _unknown_columns(sens, knowns, nos):
    maxno = sens.shape[2]
    unk = np.array([[s < no and not (int(kn) >> s) & 1 for s in range(maxno)] for kn, no in zip(knowns, nos)])
    return np.where(unk[:, None, :], sens, 0.0)


def _continuous_bound(dim, c, xq, xi, pp, J, d2, r, sens_p, dfk_p, fk_p, fi_in_p, fi_out_p):
    """per query and operator: the nearest-mode identity bound of every pair with |alpha c_q|, summed over the pairs,
    plus the rounding of the weighted average (a weight's error is about eps * sqrt(w) / S relative to the value)"""
    alpha, wgt, S = cref.weights(pp, d2, r)
    q_of = np.searchsorted(pp, np.arange(len(J)), side="right") - 1
    h_abs = np.abs(xq[q_of] - xi[J])
    cq_abs = np.stack([iref.coefficient_rows_at(dim, np.abs(c), h_abs[p]) for p in range(len(J))])   # (npairs, nops, no)
    base = iref.identity_bound(np.transpose(alpha[:, None, None] * cq_abs, (1, 0, 2)), sens_p, dfk_p, fk_p, fi_in_p,
                               fi_out_p, IDENTITY_CONST)                                                # (nops, npairs)
    npq = np.diff(pp)[q_of]
    val = np.einsum("pos,ps->op", cq_abs, np.abs(fi_out_p))
    avg = 8.0 * (npq + 2) * EPS * (np.sqrt(wgt) / S[q_of] + alpha) * val
    tot = base + avg
    return np.stack([np.add.reduceat(tot[o], pp[:-1]) for o in range(len(c))])


def _identity(b, s, c, xq, r):
    rng = np.random.default_rng(1)
    n, maxno, maxnk, npoints = len(b["nk"]), s._maxno, s._maxnk, len(b["x"])
    f = rng.standard_normal(npoints)
    fi_in = rng.standard_normal((n, maxno))
    fi_out = fi_in.copy()
    sens = np.zeros((n, maxnk, maxno))
    s.solve_hoods(f, fi_out, sens)
    E, K, (pp, J) = s.interp_operator(_x(b, xq), c, mode="continuous", r=r)
    assert (np.diff(pp) > 0).all()
    Kfi = np.einsum("ops,ps->op", K, fi_in[J])
    lhs = np.stack([E[o] @ f for o in range(len(E))]) + np.stack([np.add.reduceat(Kfi[o], pp[:-1]) for o in range(len(c))])
    used = np.flatnonzero(np.abs(c).sum(0))
    interp = {D: s.interpolate(_x(b, xq), mode="continuous", r=r, diff=int(D))[0] for D in used}
    rhs = np.stack([sum(c[o, D] * interp[D] for D in used) for o in range(len(c))])

    def solve(fi):
        fo = fi.copy()
        s.solve_hoods(np.zeros(npoints), fo, np.zeros((n, maxnk, maxno)))
        return fo
    dfk = iref.opref.known_weights_from_solves(solve, n, maxno, b["nos"], b["knowns"])
    fk = np.where(np.arange(maxnk)[None, :] < b["nk"][:, None], f[np.minimum(b["hoods"][:, :maxnk], npoints - 1)], 0.0)
    _, _, d2 = cref.pairs(b["xi"], xq, r)
    bound = _continuous_bound(b["dim"], c, xq.reshape(len(xq), -1), b["xi"], pp, J, d2, r,
                              _unknown_columns(sens, b["knowns"], b["nos"])[J], dfk[J], fk[J], fi_in[J], fi_out[J])
    ratio = np.abs(lhs - rhs) / bound
    assert (ratio <= 1.0).all(), float(ratio.max())
    print("continuous identity: worst ratio to the bound %.3f" % float(ratio.max()))


@pytest.mark.parametrize("knowns_mode", [0, "rand"])
@pytest.mark.parametrize("dim,orders,k", [(2, [4], 20), (3, [2, 3, 4], 40), (1, [3], 8)])
def test_identity_against_solve_and_continuous_interpolate(dim, orders, k, knowns_mode):
    b = _batch(dim, orders, k, knowns_mode, seed=21 + k, hetero_nk=len(orders) > 1)
    s = _solver(b, do_sens=True)
    s.prep_interpolate(search="gpu")
    maxno = s._maxno
    ex = iref.EXPONENTS[dim]
    lap = np.zeros(maxno)
    lap[[sl for sl in range(maxno) if sum(ex[sl]) == 2 and max(ex[sl]) == 2]] = 1.0
    first = np.eye(maxno)[[sl for sl in range(maxno) if sum(ex[sl]) == 1][:1]]
    c = np.vstack([np.eye(maxno)[[0]], first, lap[None]])
    _identity(b, s, c, _near(b, 200, seed=3), 2.0 * _spacing(b["xi"]))


@pytest.mark.parametrize("dim,order,k", [(1, 3, 8), (2, 2, 12), (2, 4, 20), (3, 2, 20)])
def test_polynomial_data_exact_derivatives(dim, order, k):
    from test_interp_operator_reference import _poly
    b = _batch(dim, [order], k, "F", center=4, seed=50 + dim)
    s = _solver(b)
    s.prep_interpolate(search="gpu")
    n = len(b["nk"])
    no, deriv = _poly(dim, order, seed=dim)
    xq = _near(b, 800, seed=9)
    f = deriv(b["x"], 0)
    r = 2.0 * _spacing(b["xi"])
    E, K, (pp, J) = s.interp_operator(_x(b, xq), np.eye(s._maxno), center=4, mode="continuous", r=r)
    assert not K.any()                                          # F is the only known and it is folded
    hr = np.median(np.linalg.norm(b["x"][b["hoods"][:, 3]] - b["xi"], axis=-1))
    distinct = np.array([len(np.unique(b["hoods"][i, :b["nk"][i]])) == b["nk"][i] for i in range(n)])
    keep = np.array([distinct[J[pp[q]:pp[q + 1]]].all() for q in range(len(xq))])
    assert keep.sum() > 30
    for D in range(no):
        want = deriv(xq.reshape(len(xq), -1), D)
        got = E[D] @ f
        tol = 1e-10 * max(1.0, np.abs(want).max()) / hr ** sum(iref.EXPONENTS[dim][D])
        assert np.abs(got - want)[keep].max() < tol, D


def _export(s, xq, c, r, center=None):
    W, K, (p1, J1) = s.interp_stencils(xq, c, mode="continuous", r=r)
    E, Ke, (p2, J2) = s.interp_operator(xq, c, center=center, mode="continuous", r=r)
    return [_np(W), _np(K), _np(Ke), _np(p1), _np(J1), _np(p2), _np(J2)], _csr_parts(E)


def _same(a, b):
    assert all(_eq(u, v) for u, v in zip(a[0], b[0]))
    for (r1, c1, v1), (r2, c2, v2) in zip(a[1], b[1]):
        assert np.array_equal(r1, r2) and np.array_equal(c1, c2) and _eq(v1, v2)


def test_edges_inputs_and_guests():
    b = _batch(2, [2, 3, 4], 20, "rand", center=5, hetero_nk=True, seed=31)
    c = np.random.default_rng(3).standard_normal((2, 15))
    h = _spacing(b["xi"])
    r = 2.0 * h
    xq = _near(b, 200, seed=4, frac=1.0)
    xq[[7, 8]] = [[5.0, 5.0], [-3.0, 0.5]]                       # no model within r
    s = _solver(b)
    with pytest.raises(RuntimeError, match="prep_interpolate"):
        s.interp_stencils(xq, c, mode="continuous", r=r)
    s.prep_interpolate(search="gpu")
    ref_out = _export(s, xq, c, r, center=5)
    pp = ref_out[0][3]
    assert pp[8] == pp[7] == pp[9] and ref_out[1][0][0][8] == ref_out[1][0][0][9]
    _same(ref_out, _export(s, xq, c, r, center=5))                                     # two calls in a row
    for bad in (0.0, -1.0, np.nan):
        with pytest.raises(ValueError):
            s.interp_stencils(xq, c, mode="continuous", r=bad)
        with pytest.raises(ValueError):
            s.interp_operator(xq, c, mode="continuous", r=bad)
    with pytest.raises(ValueError):
        s.interp_stencils(xq, c, np.zeros(len(xq), np.int64), mode="continuous", r=r)
    with pytest.raises(ValueError):
        s.interp_operator(xq, c, mode="continuous")
    W0, K0, (p0, J0) = s.interp_stencils(xq[:0], c, mode="continuous", r=r)          # nx = 0
    E0, _, _ = s.interp_operator(xq[:0], c, mode="continuous", r=r)
    assert W0.shape == (2, 0, s._maxnk) and list(p0) == [0] and len(J0) == 0 and E0[0].shape == (0, len(b["x"]))
    # the caller's pair_ptr must be the count call's
    L = _lib.lib()
    bad_pp = np.ascontiguousarray(pp.copy())
    bad_pp[50:] += 1
    out = np.zeros((2, int(pp[-1]) + 200, s._maxnk))
    assert L.wlsqm_solver_interp_continuous_stencils(s._handle, np.ascontiguousarray(xq).ctypes.data, 2, len(xq), r, 2,
                                                     np.ascontiguousarray(c).ctypes.data, bad_pp.ctypes.data, None,
                                                     out.ctypes.data, None) == _lib.E_VALUE
    # guest: its host's operators with its own model grid
    guest = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"], host=s)
    guest.prepare(None, None)
    guest.prep_interpolate(search="gpu")
    _same(ref_out, _export(guest, xq, c, r, center=5))
    nosol = _solver(b, algorithm=w.ALGO_ITERATIVE, max_iter=3)
    nosol.keep_solution(False)
    nosol.prep_interpolate(search="gpu")
    _same(ref_out, _export(nosol, xq, c, r, center=5))
    dev = torch.device("cuda", s.device)
    st = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"])
    st.prepare_hoods(torch.as_tensor(b["x"], device=dev), torch.as_tensor(b["hoods"], device=dev),
                     xi=torch.as_tensor(b["xi"], device=dev))
    st.prep_interpolate()
    xt = torch.as_tensor(xq, device=dev)
    _same(ref_out, _export(st, xt, c, r, center=5))                                   # CUDA inputs and outputs
    _same(ref_out, _export(st, xq, c, r, center=5))                                   # numpy queries, CUDA solver
    E_t, K_t, (p_t, J_t) = st.interp_operator(xt, c[0], mode="continuous", r=r)
    assert E_t.layout == torch.sparse_csr and E_t.device == dev and p_t.device == dev and J_t.dtype == torch.int64
    # a plain prepare() after prepare_hoods(): the stencils still, the global operator no longer
    xk = b["x"][np.where(np.arange(20)[None, :] < b["nk"][:, None], b["hoods"], 0)]
    s.prepare(b["xi"], xk)
    s.prep_interpolate(search="gpu")
    s.interp_stencils(xq, c, mode="continuous", r=r)
    with pytest.raises(RuntimeError):
        s.interp_operator(xq, c, mode="continuous", r=r)


def test_members_only_at_exactly_r_give_nan():
    """1D lattice origins 1/16 apart, queries half-way between two of them with r = 1/32: S = 0, as interpolate's 0/0"""
    xi = (np.arange(64) / 16.0)[:, None]
    s = _lattice_solver(1, xi, order=1)
    xq = np.array([10.5, 20.5, 30.0]) / 16.0
    r = 1.0 / 32.0
    W, K, (pp, J) = s.interp_stencils(xq, 0, mode="continuous", r=r)
    assert list(np.diff(pp)) == [2, 2, 1]
    assert np.isnan(W[:4]).all() and not np.isnan(W[4]).any()
    E, _, _ = s.interp_operator(xq, 0, mode="continuous", r=r)
    assert np.isnan(E.data[:E.indptr[2]]).all() and not np.isnan(E.data[E.indptr[2]:]).any()
    s.solve_hoods(np.ones(64), np.zeros((64, 2)))
    assert np.isnan(s.interpolate(xq[:2], mode="continuous", r=r)[0]).all()


def test_full_size_cfg2_transfer_queries():
    """cfg2 (1M points, 2D order 4, k = 30) with 1M transfer queries at r = 1.5 h0: the pairs against cKDTree, the
    identity against solve_hoods + interpolate(mode='continuous') on every 2000th query"""
    n, k = 1_000_000, 30
    dev = torch.device("cuda", _lib.default_device())
    g = torch.Generator(device="cpu").manual_seed(1)
    x = torch.rand((n, 2), generator=g, dtype=torch.float64).to(dev)
    xq = torch.rand((n, 2), generator=g, dtype=torch.float64).to(dev)
    hoods = w.knn_hoods(x, k)
    s = w.ExpertSolver(2, np.full(n, k, np.int32), np.full(n, 4, np.int32), np.zeros(n, np.int64),
                       np.full(n, 1, np.int32), do_sens=True)
    s.prepare_hoods(x, hoods)
    s.prep_interpolate()
    r = 1.5 / math.sqrt(n)
    lap = np.zeros(15)
    lap[[defs.i2_X2, defs.i2_Y2]] = 1.0
    E, K, (pp, J) = s.interp_operator(xq, lap, mode="continuous", r=r)
    xh, xqh = _np(x), _np(xq)
    want_p, want_J = _kdtree_rows(xh, xqh, r)
    assert np.array_equal(_np(pp), want_p) and np.array_equal(_np(J), want_J)
    print("cfg2: %.2f pairs per query, %.1f entries per row" % (len(want_J) / n, E.values().numel() / n))
    sens = torch.empty((n, k, 15), dtype=torch.float64, device=dev)
    f = torch.sin(3 * x[:, 0]) * torch.cos(2 * x[:, 1])
    fi_out = torch.zeros((n, 15), dtype=torch.float64, device=dev)
    s.solve_hoods(f, fi_out, sens)
    rows = np.arange(0, n, 2000)
    ppn, Jn = _np(pp), _np(J)
    have = np.diff(ppn)[rows] > 0
    rows = rows[have]
    lhs = _np(E @ f)[rows]                                      # no knowns: K is 0
    rhs = _np(s.interpolate(xq[torch.as_tensor(rows, device=dev)], mode="continuous", r=r, diff=defs.i2_X2)[0]
              + s.interpolate(xq[torch.as_tensor(rows, device=dev)], mode="continuous", r=r, diff=defs.i2_Y2)[0])
    sub_p = np.concatenate([[0], np.cumsum(np.diff(ppn)[rows])])
    sub_J = np.concatenate([Jn[ppn[q]:ppn[q + 1]] for q in rows])
    _, _, d2 = cref.pairs(xh, xqh[rows], r)
    Jt = torch.as_tensor(sub_J, device=dev)
    sens_p = _np(sens[Jt])
    fk_p = _np(f[hoods[Jt].long()])
    fi_o = _np(fi_out[Jt])
    bound = _continuous_bound(2, lap[None], xqh[rows], xh, sub_p, sub_J, d2, r, sens_p, np.zeros((len(sub_J), 15, 15)),
                              fk_p, np.zeros_like(fi_o), fi_o)[0]
    ratio = np.abs(lhs - rhs) / bound
    assert (ratio <= 1.0).all(), float(ratio.max())
    print("cfg2 continuous identity on %d queries: worst ratio to the bound %.3f" % (len(rows), float(ratio.max())))
    torch.cuda.synchronize()
