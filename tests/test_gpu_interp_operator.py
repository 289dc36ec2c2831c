"""GPU tests of the interpolation operators: ExpertSolver.interp_stencils / .interp_operator (csrc/wlsqm_operator.cu).

A row at query q is the node operator of its model I[q] contracted with the coefficient rows c_q (include/wlsqm_b200.h).
Exact checks: at a model origin c_q = coeffs, so the row must equal that model's stencils / operator row bit for bit;
elsewhere it must equal stencils(c_q)[I[q]] with c_q formed on the host (tests/interp_operator_reference.py), and the
CSR the host merge of the same weights.  Against solve + interpolate the rows are held to the identity bound fixed on
the oracle in tests/test_interp_operator_reference.py.  Clouds and query offsets are dyadic, so that a 2^12
translation is exact.
"""
import ctypes as C

import numpy as np
import pytest
from scipy.spatial import cKDTree

import wlsqm_b200 as w
from wlsqm_b200 import _lib
from wlsqm_b200.fitter import defs
import interp_operator_reference as ref
from test_interp_operator_reference import IDENTITY_CONST

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _batch(dim, orders, k, knowns_mode, n=400, center=0, seed=0, hetero_nk=False, extra=37):
    """points x (dyadic), origins x[center:center+n], ragged hoods with duplicates and garbage padding"""
    rng = np.random.default_rng(seed)
    npoints = n + center + extra
    x = rng.integers(0, 2 ** 24, size=(npoints, dim)) / 2.0 ** 24
    xi = x[center:center + n]
    _, hoods = cKDTree(x).query(xi, k)
    hoods = hoods.astype(np.int32)
    hoods[::7, 2] = hoods[::7, 0]                      # the centre twice
    hoods[3::11, 5] = hoods[3::11, 4]                  # other duplicates
    hoods[::9, 1] = hoods[::9, 0]                      # ... three times in every 63rd row: merge order matters
    nk = np.full(n, k, np.int32)
    if hetero_nk:
        nk = rng.integers(k - 5, k + 1, size=n).astype(np.int32)
    nk[::13] = k - 3
    for i in range(n):
        hoods[i, nk[i]:] = npoints + 1000 + i          # never read
    order = rng.choice(orders, size=n).astype(np.int32)
    nos = np.array([defs.NUMBER_OF_DOFS[dim][o] for o in order])
    if knowns_mode == 0:
        knowns = np.zeros(n, np.int64)
    elif knowns_mode == "F":
        knowns = np.ones(n, np.int64)
    else:
        knowns = np.array([int(rng.integers(0, 2 ** no)) & int(rng.integers(0, 2 ** no)) for no in nos], np.int64)
    wm = rng.choice([1, 2], size=n).astype(np.int32)
    return dict(dim=dim, x=x, xi=xi, hoods=hoods, nk=nk, order=order, knowns=knowns, wm=wm, nos=nos, center=center)


def _solver(b, **kw):
    s = w.ExpertSolver(b["dim"], b["nk"], b["order"], b["knowns"], b["wm"], **kw)
    s.prepare_hoods(b["x"], b["hoods"], xi=b["xi"])
    return s


def _queries(b, nq, seed, spread=2 ** 14):
    """dyadic query points near the origins, and their models (the nearest origin)"""
    rng = np.random.default_rng(seed)
    n, dim = len(b["nk"]), b["dim"]
    xq = b["xi"][rng.integers(0, n, nq)] + rng.integers(-spread, spread + 1, size=(nq, dim)) / 2.0 ** 24
    _, I = cKDTree(b["xi"]).query(xq, 1)
    return xq, I.astype(np.int64)


def _np(a):
    return a.detach().cpu().numpy() if _lib._is_torch_tensor(a) else np.asarray(a)


def _eq(a, b):
    return np.array_equal(_np(a), _np(b), equal_nan=True)


def _csr_parts(D):
    D = D if isinstance(D, list) else [D]
    if _lib._is_torch_tensor(D[0]):
        return [(_np(d.crow_indices()), _np(d.col_indices()), _np(d.values())) for d in D]
    return [(d.indptr, d.indices, d.data) for d in D]


def _x(b, xq):
    return xq if b["dim"] > 1 else xq[:, 0]


CFGS = [(1, [0], 6), (1, [4], 10), (2, [2], 12), (2, [4], 20), (3, [1], 10), (3, [3], 26), (3, [4], 40),
        (2, [2, 3, 4], 20), (3, [0, 2, 3, 4], 40)]


@pytest.mark.parametrize("knowns_mode", [0, "F", "rand"])
@pytest.mark.parametrize("dim,orders,k", CFGS)
def test_origin_queries_equal_node_rows(dim, orders, k, knowns_mode):
    """queries at model origins, I permuted and repeated: the stencils / operator rows of those models, bit for bit"""
    center = 0 if knowns_mode == 0 else 7
    b = _batch(dim, orders, k, knowns_mode, center=center, hetero_nk=len(orders) > 1, seed=dim * 10 + k)
    s = _solver(b)
    n, maxno = len(b["nk"]), s._maxno
    rng = np.random.default_rng(k)
    I = np.concatenate([rng.permutation(n), rng.integers(0, n, 150)])
    xq = b["xi"][I]
    c = np.vstack([np.eye(maxno)[:33], rng.standard_normal((2, maxno))])
    W, K = s.stencils(c)
    Wq, Kq, I_out = s.interp_stencils(_x(b, xq), c, I)
    assert Wq.shape == (len(c), len(I), s._maxnk) and Kq.shape == (len(c), len(I), maxno)
    assert _eq(Wq, W[:, I]) and _eq(Kq, K[:, I]) and _eq(I_out, I)
    fold = None if knowns_mode == 0 else center
    D, Kd = s.operator(c, center=fold)
    E, Ke, _ = s.interp_operator(_x(b, xq), c, I, center=fold)
    assert _eq(Ke, Kd[:, I])
    for (r0, c0, v0), (r1, c1, v1) in zip(_csr_parts(D), _csr_parts(E)):
        m = ref.opref.sp.csr_array((v0, c0, r0), shape=(n, len(b["x"])))[I]
        assert np.array_equal(m.indptr, r1) and np.array_equal(m.indices, c1) and _eq(m.data, v1)


@pytest.mark.parametrize("knowns_mode", [0, "F", "rand"])
@pytest.mark.parametrize("dim,orders,k", CFGS)
def test_off_node_rows_equal_stencils_of_host_coefficient_rows(dim, orders, k, knowns_mode):
    b = _batch(dim, orders, k, knowns_mode, hetero_nk=len(orders) > 1, seed=dim * 10 + k + 1)
    s = _solver(b)
    n, maxno = len(b["nk"]), s._maxno
    xq, I = _queries(b, 300, seed=k)
    rng = np.random.default_rng(k + 1)
    lap = np.zeros(maxno)
    lap[[sl for sl in range(maxno) if sum(ref.EXPONENTS[dim][sl]) == 2]] = 1.0
    for c in (np.eye(maxno)[[0]], np.eye(maxno)[[min(1, maxno - 1)]], lap[None], rng.standard_normal((3, maxno))):
        if not c.any():
            continue
        Wq, Kq, _ = s.interp_stencils(_x(b, xq), c, I)
        cq = ref.query_rows(dim, c, xq, b["xi"], I, n)           # (nq, nops, maxno)
        per = max(1, 35 // len(c))                                # up to 35 coefficient rows per stencils call
        sample = rng.choice(len(I), 60, replace=False)
        for j0 in range(0, len(sample), per):
            qs = sample[j0:j0 + per]
            Ws, Ks = s.stencils(cq[qs].reshape(-1, maxno))
            for t, q in enumerate(qs):
                rows = slice(t * len(c), (t + 1) * len(c))
                assert _eq(Wq[:, q], Ws[rows, I[q]]), (q, I[q])
                assert _eq(Kq[:, q], Ks[rows, I[q]]), (q, I[q])


def _c_abi_csr(s, xq, I, c, center, bits):
    L = _lib.lib()
    nnz = C.c_int64()
    xq = np.ascontiguousarray(xq)
    I = np.ascontiguousarray(I, np.int64)
    _lib.check(L.wlsqm_solver_interp_operator_nnz(s._handle, I.ctypes.data, len(I), center, C.byref(nnz)))
    it = np.int32 if bits == 32 else np.int64
    rowptr, col = np.zeros(len(I) + 1, it), np.zeros(nnz.value, it)
    values = np.zeros((c.shape[0], nnz.value))
    K = np.zeros((c.shape[0], len(I), s._maxno))
    _lib.check(L.wlsqm_solver_interp_operator_csr(s._handle, xq.ctypes.data, xq.shape[1] if xq.ndim > 1 else 1, I.ctypes.data,
                                                  len(I), c.shape[0], c.ctypes.data, center, bits, rowptr.ctypes.data,
                                                  col.ctypes.data, values.ctypes.data, K.ctypes.data))
    return rowptr, col, values, K


@pytest.mark.parametrize("knowns_mode,center", [(0, None), ("F", 0), ("F", 23), ("rand", 23)])
@pytest.mark.parametrize("dim,orders,k", [(2, [4], 20), (3, [2, 3, 4], 40), (1, [2], 8)])
def test_csr_equals_host_merge(dim, orders, k, knowns_mode, center):
    b = _batch(dim, orders, k, knowns_mode, center=center or 0, hetero_nk=True, seed=7 + k)
    s = _solver(b)
    n, maxno, npoints = len(b["nk"]), s._maxno, len(b["x"])
    xq, I = _queries(b, 500, seed=k)
    I[::37] = I[0]                                                # runs of one model
    c = np.vstack([np.eye(maxno)[:4], np.random.default_rng(k).standard_normal((2, maxno))])
    W, K, _ = s.interp_stencils(_x(b, xq), c, I)
    rp, col, vals, Kf = ref.csr(W, K, b["hoods"], b["nk"], b["knowns"], npoints, I, n, center=center)
    E, Ke, _ = s.interp_operator(_x(b, xq), c, I, center=center)
    assert len(E) == len(c) and Ke.shape == (len(c), len(I), maxno)
    for o in range(len(c)):
        assert E[o].shape == (len(I), npoints) and E[o].indices.dtype == np.int32
        assert np.array_equal(E[o].indptr, rp) and np.array_equal(E[o].indices, col)
        assert _eq(E[o].data, vals[o]), o
    assert _eq(Ke, Kf)
    cen = -1 if center is None else center
    r32 = _c_abi_csr(s, xq, I, c, cen, 32)
    r64 = _c_abi_csr(s, xq, I, c, cen, 64)
    assert r64[0].dtype == np.int64 and np.array_equal(r32[0], r64[0]) and np.array_equal(r32[1], r64[1])
    assert _eq(r32[2], r64[2]) and _eq(r32[3], r64[3]) and _eq(r32[2], vals) and np.array_equal(r32[0], rp)


def _unknown_columns(sens, knowns, nos):
    """sens with the columns of known slots and of slots beyond each case's model set to 0 (the solve leaves them
    unspecified; they are not part of the operator)"""
    maxno = sens.shape[2]
    unk = np.array([[s < no and not (int(kn) >> s) & 1 for s in range(maxno)] for kn, no in zip(knowns, nos)])
    return np.where(unk[:, None, :], sens, 0.0)


def _identity(b, s, c, xq, I):
    """E @ f + K . fi_in against sum_D c[D] interpolate(x, diff=D, I) after solve_hoods(f, fi), within the bound"""
    rng = np.random.default_rng(1)
    n, maxno, maxnk, npoints = len(b["nk"]), s._maxno, s._maxnk, len(b["x"])
    f = rng.standard_normal(npoints)
    fi_in = rng.standard_normal((n, maxno))
    fi_out = fi_in.copy()
    sens = np.zeros((n, maxnk, maxno))
    s.solve_hoods(f, fi_out, sens)
    E, K, _ = s.interp_operator(_x(b, xq), c, I)
    lhs = np.stack([E[o] @ f for o in range(len(E))]) + (K * fi_in[I][None]).sum(-1)
    s.prep_interpolate()
    used = np.flatnonzero(np.abs(c).sum(0))
    interp = {D: s.interpolate(_x(b, xq), diff=int(D), I=I)[0] for D in used}
    rhs = np.stack([sum(c[o, D] * interp[D] for D in used) for o in range(len(c))])
    # |c_q| magnitudes: |coeffs| at |h|
    cq_abs = ref.query_rows(b["dim"], np.abs(c), np.abs(xq - b["xi"][I]), np.zeros_like(b["xi"]), I, n)

    def solve(fi):
        fo = fi.copy()
        s.solve_hoods(np.zeros(npoints), fo, np.zeros((n, maxnk, maxno)))
        return fo
    dfk = ref.opref.known_weights_from_solves(solve, n, maxno, b["nos"], b["knowns"])
    fk = np.where(np.arange(maxnk)[None, :] < b["nk"][:, None], f[np.minimum(b["hoods"][:, :maxnk], npoints - 1)], 0.0)
    bound = ref.identity_bound(np.transpose(cq_abs, (1, 0, 2)), _unknown_columns(sens, b["knowns"], b["nos"])[I], dfk[I],
                               fk[I], fi_in[I], fi_out[I], IDENTITY_CONST)
    ok = np.isfinite(rhs)
    ratio = np.abs(lhs - rhs)[ok] / bound[ok]
    assert (ratio <= 1.0).all(), float(ratio.max())
    print("identity: worst ratio to the bound %.3f" % float(ratio.max()))


@pytest.mark.parametrize("knowns_mode", [0, "rand"])
@pytest.mark.parametrize("dim,orders,k", [(2, [4], 20), (3, [2, 3, 4], 40), (1, [3], 8)])
def test_identity_against_solve_and_interpolate(dim, orders, k, knowns_mode):
    b = _batch(dim, orders, k, knowns_mode, seed=21 + k, hetero_nk=len(orders) > 1)
    s = _solver(b, do_sens=True)
    maxno = s._maxno
    xq, I = _queries(b, 400, seed=3)
    ex = ref.EXPONENTS[dim]
    lap = np.zeros(maxno)
    lap[[sl for sl in range(maxno) if sum(ex[sl]) == 2 and max(ex[sl]) == 2]] = 1.0
    first = np.eye(maxno)[[sl for sl in range(maxno) if sum(ex[sl]) == 1]]
    c = np.vstack([np.eye(maxno)[[0]], first, lap[None], np.random.default_rng(2).standard_normal((3, maxno))])
    _identity(b, s, c, xq, I)


@pytest.mark.parametrize("dim,order,k", [(1, 3, 8), (2, 2, 12), (2, 4, 20), (3, 2, 20)])
def test_polynomial_data_exact_derivatives(dim, order, k):
    from test_interp_operator_reference import _poly
    b = _batch(dim, [order], k, "F", center=4, seed=50 + dim)
    s = _solver(b)
    n, maxno = len(b["nk"]), s._maxno
    no, deriv = _poly(dim, order, seed=dim)
    xq, I = _queries(b, 300, seed=9)
    f = deriv(b["x"], 0)
    E, K, _ = s.interp_operator(_x(b, xq), np.eye(maxno), I, center=4)
    r = np.median(np.linalg.norm(b["x"][b["hoods"][:, 3]] - b["xi"], axis=-1))
    # models whose neighbour list repeats points (the centre three times, say) are ill-conditioned: checked elsewhere
    distinct = np.array([len(np.unique(b["hoods"][i, :b["nk"][i]])) == b["nk"][i] for i in range(n)])
    keep = distinct[I]
    assert keep.sum() > 100
    for D in range(no):
        want = deriv(xq, D)
        got = E[D] @ f                                             # the known F is folded into column center + I[q]
        tol = 1e-10 * max(1.0, np.abs(want).max()) / r ** sum(ref.EXPONENTS[dim][D])
        assert np.abs(got - want)[keep].max() < tol, D


def _export(s, xq, c, I=None, center=None):
    W, K, I1 = s.interp_stencils(xq, c, I)
    E, Ke, I2 = s.interp_operator(xq, c, I, center=center)
    return _np(W), _np(K), _csr_parts(E), _np(Ke), _np(I1), _np(I2)


def _same(a, b):
    W1, K1, D1, Kd1, I1, J1 = a
    W2, K2, D2, Kd2, I2, J2 = b
    assert _eq(W1, W2) and _eq(K1, K2) and _eq(Kd1, Kd2) and _eq(I1, I2) and _eq(J1, J2) and len(D1) == len(D2)
    for (r1, c1, v1), (r2, c2, v2) in zip(D1, D2):
        assert np.array_equal(r1, r2) and np.array_equal(c1, c2) and _eq(v1, v2)


def test_invariances_bitwise():
    b = _batch(2, [2, 3, 4], 20, "rand", center=5, hetero_nk=True, seed=31)
    c = np.random.default_rng(3).standard_normal((4, 15))
    xq, I = _queries(b, 700, seed=4)
    base = _solver(b)
    ref_out = _export(base, xq, c, I, center=5)
    _same(ref_out, _export(base, xq, c, I, center=5))                                   # two calls in a row
    base.prep_interpolate()                                                               # cKDTree: I=None finds I
    _same(ref_out, _export(base, xq, c, None, center=5))
    base.prep_interpolate(search="gpu")                                                   # the device grid too
    _same(ref_out, _export(base, xq, c, None, center=5))
    bt = dict(b, x=b["x"] + 4096.0, xi=b["xi"] + 4096.0)                                  # translation by 2^12
    _same(ref_out, _export(_solver(bt), xq + 4096.0, c, I, center=5))
    _same(ref_out, _export(_solver(b, algorithm=w.ALGO_ITERATIVE, max_iter=3), xq, c, I, center=5))
    guest = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"], host=base)
    guest.prepare(None, None)
    _same(ref_out, _export(guest, xq, c, I, center=5))
    nosol = _solver(b)
    nosol.keep_solution(False)
    _same(ref_out, _export(nosol, xq, c, I, center=5))
    dev = torch.device("cuda", base.device)
    st = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"])
    st.prepare_hoods(torch.as_tensor(b["x"], device=dev), torch.as_tensor(b["hoods"], device=dev),
                     xi=torch.as_tensor(b["xi"], device=dev))
    xt, It = torch.as_tensor(xq, device=dev), torch.as_tensor(I, device=dev)
    _same(ref_out, _export(st, xt, c, It, center=5))                                     # CUDA inputs and outputs
    _same(ref_out, _export(st, xq, c, I, center=5))                                      # numpy queries, CUDA solver
    st.prep_interpolate()
    _same(ref_out, _export(st, xt, c, None, center=5))
    E_t, _, I_t = st.interp_operator(xt, c[0], It)
    assert E_t.layout == torch.sparse_csr and E_t.device == dev and E_t.crow_indices().dtype == torch.int32
    # a permutation of the queries permutes the rows
    p = np.random.default_rng(5).permutation(len(I))
    Wp, Kp, Dp, Kdp, _, _ = _export(base, xq[p], c, I[p], center=5)
    W0, K0, D0, Kd0, _, _ = ref_out
    assert _eq(Wp, W0[:, p]) and _eq(Kp, K0[:, p]) and _eq(Kdp, Kd0[:, p])
    for (r0, c0, v0), (r1, c1, v1) in zip(D0, Dp):
        m = ref.opref.sp.csr_array((v0, c0, r0), shape=(len(p), len(b["x"])))[p]
        assert np.array_equal(m.indptr, r1) and np.array_equal(m.indices, c1) and _eq(m.data, v1)


def test_queries_without_a_model():
    b = _batch(2, [2], 12, "F", center=3, seed=71)
    s = _solver(b)
    n = len(b["nk"])
    xq, I = _queries(b, 40, seed=1)
    I[[2, 5, 9, 30]] = [n, -1, n + 100, 2 ** 40]
    c = np.eye(6)[[0, 3]]
    W, K, _ = s.interp_stencils(xq, c, I)
    E, Ke, _ = s.interp_operator(xq, c, I, center=3)
    bad = np.zeros(len(I), bool)
    bad[[2, 5, 9, 30]] = True
    assert not W[:, bad].any() and np.isnan(K[:, bad]).all() and np.isnan(Ke[:, bad]).all()
    assert np.isfinite(K[:, ~bad]).all()
    for o in range(2):
        rows = np.diff(E[o].indptr)
        assert (rows[bad] == 0).all() and (rows[~bad] > 0).all()
    # NaN query points: the device search reports ncases, the rows are those of a query without a model
    xn = xq.copy()
    xn[[4, 7]] = np.nan
    s.prep_interpolate(search="gpu")
    W2, K2, I2 = s.interp_stencils(xn, c)
    assert (I2[[4, 7]] == n).all() and np.isnan(K2[:, [4, 7]]).all() and not W2[:, [4, 7]].any()
    E2, _, _ = s.interp_operator(xn, c)
    assert (np.diff(E2[0].indptr)[[4, 7]] == 0).all()


def test_errors():
    b = _batch(2, [2], 12, "F", center=3, seed=51)
    s = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"])
    xq, I = _queries(b, 20, seed=2)
    with pytest.raises(RuntimeError):
        s.interp_stencils(xq, 0, I)
    s.prepare_hoods(b["x"], b["hoods"], xi=b["xi"])
    npoints, n = len(b["x"]), len(b["nk"])
    with pytest.raises(RuntimeError):
        s.interp_stencils(xq, 0)                       # no I and no prep_interpolate()
    s.interp_operator(xq, 0, I, center=npoints - n)
    for bad in (npoints - n + 1, -1, -5):
        with pytest.raises(ValueError):
            s.interp_operator(xq, 0, I, center=bad)
    for bad in (6, -1, np.zeros(7), np.zeros((2, 5)), np.zeros((36, 6)), np.full(6, np.nan), np.full(6, np.inf)):
        with pytest.raises(ValueError):
            s.interp_stencils(xq, bad, I)
        with pytest.raises(ValueError):
            s.interp_operator(xq, bad, I)
    with pytest.raises(ValueError):
        s.interp_stencils(xq, 0, I[:-1])
    L = _lib.lib()
    c = np.zeros((36, 6))
    Ic = np.ascontiguousarray(I)
    assert L.wlsqm_solver_interp_stencils(s._handle, xq.ctypes.data, 2, Ic.ctypes.data, len(I), 36, c.ctypes.data,
                                          c.ctypes.data, None) == _lib.E_VALUE
    assert L.wlsqm_solver_interp_stencils(s._handle, xq.ctypes.data, 2, Ic.ctypes.data, len(I), 0, c.ctypes.data,
                                          c.ctypes.data, None) == _lib.E_VALUE
    # nx = 0: rowptr = [0]
    rowptr = np.full(1, 7, np.int32)
    _lib.check(L.wlsqm_solver_interp_operator_csr(s._handle, xq.ctypes.data, 2, Ic.ctypes.data, 0, 1, c.ctypes.data, -1, 32,
                                                  rowptr.ctypes.data, None, None, None))
    assert rowptr[0] == 0
    # a plain prepare() after prepare_hoods(): stencils still, the global operator no longer
    xk = b["x"][np.where(np.arange(12)[None, :] < b["nk"][:, None], b["hoods"], 0)]
    s.prepare(b["xi"], xk)
    s.interp_stencils(xq, 0, I)
    with pytest.raises(RuntimeError):
        s.interp_operator(xq, 0, I)


def test_full_size_cfg2_16m_queries():
    """cfg2 (1M points, 2D order 4, k = 30, F known) with 16M queries of a second cloud: sampled rows against
    stencils(c_q), the identity against solve_hoods + interpolate on every 1000th row"""
    n, k, nq = 1_000_000, 30, 16_000_000
    dev = torch.device("cuda", _lib.default_device())
    g = torch.Generator(device="cpu").manual_seed(0)
    x = (torch.randint(0, 2 ** 24, (n, 2), generator=g) / 2.0 ** 24).double().to(dev)
    xq = (torch.randint(0, 2 ** 24, (nq, 2), generator=g) / 2.0 ** 24).double().to(dev)
    hoods = w.knn_hoods(x, k)
    s = w.ExpertSolver(2, np.full(n, k, np.int32), np.full(n, 4, np.int32), np.ones(n, np.int64),
                       np.full(n, 1, np.int32), do_sens=True)
    s.prepare_hoods(x, hoods)
    s.prep_interpolate()
    lap = np.zeros(15)
    lap[[defs.i2_X2, defs.i2_Y2]] = 1.0
    E, K, I = s.interp_operator(xq, lap)
    assert E.shape == (nq, n) and E.values().numel() == nq * k
    W, K2, I2 = s.interp_stencils(xq, lap, I)
    assert bool((K == K2).all()) and bool((I == I2).all())
    rng = np.random.default_rng(0)
    sample = rng.choice(nq, 35, replace=False)
    xs, Is = _np(xq[sample]), _np(I[sample])
    cq = ref.query_rows(2, lap, xs, _np(x[torch.as_tensor(Is, device=dev)]), np.arange(35), 35)
    Ws, Ks = s.stencils(cq[:, 0])
    for t in range(35):
        assert _eq(W[sample[t]], Ws[t, Is[t]]) and _eq(K[sample[t]], Ks[t, Is[t]])
    # identity on every 1000th row
    sens = torch.empty((n, k, 15), dtype=torch.float64, device=dev)
    d1 = torch.zeros((n, 15), dtype=torch.float64, device=dev)
    d1[:, 0] = 1.0
    s.solve_hoods(torch.zeros(n, dtype=torch.float64, device=dev), d1, sens)     # d fi / d fi_known[F]
    f = torch.sin(3 * x[:, 0]) * torch.cos(2 * x[:, 1])
    fi_in = torch.zeros((n, 15), dtype=torch.float64, device=dev)
    fi_in[:, 0] = f
    fi_out = fi_in.clone()
    s.solve_hoods(f, fi_out, sens)
    rows = torch.arange(0, nq, 1000, device=dev)
    Ir = I[rows]
    lhs = (E @ f)[rows] + (K[rows] * fi_in[Ir]).sum(-1)
    rhs = s.interpolate(xq[rows], diff=defs.i2_X2, I=Ir)[0] + s.interpolate(xq[rows], diff=defs.i2_Y2, I=Ir)[0]
    Ih = _np(Ir)
    cq_abs = ref.query_rows(2, lap, np.abs(_np(xq[rows]) - _np(x)[Ih]), np.zeros((len(Ih), 2)), np.arange(len(Ih)), len(Ih))
    dfk = np.zeros((len(Ih), 15, 15))
    dfk[:, 0, :] = _np(d1[Ir])
    sens_q = _np(sens[Ir])
    sens_q[:, :, 0] = 0.0                                           # F is known
    bound = ref.identity_bound(np.transpose(cq_abs, (1, 0, 2)), sens_q, dfk, _np(f[hoods[Ir].long()]),
                               _np(fi_in[Ir]), _np(fi_out[Ir]), IDENTITY_CONST)[0]
    ratio = np.abs(_np(lhs) - _np(rhs)) / bound
    assert (ratio <= 1.0).all(), float(ratio.max())
    print("16M queries: identity on %d rows, worst ratio to the bound %.3f" % (len(Ih), float(ratio.max())))
    torch.cuda.synchronize()
