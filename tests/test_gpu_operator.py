"""GPU tests of the operator export: ExpertSolver.stencils / .operator (csrc/wlsqm_operator.cu).

Exact checks use one-hot coefficients, where every product is exact: W must equal the solver's own `sens` bit for bit,
K the result of a solve with fk = 0 and a unit known value, and the CSR values the host merge of the same entries
(tests/operator_reference.py).  General coefficients are held to the identity bound fixed on the oracle in
tests/test_operator_reference.py.  Clouds are dyadic (multiples of 2^-24), so that a 2^12 translation is exact.
"""
import ctypes as C

import numpy as np
import pytest
from scipy.spatial import cKDTree

import wlsqm_b200 as w
from wlsqm_b200 import _lib
from wlsqm_b200.fitter import defs
import operator_reference as ref
from test_operator_reference import IDENTITY_CONST

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


def _sens_and_dfk(b, s):
    """sens from solve_hoods and d fi / d fi_known from solves with fk = 0 (the GPU's own operator)"""
    n, maxnk, maxno = len(b["nk"]), s._maxnk, s._maxno
    sens = np.zeros((n, maxnk, maxno))
    s.solve_hoods(np.zeros(len(b["x"])), np.zeros((n, maxno)), sens)

    def solve(fi_in):
        fi = fi_in.copy()
        s.solve_hoods(np.zeros(len(b["x"])), fi, np.zeros((n, maxnk, maxno)))
        return fi
    return sens, ref.known_weights_from_solves(solve, n, maxno, b["nos"], b["knowns"])


def _eq(a, b):
    return np.array_equal(np.asarray(a), np.asarray(b), equal_nan=True)


CFGS = [(1, [0], 6), (1, [4], 10), (2, [2], 12), (2, [4], 20), (3, [1], 10), (3, [3], 26), (3, [4], 40),
        (2, [2, 3, 4], 20), (3, [0, 2, 3, 4], 40)]


@pytest.mark.parametrize("knowns_mode", [0, "F", "rand"])
@pytest.mark.parametrize("dim,orders,k", CFGS)
def test_stencils_equal_sens_and_known_solves(dim, orders, k, knowns_mode):
    b = _batch(dim, orders, k, knowns_mode, hetero_nk=len(orders) > 1, seed=dim * 10 + k)
    s = _solver(b, do_sens=True)
    sens, dfk = _sens_and_dfk(b, s)
    n, maxno = len(b["nk"]), s._maxno
    singular = 0
    for slot in range(maxno):
        W, K = s.stencils(slot)
        assert W.shape == (n, s._maxnk) and K.shape == (n, maxno)
        for i in range(n):
            nk, no, kn = b["nk"][i], b["nos"][i], int(b["knowns"][i])
            assert not W[i, nk:].any()
            if slot >= no:
                assert not W[i].any() and not K[i].any()
            elif (kn >> slot) & 1:
                assert not W[i].any()
                assert _eq(K[i], np.eye(maxno)[slot])
            else:
                assert _eq(W[i, :nk], sens[i, :nk, slot]), (slot, i)
                row = dfk[i, :, slot]
                if not np.isfinite(sens[i, :nk, slot]).all():
                    singular += 1
                    continue
                assert _eq(K[i], row), (slot, i)
    print("dim %d orders %s knowns %s: %d singular (case, slot) pairs excluded from the K check" % (dim, orders, knowns_mode, singular))


def test_zero_coefficients_are_skipped():
    """singular cases (every neighbour the same point) have non-finite blocks: a zero coefficient must not pull
    them into an operator -- the weights of a known slot stay exactly 0, those of a slot nobody uses too"""
    b = _batch(2, [2], 12, "F", seed=61)
    b["hoods"][::10, :] = b["hoods"][::10, :1]
    s = _solver(b, do_sens=True)
    sens, _ = _sens_and_dfk(b, s)
    bad = ~np.isfinite(sens[:, :, 1:]).all(axis=(1, 2))
    assert bad.sum() >= 10, bad.sum()
    W, K = s.stencils(0)                                 # F is known everywhere
    assert not W.any() and _eq(K, np.tile(np.eye(6)[0], (len(b["nk"]), 1)))
    D, Kd = s.operator(0)
    assert not D.data.any() and _eq(Kd, K)
    W, K = s.stencils(np.eye(6)[[1, 2]])
    assert _eq(W[0][~bad], sens[~bad, :, 1]) and not np.isfinite(W[0][bad]).all()


def _c_abi_csr(s, c, center, bits):
    L = _lib.lib()
    nnz = C.c_int64()
    _lib.check(L.wlsqm_solver_operator_nnz(s._handle, center, C.byref(nnz)))
    it = np.int32 if bits == 32 else np.int64
    n = s.ncases
    rowptr, col = np.zeros(n + 1, it), np.zeros(nnz.value, it)
    values = np.zeros((c.shape[0], nnz.value))
    K = np.zeros((c.shape[0], n, s._maxno))
    _lib.check(L.wlsqm_solver_operator_csr(s._handle, c.shape[0], c.ctypes.data, center, bits, rowptr.ctypes.data,
                                           col.ctypes.data, values.ctypes.data, K.ctypes.data))
    return rowptr, col, values, K


@pytest.mark.parametrize("knowns_mode,center", [(0, None), ("F", 0), ("F", 23), ("rand", 23)])
@pytest.mark.parametrize("dim,orders,k", [(2, [4], 20), (3, [2, 3, 4], 40), (1, [2], 8)])
def test_csr_equals_host_merge_of_sens(dim, orders, k, knowns_mode, center):
    b = _batch(dim, orders, k, knowns_mode, center=center or 0, hetero_nk=True, seed=7 + k)
    s = _solver(b, do_sens=True)
    sens, dfk = _sens_and_dfk(b, s)
    n, maxno, npoints = len(b["nk"]), s._maxno, len(b["x"])
    c = np.eye(maxno)
    Wr, Kr = ref.stencils(sens, dfk, b["nk"], b["nos"], b["knowns"], c)
    rp, col, vals, Kf = ref.csr(Wr, Kr, b["hoods"], b["nk"], b["knowns"], npoints, center=center)
    D, K = s.operator(c, center=center)
    assert len(D) == maxno and K.shape == (maxno, n, maxno)
    for o in range(maxno):
        assert D[o].shape == (n, npoints) and D[o].indices.dtype == np.int32
        assert np.array_equal(D[o].indptr, rp) and np.array_equal(D[o].indices, col)
        assert np.shares_memory(D[o].indices, D[0].indices)
        assert _eq(D[o].data, vals[o]), o
    assert _eq(K, Kf)
    # canonical scipy CSR of the used hood entries (+ the folded diagonal)
    rows = np.repeat(np.arange(n), b["nk"])
    cols = np.concatenate([b["hoods"][i, :b["nk"][i]] for i in range(n)])
    if center is not None:
        f = (b["knowns"] & 1).astype(bool)
        rows, cols = np.concatenate([rows, np.arange(n)[f]]), np.concatenate([cols, center + np.arange(n)[f]])
    canon = ref.sp.csr_array((np.ones(len(rows)), (rows, cols)), shape=(n, npoints))
    canon.sum_duplicates()
    canon.sort_indices()
    assert np.array_equal(canon.indptr, rp) and np.array_equal(canon.indices, col)
    # 64-bit indices through the C ABI: the same matrix
    r32 = _c_abi_csr(s, c, -1 if center is None else center, 32)
    r64 = _c_abi_csr(s, c, -1 if center is None else center, 64)
    assert r64[0].dtype == np.int64 and np.array_equal(r32[0], r64[0]) and np.array_equal(r32[1], r64[1])
    assert _eq(r32[2], r64[2]) and _eq(r32[3], r64[3]) and _eq(r32[2], vals)
    _duplicates_carry_equal_weights(b, sens)


def _duplicates_carry_equal_weights(b, sens):
    """every repeat of a neighbour index carries bitwise the weights of its first occurrence (the same point enters the
    fit the same way), so the order in which repeats are merged cannot change a value"""
    for i in range(len(b["nk"])):
        h = b["hoods"][i, :b["nk"][i]]
        for k in range(len(h)):
            f = int(np.argmax(h == h[k]))
            assert _eq(sens[i, k], sens[i, f]), (i, k, f)


@pytest.mark.parametrize("k", [1000, 6000])
def test_csr_large_neighbourhoods(k):
    """max nk beyond the default 48 KB of dynamic shared memory per CTA (1000) and beyond eight staged rows per CTA
    (6000): the CSR against the host merge, with duplicates and folding"""
    b = _batch(2, [1], k, "F", n=24, center=5, extra=k + 50, seed=k)
    s = _solver(b, do_sens=True)
    sens, dfk = _sens_and_dfk(b, s)
    n, npoints = len(b["nk"]), len(b["x"])
    c = np.eye(3)
    Wr, Kr = ref.stencils(sens, dfk, b["nk"], b["nos"], b["knowns"], c)
    rp, col, vals, Kf = ref.csr(Wr, Kr, b["hoods"], b["nk"], b["knowns"], npoints, center=5)
    D, K = s.operator(c, center=5)
    for o in range(3):
        assert np.array_equal(D[o].indptr, rp) and np.array_equal(D[o].indices, col)
        assert _eq(D[o].data, vals[o]), o
    assert _eq(K, Kf)
    _duplicates_carry_equal_weights(b, sens)


def _identity_check(b, s, c):
    rng = np.random.default_rng(1)
    n, maxno, npoints = len(b["nk"]), s._maxno, len(b["x"])
    f = rng.standard_normal(npoints)
    fi_in = rng.standard_normal((n, maxno))
    fi_out = fi_in.copy()
    s.solve_hoods(f, fi_out)
    D, K = s.operator(c)
    W, K2 = s.stencils(c)
    assert _eq(K, K2)
    fk = np.where(np.arange(s._maxnk)[None, :] < b["nk"][:, None], f[np.minimum(b["hoods"], npoints - 1)], 0.0)
    rhs = (fi_out[None] * c[:, None, :]).sum(-1)
    lhs = np.stack([D[o] @ f for o in range(len(D))]) + (K * fi_in[None]).sum(-1)
    bound = ref.identity_bound(W, K, c, fk[None], fi_in[None], fi_out, IDENTITY_CONST)
    ok = np.isfinite(rhs)
    assert (np.abs(lhs - rhs)[ok] <= bound[ok]).all(), float((np.abs(lhs - rhs)[ok] / bound[ok]).max())
    print("identity: worst ratio to the bound %.3f" % float((np.abs(lhs - rhs)[ok] / bound[ok]).max()))


@pytest.mark.parametrize("knowns_mode", [0, "rand"])
def test_identity_laplacian_gradient_dense(knowns_mode):
    b = _batch(2, [4], 20, knowns_mode, seed=21)
    s = _solver(b)
    lap = np.zeros((1, 15))
    lap[0, [defs.i2_X2, defs.i2_Y2]] = 1.0
    grad = np.zeros((2, 15))
    grad[0, defs.i2_X] = grad[1, defs.i2_Y] = 1.0
    _identity_check(b, s, lap)
    _identity_check(b, s, grad)
    b3 = _batch(3, [4], 40, knowns_mode, seed=22)
    s3 = _solver(b3)
    _identity_check(b3, s3, np.random.default_rng(2).standard_normal((35, 35)))


def _export(s, c, center=None):
    W, K = s.stencils(c)
    D, Kd = s.operator(c, center=center)
    D = D if isinstance(D, list) else [D]
    if _lib._is_torch_tensor(W):
        W, K, Kd = W.cpu().numpy(), K.cpu().numpy(), Kd.cpu().numpy()
        D = [(d.crow_indices().cpu().numpy(), d.col_indices().cpu().numpy(), d.values().cpu().numpy()) for d in D]
    else:
        D = [(d.indptr, d.indices, d.data) for d in D]
    return W, K, D, Kd


def _same(a, b):
    W1, K1, D1, Kd1 = a
    W2, K2, D2, Kd2 = b
    assert _eq(W1, W2) and _eq(K1, K2) and _eq(Kd1, Kd2) and len(D1) == len(D2)
    for (r1, c1, v1), (r2, c2, v2) in zip(D1, D2):
        assert np.array_equal(r1, r2) and np.array_equal(c1, c2) and _eq(v1, v2)


def test_invariances_bitwise():
    b = _batch(2, [2, 3, 4], 20, "rand", center=5, hetero_nk=True, seed=31)
    c = np.random.default_rng(3).standard_normal((4, 15))
    base = _solver(b)
    ref_out = _export(base, c, center=5)
    _same(ref_out, _export(base, c, center=5))                                   # two calls in a row
    bt = dict(b, x=b["x"] + 4096.0, xi=b["xi"] + 4096.0)                         # translation by 2^12
    _same(ref_out, _export(_solver(bt), c, center=5))
    _same(ref_out, _export(_solver(b, algorithm=w.ALGO_ITERATIVE, max_iter=3), c, center=5))
    guest = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"], host=base)
    guest.prepare(None, None)
    _same(ref_out, _export(guest, c, center=5))
    dev = torch.device("cuda", base.device)
    st = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"])
    st.prepare_hoods(torch.as_tensor(b["x"], device=dev), torch.as_tensor(b["hoods"], device=dev),
                     xi=torch.as_tensor(b["xi"], device=dev))
    out_t = _export(st, c, center=5)
    _same(ref_out, out_t)
    D_t, _ = st.operator(c[0])
    assert D_t.layout == torch.sparse_csr and D_t.device == dev and D_t.crow_indices().dtype == torch.int32
    # a permutation of the cases permutes the rows
    p = np.random.default_rng(4).permutation(len(b["nk"]))
    bp = dict(b, hoods=b["hoods"][p], nk=b["nk"][p], order=b["order"][p], knowns=b["knowns"][p], wm=b["wm"][p],
              nos=b["nos"][p], xi=b["xi"][p])
    Wp, Kp, Dp, Kdp = _export(_solver(bp), c)
    W0, K0, D0, Kd0 = _export(base, c)
    assert _eq(Wp, W0[:, p]) and _eq(Kp, K0[:, p]) and _eq(Kdp, Kd0[:, p])
    for (r0, c0, v0), (r1, c1, v1) in zip(D0, Dp):
        m = ref.sp.csr_array((v0, c0, r0), shape=(len(p), len(b["x"])))[p]
        assert np.array_equal(m.indptr, r1) and np.array_equal(m.indices, c1) and _eq(m.data, v1)


@pytest.mark.parametrize("fold", [False, True])
def test_sharded_ranks_stack_to_the_unsharded_operator(fold):
    from wlsqm_b200.parallel import ShardedExpertSolver
    b = _batch(2, [2, 4], 20, "F", center=0, hetero_nk=True, seed=41)
    c = np.random.default_rng(5).standard_normal((3, 15))
    whole = _solver(b)
    D, K = whole.operator(c, center=0 if fold else None)
    blocks, Ks = [], []
    for r in range(2):
        sh = ShardedExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"], rank=r, world=2)
        sh.prepare_hoods(b["x"], b["hoods"])
        Dr, Kr = sh.operator(c, fold_center=fold)
        blocks.append(Dr)
        Ks.append(Kr)
    assert _eq(np.concatenate(Ks, axis=1), K)
    for o in range(3):
        st = ref.sp.vstack([blocks[0][o], blocks[1][o]], format="csr")
        assert np.array_equal(st.indptr, D[o].indptr) and np.array_equal(st.indices, D[o].indices)
        assert _eq(st.data, D[o].data)


def test_errors():
    b = _batch(2, [2], 12, "F", center=3, seed=51)
    s = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"])
    with pytest.raises(RuntimeError):
        s.stencils(0)
    with pytest.raises(RuntimeError):
        s.operator(0)
    s.prepare_hoods(b["x"], b["hoods"], xi=b["xi"])
    npoints, n = len(b["x"]), len(b["nk"])
    s.operator(0, center=npoints - n)
    for bad in (npoints - n + 1, -1, -5):
        with pytest.raises(ValueError):
            s.operator(0, center=bad)
    for bad in (6, -1, np.zeros(7), np.zeros((2, 5)), np.zeros((36, 6)), np.zeros((1, 1, 6)), np.full(6, np.nan)):
        with pytest.raises(ValueError):
            s.stencils(bad)
        with pytest.raises(ValueError):
            s.operator(bad)
    L = _lib.lib()
    c = np.zeros((36, 6))
    assert L.wlsqm_solver_stencils(s._handle, 36, c.ctypes.data, c.ctypes.data, None) == _lib.E_VALUE
    assert L.wlsqm_solver_operator_csr(s._handle, 1, c.ctypes.data, -1, 16, c.ctypes.data, c.ctypes.data,
                                       c.ctypes.data, None) == _lib.E_VALUE
    # a plain prepare() after prepare_hoods(): the neighbour lists no longer belong to the operators
    xk = b["x"][np.where(np.arange(12)[None, :] < b["nk"][:, None], b["hoods"], 0)]
    s.prepare(b["xi"], xk)
    s.stencils(0)
    with pytest.raises(RuntimeError):
        s.operator(0)
    # a failed prepare_hoods() (an index outside x) leaves no operator behind either
    s.prepare_hoods(b["x"], b["hoods"], xi=b["xi"])
    bad_hoods = b["hoods"].copy()
    bad_hoods[7, 0] = npoints
    with pytest.raises(ValueError):
        s.prepare_hoods(b["x"], bad_hoods, xi=b["xi"])
    with pytest.raises(RuntimeError):
        s.operator(0)


def test_empty_batch_through_the_abi():
    """a solver over no cases: prepare_hoods succeeds and the global operator is the empty (0, npoints) matrix"""
    L = _lib.lib()
    z32, z64 = np.zeros(1, np.int32), np.zeros(1, np.int64)
    h = C.c_void_p()
    _lib.check(L.wlsqm_solver_create(2, 0, z32.ctypes.data, z32.ctypes.data, z64.ctypes.data, z32.ctypes.data, 1, 0, 10,
                                     0, _lib.default_device(), C.byref(h)))
    try:
        x = np.zeros((5, 2))
        _lib.check(L.wlsqm_solver_prepare_hoods(h, x.ctypes.data, 2, 5, z32.ctypes.data, 1, None, 0))
        nnz = C.c_int64(-1)
        _lib.check(L.wlsqm_solver_operator_nnz(h, 0, C.byref(nnz)))
        assert nnz.value == 0
        rowptr = np.full(1, 7, np.int32)
        c = np.ones((1, 1))
        _lib.check(L.wlsqm_solver_operator_csr(h, 1, c.ctypes.data, -1, 32, rowptr.ctypes.data, None, None, None))
        assert rowptr[0] == 0
    finally:
        L.wlsqm_solver_destroy(h)


def test_full_size_cfg2_one_slot():
    n, k = 1_000_000, 30
    dev = torch.device("cuda", _lib.default_device())
    g = torch.Generator(device="cpu").manual_seed(0)
    x = (torch.randint(0, 2 ** 24, (n, 2), generator=g) / 2.0 ** 24).double().to(dev)
    hoods = w.knn_hoods(x, k)
    ones = np.ones(n)
    s = w.ExpertSolver(2, np.full(n, k, np.int32), np.full(n, 4, np.int32), np.zeros(n, np.int64),
                       np.full(n, 1, np.int32), do_sens=True)
    s.prepare_hoods(x, hoods)
    sens = torch.empty((n, k, 15), dtype=torch.float64, device=dev)
    fi = torch.zeros((n, 15), dtype=torch.float64, device=dev)
    s.solve_hoods(torch.as_tensor(ones, device=dev), fi, sens)
    W, K = s.stencils(defs.i2_X2)
    a, bb = W, sens[:, :, defs.i2_X2]
    assert bool(((a == bb) | (torch.isnan(a) & torch.isnan(bb))).all())
    D, _ = s.operator(defs.i2_X2)
    assert D.values().numel() == n * k           # kNN lists hold distinct indices
    torch.cuda.synchronize()
