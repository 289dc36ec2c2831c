"""GPU tests of the device-side fixed-radius search (PointGrid.ball, query_ball_point, ball_hoods), compared entry for
entry with scipy.spatial.cKDTree.query_ball_point -- the search the reference's callers use to build radius
neighbourhoods (examples/wlsqm_example.py:100-132).  The set of points within r is unique, so every comparison is
exact; random clouds are first checked to have no pair within a relative 1e-12 of its sphere."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

pytestmark = pytest.mark.gpu

wlsqm = pytest.importorskip("wlsqm_b200")


def _cloud(n, dim, kind, seed=0):
    rng = np.random.default_rng(seed)
    if kind == "uniform":
        x = rng.random((n, dim))
    elif kind == "clustered":
        c = rng.random((20, dim))
        x = c[rng.integers(0, 20, n)] + 0.01 * rng.standard_normal((n, dim))
    else:
        x = rng.random((n, dim)) * np.array([100.0, 1.0, 0.01])[:dim]
    return x[:, 0].copy() if dim == 1 else x


def _d2(x, q):
    """the membership distance of include/wlsqm_b200.h: per-axis rounded squares summed in axis order"""
    dd = np.asarray(x, np.float64) - np.asarray(q, np.float64)
    d2 = dd[..., 0] * dd[..., 0]
    for d in range(1, dd.shape[-1]):
        d2 = d2 + dd[..., d] * dd[..., d]
    return d2


def _rows(rowptr, col):
    rowptr, col = np.asarray(rowptr), np.asarray(col)
    return [col[rowptr[i]:rowptr[i + 1]].tolist() for i in range(len(rowptr) - 1)]


def _assert_clear_of_sphere(x2, q2, r):
    """no pair lies within a relative 1e-12 of its sphere, so cKDTree's arithmetic and ours agree on membership"""
    r = np.broadcast_to(np.asarray(r, np.float64), (len(q2),))
    near = cKDTree(x2).query_ball_point(q2, r * (1 + 1e-9))
    for i, lst in enumerate(near):
        d2 = _d2(x2[lst], q2[i])
        assert not np.any(np.abs(d2 - r[i] ** 2) <= 1e-12 * r[i] ** 2), "a pair lies on its sphere: pick another seed"


@pytest.mark.parametrize("dim,kind,n,mean", [(1, "uniform", 20000, 12), (1, "clustered", 5000, 20), (2, "uniform", 20000, 30),
                                             (2, "clustered", 20000, 25), (2, "anisotropic", 10000, 30),
                                             (3, "uniform", 8000, 60), (3, "anisotropic", 8000, 20),
                                             (3, "clustered", 8000, 40)])
@pytest.mark.parametrize("per_point", [False, True])
def test_self_queries_match_ckdtree(dim, kind, n, mean, per_point):
    x = _cloud(n, dim, kind)
    x2 = x.reshape(n, -1)
    tree = cKDTree(x2)
    r0 = float(np.median(tree.query(x2[:2000], mean + 1)[0][:, -1]))
    r = r0 * (0.7 + 0.6 * np.random.default_rng(5).random(n)) if per_point else r0
    _assert_clear_of_sphere(x2, x2, r)
    ref = tree.query_ball_point(x2, r)
    g = wlsqm.PointGrid(x)
    rowptr, col = g.ball(r, exclude_self=False)
    assert rowptr.dtype == np.int64 and col.dtype == np.int32 and rowptr.shape == (n + 1,)
    assert _rows(rowptr, col) == [sorted(l) for l in ref]
    rowptr, col = g.ball(r)                       # exclude_self defaults to True for the grid's own points
    assert _rows(rowptr, col) == [[j for j in sorted(l) if j != i] for i, l in enumerate(ref)]


@pytest.mark.parametrize("dim", [1, 2, 3])
def test_dyadic_lattice_exact_boundaries(dim):
    """members on cell edges and at exactly r are included, as cKDTree includes them"""
    m = {1: 64, 2: 24, 3: 10}[dim]
    ax = np.arange(m) * 0.25
    x = np.stack(np.meshgrid(*([ax] * dim), indexing="ij"), -1).reshape(-1, dim)
    n = len(x)
    g = wlsqm.PointGrid(x[:, 0].copy() if dim == 1 else x)
    h = g.info()[1]
    rng = np.random.default_rng(1)
    # dyadic queries (lattice points and midpoints, exact arithmetic everywhere: cKDTree is the oracle) and queries on
    # the cell edges and corners of the search grid (the numpy restatement of the rule is the oracle)
    xq = rng.choice(np.concatenate([ax, ax + 0.125]), (2000, dim))
    edges = np.floor(ax / h) * h
    xe = rng.choice(np.concatenate([edges, edges + h, ax]), (2000, dim))
    tree = cKDTree(x)
    for r in (0.25, 0.5, 0.75, 1.0):
        ref = tree.query_ball_point(xq, r)
        rowptr, col = g.ball(r, xq[:, 0].copy() if dim == 1 else xq)
        got = _rows(rowptr, col)
        assert got == [sorted(l) for l in ref]
        # members at exactly r
        assert sum(int(np.any(_d2(x[l], xq[i]) == r * r)) for i, l in enumerate(ref[:200])) > 0
        rowptr, col = g.ball(r, xe[:, 0].copy() if dim == 1 else xe)
        got = _rows(rowptr, col)
        d2 = _d2(x[None, :, :], xe[:, None, :])
        assert got == [np.nonzero(row <= r * r)[0].tolist() for row in d2]
    rowptr, col = g.ball(0.5)
    self_ref = tree.query_ball_point(x, 0.5)
    assert _rows(rowptr, col) == [[j for j in sorted(l) if j != i] for i, l in enumerate(self_ref)]


@pytest.mark.parametrize("dim", [2, 3])
def test_arbitrary_queries_nan_and_outside(dim):
    n, nq = 15000, 5000
    x = _cloud(n, dim, "uniform", 2)
    x[7] = np.nan
    x[11, 0] = np.inf
    rng = np.random.default_rng(3)
    xq = rng.random((nq, dim)) * 1.4 - 0.2             # many queries outside the bounding box
    r = 0.03 if dim == 2 else 0.08
    ok = np.isfinite(x).all(1)
    xf = x[ok]
    _assert_clear_of_sphere(xf, xq, r)
    idx = np.nonzero(ok)[0]
    ref = [sorted(idx[l].tolist()) for l in cKDTree(xf).query_ball_point(xq, r)]
    g = wlsqm.PointGrid(x)
    xq[5] = np.nan
    xq[6, 1] = np.nan
    ref[5] = ref[6] = []
    rowptr, col = g.ball(r, xq)
    got = _rows(rowptr, col)
    assert got == ref
    assert 7 not in col and 11 not in col
    # r = inf: every finite point, never the NaN / inf ones
    rowptr, col = g.ball(np.inf, xq[:3])
    assert _rows(rowptr, col)[0] == idx.tolist()
    # query_ball_point twin, including the point itself
    assert g.query_ball_point(xq[:50], r).tolist() == [sorted(l) for l in ref[:50]]
    assert g.query_ball_point(xq[0], r) == ref[0]


@pytest.mark.parametrize("dim", [1, 2, 3])
def test_distance_order(dim):
    n = 6000
    x = _cloud(n, dim, "uniform", 4)
    x2 = x.reshape(n, -1)
    r = {1: 3e-3, 2: 0.03, 3: 0.09}[dim]
    g = wlsqm.PointGrid(x)
    rowptr, col = g.ball(r, order="distance", exclude_self=False)
    ri, ci = g.ball(r, exclude_self=False)
    assert np.array_equal(rowptr, ri)
    for i in range(0, n, 7):
        lst = np.asarray(ci[ri[i]:ri[i + 1]])
        d2 = _d2(x2[lst], x2[i])
        assert np.array_equal(col[rowptr[i]:rowptr[i + 1]], lst[np.lexsort((lst, d2))])


@pytest.mark.parametrize("dim,max_k", [(2, 10), (2, 30), (3, 60), (1, 8), (3, 128)])
def test_max_k(dim, max_k):
    n = 5000
    x = _cloud(n, dim, "uniform", 6)
    x2 = x.reshape(n, -1)
    r = {1: 2e-3, 2: 0.04, 3: 0.12}[dim]
    g = wlsqm.PointGrid(x)
    rp, cd = g.ball(r, order="distance")
    full = _rows(rp, cd)
    for order in ("distance", "index"):
        rowptr, col = g.ball(r, max_k=max_k, order=order)
        got = _rows(rowptr, col)
        want = [l[:max_k] for l in full]
        assert got == (want if order == "distance" else [sorted(l) for l in want])
    assert any(len(l) > max_k for l in full) or max_k >= 60
    # r = inf: the k nearest neighbours.  knn may fuse d2 into FMAs, so the rows agree where the distances of every
    # compared row, up to the (k+1)-th neighbour, are distinct beyond rounding -- asserted for all n rows.
    kk = min(max_k, 100)
    rowptr, col = g.ball(np.inf, max_k=kk, order="distance")
    nb = cKDTree(x2).query(x2, kk + 2)[1]
    dref = np.sort(_d2(x2[nb], x2[:, None, :]), axis=1)[:, 1:kk + 2]
    assert (np.diff(dref, axis=1) > 1e-12 * dref[:, 1:]).all()
    assert np.array_equal(np.asarray(col).reshape(n, kk), g.knn(kk))


@pytest.mark.parametrize("dim", [2, 3])
def test_capped_walk_far_from_origin(dim):
    """The capped walk ends on the same cell box as the uncapped one: far from the origin (coordinates about 1e3,
    radii about 1e-3, cell edges rounded at ulp(1e3)) it misses no member, on a dyadic lattice with members on cell
    edges and at exactly r and on a random cloud."""
    m = {2: 40, 3: 14}[dim]
    ax = 1024.0 + np.arange(m) * 2.0 ** -12
    lat = np.stack(np.meshgrid(*([ax] * dim), indexing="ij"), -1).reshape(-1, dim)
    rnd = 1000.0 + np.random.default_rng(40).random((8000, dim)) * 0.02
    for x, radii in ((lat, [2.0 ** -12, 2.0 ** -11, 3 * 2.0 ** -12]), (rnd, {2: [5e-4, 1e-3], 3: [1e-3, 2e-3]}[dim])):
        g = wlsqm.PointGrid(x)
        for r in radii:
            rp, cd = g.ball(r, order="distance", exclude_self=False)
            rows = _rows(rp, cd)
            assert max(len(l) for l in rows) <= 128
            for i in range(0, len(x), 37):
                assert sorted(rows[i]) == np.nonzero(_d2(x, x[i]) <= r * r)[0].tolist()
            rpk, cdk = g.ball(r, order="distance", exclude_self=False, max_k=128)
            assert _rows(rpk, cdk) == rows
            if x is lat:
                assert any(np.any(_d2(x[l], x[i]) == r * r) for i, l in enumerate(rows[:50]))


def test_counts_shapes_and_duplicates():
    rng = np.random.default_rng(9)
    x = rng.random((3000, 2))
    x[100:110] = x[5]                                   # duplicates of point 5
    g = wlsqm.PointGrid(x)
    tree = cKDTree(x)
    xq = rng.random((400, 2))
    r = 0.05
    cnt = g.query_ball_point(xq, r, return_length=True)
    assert np.array_equal(cnt, tree.query_ball_point(xq, r, return_length=True))
    rowptr, col = g.ball(r, xq)
    assert rowptr[0] == 0 and np.array_equal(np.diff(rowptr), cnt) and rowptr[-1] == col.shape[0]
    # r = 0: only coincident points, never the point itself
    rowptr, col = g.ball(0.0)
    assert _rows(rowptr, col)[5] == list(range(100, 110))
    assert _rows(rowptr, col)[100] == [5] + list(range(101, 110))
    assert rowptr[-1] == 110 and rowptr[200] - rowptr[199] == 0
    x2 = rng.random((500, 2))
    rowptr, col = wlsqm.PointGrid(x2).ball(0.0)
    assert rowptr.shape == (501,) and (rowptr == 0).all() and col.shape == (0,)
    rowptr, col = g.ball(r, np.zeros((0, 2)))
    assert rowptr.shape == (1,) and rowptr[0] == 0 and col.shape == (0,)
    h, nk = wlsqm.ball_hoods(x2, 0.0)
    assert h.shape == (500, 1) and (h == 500).all() and (nk == 0).all()


def test_cuda_tensors_and_side_stream():
    torch = pytest.importorskip("torch")
    n = 40000
    x = _cloud(n, 2, "uniform", 12)
    r = 0.012
    ref = cKDTree(x).query_ball_point(x, r)
    xt = torch.from_numpy(x).cuda()
    g = wlsqm.PointGrid(xt)
    rowptr, col = g.ball(r)
    assert rowptr.is_cuda and col.is_cuda and rowptr.dtype == torch.int64 and col.dtype == torch.int32
    assert _rows(rowptr.cpu(), col.cpu()) == [[j for j in sorted(l) if j != i] for i, l in enumerate(ref)]
    # per-query radii on the device (also as a 0-d tensor for one radius)
    rq_d = torch.full((n,), r, dtype=torch.float64, device="cuda")
    assert torch.equal(g.ball(rq_d)[1], col) and torch.equal(g.ball(torch.tensor(r, dtype=torch.float64, device="cuda"))[1], col)
    # queries produced late on a side stream: the search must order itself after them (host radii: no host sync
    # before the search is launched)
    side = torch.cuda.Stream()
    rng = np.random.default_rng(13)
    xq_h = rng.random((20000, 2))
    rq_h = 0.005 + 0.01 * rng.random(20000)
    src = torch.from_numpy(xq_h).cuda()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(20_000_000)                   # the copies below run late on the side stream
        xq = src * 1.0
        rowptr, col = g.ball(rq_h, xq)
        hoods, nk = wlsqm.ball_hoods(xt, r)
    torch.cuda.synchronize()
    refq = cKDTree(x).query_ball_point(xq_h, rq_h)
    assert _rows(rowptr.cpu(), col.cpu()) == [sorted(l) for l in refq]
    assert hoods.is_cuda and nk.is_cuda
    assert np.array_equal(nk.cpu().numpy(), [len(l) - 1 for l in ref])


def _padded_from_ckdtree(x, r, max_k=None):
    """the reference user's pipeline: query_ball_point lists without the point itself, padded with n"""
    n = len(x)
    tree = cKDTree(x)
    lists = [[j for j in sorted(l) if j != i] for i, l in enumerate(tree.query_ball_point(x, r))]
    if max_k is not None:
        for i, l in enumerate(lists):
            if len(l) > max_k:
                d2 = _d2(x[l], x[i])
                la = np.asarray(l)
                lists[i] = sorted(la[np.lexsort((la, d2))][:max_k].tolist())
    nk = np.array([len(l) for l in lists], np.int32)
    hoods = np.full((n, max(nk.max(), 1)), n, np.int32)
    for i, l in enumerate(lists):
        hoods[i, :len(l)] = l
    return hoods, nk


@pytest.mark.parametrize("dim,algo,max_k", [(2, 1, None), (2, 2, None), (3, 1, None), (3, 2, None),
                                            (2, 1, 12), (3, 2, 20), (2, 2, 12), (3, 1, 20)])
def test_fit_pipeline_bit_for_bit(dim, algo, max_k):
    n, order = 3000, 2
    rng = np.random.default_rng(20 + dim)
    x = rng.random((n, dim))
    f = np.sin(3 * x[:, 0]) + np.cos(2 * x[:, -1])
    no = wlsqm.number_of_dofs(dim, order)
    r = 0.06 if dim == 2 else 0.22
    _assert_clear_of_sphere(x, x, r)
    hoods, nk = wlsqm.ball_hoods(x, r, max_k=max_k)
    href, nkref = _padded_from_ckdtree(x, r, max_k)
    assert np.array_equal(nk, nkref) and np.array_equal(hoods, href)
    assert nk.min() >= no, "every neighbourhood must have at least as many points as DOFs"
    od, kn, wm = np.full(n, order, np.int32), np.zeros(n, np.int64), np.full(n, 1, np.int32)
    fi0 = np.zeros((n, no))
    w = hoods.shape[1]
    s1 = wlsqm.ExpertSolver(dim, nk, od, kn, wm, algorithm=algo, do_sens=True, max_iter=3)
    s1.prepare_hoods(x, hoods)
    fi_a, sens_a = fi0.copy(), np.zeros((n, w, no))
    s1.solve_hoods(f, fi_a, sens_a)
    xp = np.concatenate([x, np.zeros((1, dim))])
    fp = np.concatenate([f, [0.0]])
    xk, fk = np.ascontiguousarray(xp[href]), np.ascontiguousarray(fp[href])
    s2 = wlsqm.ExpertSolver(dim, nkref, od, kn, wm, algorithm=algo, do_sens=True, max_iter=3)
    s2.prepare(x, xk)
    fi_b, sens_b = fi0.copy(), np.zeros((n, w, no))
    s2.solve(fk, fi_b, sens_b)
    assert np.array_equal(fi_a, fi_b)
    for i in range(0, n, 50):
        assert np.array_equal(sens_a[i, :nk[i]], sens_b[i, :nk[i]])


def test_full_size_1m_2d():
    n = 1_000_000
    x = np.random.default_rng(30).random((n, 2))
    r = np.sqrt(30.0 / (np.pi * n))                     # mean of about 30 neighbours
    g = wlsqm.PointGrid(x)
    rowptr, col = g.ball(r, exclude_self=False)
    ref = cKDTree(x).query_ball_point(x, r, workers=-1, return_sorted=True)
    lens = np.fromiter((len(l) for l in ref), np.int64, n)
    assert np.array_equal(np.diff(rowptr), lens)
    assert np.array_equal(col, np.concatenate([np.asarray(l, np.int32) for l in ref]))
    assert 25 < col.shape[0] / n < 35


def test_validation():
    x = _cloud(1000, 2, "uniform")
    g = wlsqm.PointGrid(x)
    with pytest.raises(ValueError):
        g.ball(np.full(999, 0.1))                       # r of the wrong length
    with pytest.raises(ValueError):
        g.ball(-0.1)
    with pytest.raises(ValueError):
        g.ball(np.nan)
    r = np.full(1000, 0.1)
    r[3] = np.nan
    with pytest.raises(ValueError):
        g.ball(r)
    for k in (0, 129, -1):
        with pytest.raises(ValueError):
            g.ball(0.1, max_k=k)
    with pytest.raises(ValueError):
        g.ball(0.1, x[:10], exclude_self=True)
    with pytest.raises(ValueError):
        g.ball(0.1, np.zeros((10, 3)))                  # dimension mismatch
    with pytest.raises(ValueError):
        g.ball(0.1, order="nearest")
    torch = pytest.importorskip("torch")
    with pytest.raises(ValueError, match="ball"):
        g.query_ball_point(torch.zeros((3, 2), dtype=torch.float64, device="cuda"), 0.1)
    rt = torch.full((1000,), 0.1, dtype=torch.float64, device="cuda")
    rt[5] = -1.0
    with pytest.raises(ValueError):
        g.ball(rt)
    with pytest.raises(ValueError):
        g.ball(torch.tensor(float("nan"), dtype=torch.float64, device="cuda"))
    # no queries: the arguments are still checked
    empty = np.zeros((0, 2))
    for bad in (dict(r=-1.0), dict(r=0.1, max_k=500), dict(r=0.1, order="x"), dict(r=np.full(3, 0.1))):
        r = bad.pop("r")
        with pytest.raises(ValueError):
            g.ball(r, empty, **bad)
