"""GPU half of the extended-precision accuracy tests: every fit path against tests/hp_reference.py on the geometry
matrix, exact relations that need no reference, and pivot ties in the batched LAPACK-style drivers.

* Bound (hp_reference.BOUND_C): one-shot fused kernel, one-shot general path, ExpertSolver (packed and one-case-per-warp
  solve kernels, register and shared-memory prepare kernels), ALGO_ITERATIVE (3D order 4 with nr = 35, 34, 33),
  heterogeneous batches (per-order launches and one launch), geometry-uniform batches with per-case knowns, `sens`
  entry by entry, `interpolate` on the GPU's own coefficients.  Every batch interleaves the spacings 2^-20, 2^10 and 1
  case by case, so neighbouring fits in a warp differ by up to 2^30 in scale.
* Translation by 2^12 (dyadic inputs, xk - xi exact): fi, sens, iteration counts and interpolate outputs bit for bit.
* Batch order: the same cases in another order (same counts and sizes, same launch plan): every row bit for bit.
* Pivot ties: mgeneralfactor / msymmetricfactor on matrices whose column maxima tie, exactly or in the high word only.
"""
import os

import numpy as np
import pytest

import hp_reference as hp
import oracle as orc

pytestmark = pytest.mark.gpu

wlsqm = pytest.importorskip("wlsqm_b200")

PATHS = {
    "oneshot": ("oneshot", {}),
    "oneshot_general": ("oneshot", {"WLSQM_FIT_DIRECT": "0"}),
    "expert": ("expert", {}),
    "expert_nopack": ("expert", {"WLSQM_SOLVE_NOPACK": "1"}),
    "expert_smem_prepare": ("expert", {"WLSQM_PREP_KERNEL": "smem"}),
    "iterative": ("iterative", {}),
}


def _batches():
    return hp.matrix_batches()


class _Env:
    def __init__(self, env):
        self.env, self.old = env, {}

    def __enter__(self):
        for k, v in self.env.items():
            self.old[k] = os.environ.get(k)
            os.environ[k] = v

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _solve(kind, dim, meta, xi, xk, fk, fi0, env=(), do_sens=False):
    """(fi, sens, per-case iterations, solver)"""
    nk, od, kn, wm = meta
    fi = fi0.copy()
    with _Env(dict(env)):
        if kind == "oneshot":
            fit = getattr(wlsqm, "fit_%dD_many_parallel" % dim)
            assert fit(xk, fk, nk, xi, fi, None, 0, od, kn, wm) == 0
            return fi, None, None, None
        algo = wlsqm.ALGO_ITERATIVE if kind == "iterative" else wlsqm.ALGO_BASIC
        s = wlsqm.ExpertSolver(dim, nk, od, kn, wm, algorithm=algo, do_sens=do_sens, max_iter=3)
        s.prepare(xi, xk)
        sens = np.zeros((len(nk), xk.shape[1], fi.shape[1])) if do_sens else None
        s.solve(fk, fi, sens)
        return fi, sens, s.iterations(), s


def _bits(a):
    return None if a is None else np.ascontiguousarray(a).view(np.uint64 if a.dtype == np.float64 else a.dtype)


def _same(a, b):
    return (a is None and b is None) or np.array_equal(_bits(a), _bits(b))


def _report(title, worst):
    print("\n" + title)
    for key in sorted(worst):
        print("   %-40s worst ratio %.3g" % (key, worst[key]))


def _report_unjudged(unjudged):
    """cases run but not judged: kappa(S) eps above hp_reference.KAPPA_EPS_MAX (or no unknowns)"""
    counts = {}
    for u in unjudged:
        counts[u] = counts.get(u, 0) + 1
    print("   %d cases run but not judged (kappa eps > %g or nr = 0)%s" % (
        len(unjudged), hp.KAPPA_EPS_MAX, "".join("\n      %-36s %d" % kv for kv in sorted(counts.items()))))


@pytest.mark.parametrize("path", list(PATHS))
def test_paths_within_bound_and_translation_exact(path):
    kind, env = PATHS[path]
    worst = {}
    fails = []
    unjudged = []
    for b in _batches():
        for poly in (False, True):
            fk, fi0 = (b.fkp, b.fi0p) if poly else (b.fk, b.fi0)
            out = {}
            for T in (0.0, hp.T_SHIFT):
                xi, xk = b.place(T)
                out[T] = _solve(kind, b.dim, b.meta, xi, xk, fk, fi0, env)
            a, t = out[0.0], out[hp.T_SHIFT]
            assert _same(a[0], t[0]), ("translation changed fi", path, b.dim, b.order, b.knowns, b.wm, b.nk)
            assert _same(a[2], t[2]), ("translation changed the iteration counts", path, b.dim, b.order)
            for o in range(b.no):
                if b.knowns >> o & 1:
                    assert _same(a[0][:, o], fi0[:, o])
            r = b.ratios(a[0], poly)
            for i in range(b.n):
                if np.isnan(r[i]):
                    if not poly:
                        unjudged.append("%s %dD order %d" % (b.geom[i], b.dim, b.order))
                    continue
                key = "%s %dD" % (b.geom[i], b.dim)
                worst[key] = max(worst.get(key, 0.0), r[i])
                if r[i] > hp.BOUND_C:
                    fails.append((b.geom[i], b.dim, b.order, b.knowns, b.wm, b.nk, b.h[i], poly, r[i]))
    _report("path %s: error / (g(nk) eps ||S^-1|| (nr ||y*|| + ||f||_w)), threshold %g" % (path, hp.BOUND_C), worst)
    _report_unjudged(unjudged)
    assert not fails, fails[:20]


def _merge(items, T=0.0, poly=False):
    """one batch from (Batch, case) pairs: per-case sizes, orders, knowns and weightings; xk / fk padded"""
    dim = items[0][0].dim
    n = len(items)
    maxnk = max(b.nk for b, _ in items)
    maxno = max(b.no for b, _ in items)
    xi = np.zeros((n, dim))
    xk = np.zeros((n, maxnk, dim))
    fk = np.zeros((n, maxnk))
    fi0 = np.zeros((n, maxno))
    placed = {}
    for j, (b, i) in enumerate(items):
        if id(b) not in placed:
            p = b.place(T)
            placed[id(b)] = (p[0].reshape(b.n, dim), p[1].reshape(b.n, b.nk, dim))
        bxi, bxk = placed[id(b)]
        xi[j] = bxi[i]
        xk[j, :b.nk] = bxk[i]
        xk[j, b.nk:] = bxi[i]
        fk[j, :b.nk] = (b.fkp if poly else b.fk)[i]
        fi0[j, :b.no] = (b.fi0p if poly else b.fi0)[i]
    meta = (np.array([b.nk for b, _ in items], np.int32), np.array([b.order for b, _ in items], np.int32),
            np.array([b.knowns for b, _ in items], np.int64), np.array([b.wm for b, _ in items], np.int32))
    if dim == 1:
        xi, xk = xi[:, 0].copy(), np.ascontiguousarray(xk[:, :, 0])
    return meta, xi, xk, fk, fi0


def _item_ratio(b, i, fi, poly):
    if not b.judged(i):
        return np.nan
    c, s, sp = b.reference()[i]
    return c.ratio(sp if poly else s, fi[:b.no])


def _hetero_items(dim):
    """round robin over the dimension's batches, so that neighbouring cases differ in size, order and spacing"""
    bs = [b for b in _batches() if b.dim == dim]
    items = []
    for i in range(max(b.n for b in bs)):
        items += [(b, i) for b in bs if i < b.n]
    return items


@pytest.mark.parametrize("dim", [1, 2, 3])
@pytest.mark.parametrize("bucket_min", ["1", str(1 << 30)])
@pytest.mark.parametrize("algo", ["expert", "iterative"])
def test_heterogeneous_batch_within_bound(dim, bucket_min, algo):
    """per-case nk / order / knowns / weighting in one batch; WLSQM_PREP_BUCKET_MIN low: one prepare launch per order,
    high: one launch for all"""
    items = _hetero_items(dim)
    env = {"WLSQM_PREP_BUCKET_MIN": bucket_min}
    worst, fails, unjudged = 0.0, [], []
    for poly in (False, True):
        res = {}
        for T in (0.0, hp.T_SHIFT):
            meta, xi, xk, fk, fi0 = _merge(items, T, poly)
            res[T] = _solve(algo, dim, meta, xi, xk, fk, fi0, env)
        assert _same(res[0.0][0], res[hp.T_SHIFT][0]), "translation changed fi"
        assert _same(res[0.0][2], res[hp.T_SHIFT][2]), "translation changed the iteration counts"
        for j, (b, i) in enumerate(items):
            r = _item_ratio(b, i, res[0.0][0][j], poly)
            if np.isnan(r):
                if not poly:
                    unjudged.append("%s %dD order %d" % (b.geom[i], dim, b.order))
            else:
                worst = max(worst, r)
                if r > hp.BOUND_C:
                    fails.append((b.geom[i], b.order, b.knowns, b.wm, b.nk, b.h[i], poly, r))
    print("\nheterogeneous %dD %s bucket_min=%s: worst ratio %.3g over %d cases" % (dim, algo, bucket_min, worst, len(items)))
    _report_unjudged(unjudged)
    assert not fails, fails[:20]


@pytest.mark.parametrize("dim,order", [(1, 3), (2, 2), (2, 4), (3, 2), (3, 3)])
def test_geometry_uniform_batch_with_per_case_knowns(dim, order):
    """same sizes, a different knowns mask per case (same count of knowns): packed / per-warp solve of uniform shapes"""
    masks = (0b1, 0b10, 1 << (hp.number_of_dofs(dim, order) - 1))
    bs = [hp.Batch(dim, order, m, hp.WEIGHT_CENTER, seed=50 + order) for m in masks]
    items = [(bs[j % 3], j // 3 % bs[0].n) for j in range(3 * bs[0].n)]
    worst = 0.0
    unjudged = [b.geom[i] for b, i in items if not b.judged(i)]
    for kind, env in (("expert", {}), ("expert", {"WLSQM_SOLVE_NOPACK": "1"})):
        for poly in (False, True):
            meta, xi, xk, fk, fi0 = _merge(items, 0.0, poly)
            fi = _solve(kind, dim, meta, xi, xk, fk, fi0, env)[0]
            for j, (b, i) in enumerate(items):
                r = _item_ratio(b, i, fi[j], poly)
                if not np.isnan(r):
                    worst = max(worst, r)
                    assert r <= hp.BOUND_C, (b.geom[i], b.knowns, b.h[i], poly, r, env)
    print("\ngeometry-uniform %dD order %d, per-case knowns: worst ratio %.3g" % (dim, order, worst))
    _report_unjudged(["%s %dD order %d" % (g, dim, order) for g in unjudged])


def test_iterative_3d_order4_nr33_to_35():
    """ALGO_ITERATIVE with 35, 34 and 33 unknowns (the exchange tree of columns 32-34 of the solve kernel)"""
    worst = {}
    for kn in (0, 1, 0b11):
        b = hp.Batch(3, 4, kn, hp.WEIGHT_UNIFORM, seed=70 + kn, geoms=("random", "lattice", "one_sided"))
        for poly in (False, True):
            fk, fi0 = (b.fkp, b.fi0p) if poly else (b.fk, b.fi0)
            xi, xk = b.place(0.0)
            fi, _, it, _ = _solve("iterative", 3, b.meta, xi, xk, fk, fi0)
            r = b.ratios(fi, poly)
            worst[35 - bin(kn).count("1")] = max(worst.get(35 - bin(kn).count("1"), 0.0), np.nanmax(r))
            assert np.nanmax(r) <= hp.BOUND_C, (kn, poly, r)
    print("\nALGO_ITERATIVE 3D order 4, worst ratio by nr:", worst)


SENS_BATCHES = [(1, 2), (1, 4), (2, 1), (2, 3), (3, 1), (3, 2)]


def test_sens_against_exact_operator():
    worst = {}
    unjudged = []
    for b in _batches():
        if (b.dim, b.order) not in SENS_BATCHES or b.wm != hp.WEIGHT_CENTER or b.geom[0] in ("square",):
            continue
        res = {}
        for T in (0.0, hp.T_SHIFT):
            xi, xk = b.place(T)
            res[T] = _solve("expert", b.dim, b.meta, xi, xk, b.fk, b.fi0, do_sens=True)
        assert _same(res[0.0][1], res[hp.T_SHIFT][1]), "translation changed sens"
        sens = res[0.0][1]
        for o in range(b.no):
            if b.knowns >> o & 1:
                assert np.isnan(sens[:, :b.nk, o]).all()
        for i in range(b.n):
            if not b.judged(i):
                unjudged.append("%s %dD order %d" % (b.geom[i], b.dim, b.order))
                continue
            c = b.reference()[i][0]
            dfk, _ = c.operator()
            r = c.operator_ratio(dfk, sens[i])
            key = "%s %dD" % (b.geom[i], b.dim)
            worst[key] = max(worst.get(key, 0.0), r)
            assert r <= hp.BOUND_C, (b.geom[i], b.dim, b.order, b.knowns, b.h[i], r)
    _report("sens vs the exact operator, threshold %g" % hp.BOUND_C, worst)
    _report_unjudged(unjudged)


def test_interpolate_against_exact_evaluation():
    """single slots and diff='all' on the GPU's own coefficients; nearest-model search and outputs unchanged by the shift"""
    worst = {}
    for b in _batches():
        if b.wm != hp.WEIGHT_UNIFORM or b.knowns != 0 or b.geom[0] in ("square", "almost_square"):
            continue
        rng = np.random.default_rng(b.dim * 10 + b.order)
        q = np.round(rng.uniform(-0.5, 0.5, (b.n, b.dim)) * 2 ** 20) / 2 ** 20
        outs = {}
        for T in (0.0, hp.T_SHIFT):
            xi, xk = b.place(T)
            fi, _, _, s = _solve("expert", b.dim, b.meta, xi, xk, b.fk, b.fi0)
            xi2 = xi.reshape(b.n, b.dim)
            xq = xi2 + b.h[:, None] * q
            assert np.array_equal(xq - xi2, b.h[:, None] * q)
            xq_in = xq if b.dim > 1 else np.ascontiguousarray(xq[:, 0])
            s.prep_interpolate()
            o_all, I = s.interpolate(xq_in, diff="all")
            assert np.array_equal(I, np.arange(b.n))
            singles = {d: s.interpolate(xq_in, diff=d, I=np.arange(b.n))[0] for d in sorted({0, 1 % b.no, b.no - 1})}
            outs[T] = (fi, o_all, singles, xi2, xq)
        fi, o_all, singles, xi2, xq = outs[0.0]
        assert _same(o_all, outs[hp.T_SHIFT][1]), "translation changed interpolate(diff='all')"
        for d in singles:
            assert _same(singles[d], outs[hp.T_SHIFT][2][d]), ("translation changed interpolate", d)
        for i in range(b.n):
            for d in range(b.no):
                v, mag = hp.hp_eval(b.dim, xi2[i], fi[i], xq[i], d)
                lim = hp.eval_bound(b.dim, b.order, mag)
                for got in ([o_all[i, d]] + ([singles[d][i]] if d in singles else [])):
                    e = abs(float(hp.mp.mpf(float(got)) - v))
                    r = e / lim if lim > 0 else (0.0 if e == 0 else np.inf)
                    key = "%dD order %d" % (b.dim, b.order)
                    worst[key] = max(worst.get(key, 0.0), r)
                    assert r <= 1.0, (b.geom[i], b.dim, b.order, b.h[i], d, got, float(v), r)
    _report("interpolate vs exact evaluation: error / ((no + 2 order + 2) eps sum|terms|)", worst)


@pytest.mark.parametrize("path", ["oneshot", "expert", "expert_nopack", "iterative", "hetero"])
def test_batch_order_does_not_change_rows(path):
    """a case's result does not depend on its neighbours in the batch (group reductions, nrmax, packing)"""
    rng = np.random.default_rng(5)
    for dim in (1, 2, 3):
        if path == "hetero":
            groups = [_hetero_items(dim)]
            kind, env = "expert", {"WLSQM_PREP_BUCKET_MIN": "1"}
        else:
            kind, env = PATHS[path]
            groups = [[(b, i) for i in range(b.n)] for b in _batches() if b.dim == dim and b.order >= 1]
        for items in groups:
            perm = rng.permutation(len(items))
            base = _merge(items)
            shuf = _merge([items[p] for p in perm])
            a = _solve(kind, dim, *base, env=env)
            s = _solve(kind, dim, *shuf, env=env)
            assert _same(a[0][perm], s[0]), (path, dim, items[0][0].order)
            if a[2] is not None:
                assert _same(a[2][perm], s[2])


# ---- pivot ties in the batched drivers ---------------------------------------------------------------------------
# A pivot decision is only comparable across implementations where it is made from the same numbers: two candidates
# that tie in exact arithmetic can fall apart by one rounding (a / d against a * (1 / d), fma against multiply-then-add),
# and then either choice is right.  So every system is replayed on the host in float64 and in extended precision (numpy
# longdouble) step by step, and its EXACT PREFIX is the run of leading pivot decisions made from a state that every
# correct implementation reaches exactly: the first decision always (it sees the input), each later one while every
# earlier pivot was a power of two (so that a / d and a * (1 / d) agree) and the two replays still agree entry for entry.
# Within the prefix a differing pivot is a tie broken the wrong way.  The generators keep the prefixes long: sparse
# matrices of +-1 entries tie at almost every step and stay integer for tens of columns.
LU_TIERS = ((1, 8, "lu_reg_kernel<8>"), (9, 16, "lu_reg_kernel<16>"), (17, 32, "lu_reg_kernel<32>"),
            (33, 72, "getrf_kernel"))
SY_TIERS = ((1, 12, "sy_thread_kernel"), (13, 40, "sy_kernel (warp)"))
LU_KINDS = ["integer", "opposite_signs", "low_word", "zero_column", "plu_ties", "sparse_plu"]
SY_KINDS = ["integer", "opposite_signs", "sparse"]
_ALPHA = (1.0 + np.sqrt(17.0)) / 8.0


def _sparse_pm1(n, rng, lower):
    """unit-diagonal triangle with about three +-1 entries per column"""
    T = np.eye(n)
    for j in range(n):
        for i in rng.choice(n, min(n, 3), replace=False):
            if (i > j) if lower else (i < j):
                T[i, j] = rng.choice([-1.0, 1.0])
    return T


def _tie_matrices(kind, n, nlhs, rng):
    if kind == "integer":
        A = rng.integers(-2, 3, (n, n, nlhs)).astype(np.float64)
    elif kind == "opposite_signs":
        A = rng.choice([-2.0, -1.0, 1.0, 2.0], (n, n, nlhs))
    elif kind == "low_word":
        # each column's two largest entries share the high 32 bits (a, nextafter(a)) or tie exactly (a, -a)
        A = rng.uniform(-1, 1, (n, n, nlhs))
        for l in range(nlhs):
            for m in range(n):
                if n < 2:
                    continue
                r1, r2 = rng.choice(n, 2, replace=False)
                a = 2.0 + rng.uniform(0, 1)
                A[r1, m, l] = a * rng.choice([-1, 1])
                A[r2, m, l] = (np.nextafter(a, 4.0) if l % 3 == 0 else (a if l % 3 == 1 else np.nextafter(a, 0.0))) * rng.choice([-1, 1])
    elif kind == "zero_column":   # last column exactly zero (LAPACK still returns a pivot for it)
        A = rng.integers(-2, 3, (n, n, nlhs)).astype(np.float64)
        A[:, n - 1, :] = 0.0
    elif kind == "plu_ties":      # P L U with |l_ij| in {0, 1} and pivots +-1, +-2
        A = np.empty((n, n, nlhs))
        for l in range(nlhs):
            L = np.tril(rng.integers(-1, 2, (n, n)), -1) + np.eye(n)
            U = np.triu(rng.integers(-1, 2, (n, n)), 1) + np.diag(rng.choice([-2.0, -1.0, 1.0, 2.0], n))
            A[:, :, l] = (L @ U)[rng.permutation(n)]
    else:                         # sparse_plu: P L U with sparse +-1 triangles and a +-1 diagonal
        A = np.empty((n, n, nlhs))
        for l in range(nlhs):
            U = _sparse_pm1(n, rng, False) * rng.choice([-1.0, 1.0], n)[:, None]
            A[:, :, l] = (_sparse_pm1(n, rng, True) @ U)[rng.permutation(n)]
    return np.asfortranarray(A)


def _pow2(v):
    v = abs(float(v))
    return v > 0 and np.frexp(v)[0] == 0.5


def _high_word_tie(cands):
    """two or more candidates share the high 32 bits of the largest magnitude (exact ties included)"""
    hi = (np.abs(np.asarray(cands, np.float64)).view(np.uint64) >> np.uint64(32))
    return len(hi) > 1 and int((hi == hi.max()).sum()) > 1


def _lu_prefix(A):
    """(length of the exact prefix, its decisions that chose among tied candidates, the replay's ipiv)"""
    a, b = A.astype(np.float64), A.astype(np.longdouble)
    n = a.shape[0]
    ties = 0
    ipiv = []
    for p in range(n):
        ties += _high_word_tie(a[p:, p])
        q = p + int(np.argmax(np.abs(a[p:, p])))
        ipiv.append(q + 1)
        a[[p, q]], b[[p, q]] = a[[q, p]], b[[q, p]]
        if p == n - 1 or not _pow2(a[p, p]):
            return p + 1, ties, ipiv
        for x in (a, b):
            x[p + 1:, p] /= x[p, p]
            x[p + 1:, p + 1:] -= np.outer(x[p + 1:, p], x[p, p + 1:])
        if not np.array_equal(a.astype(np.longdouble), b):
            return p + 1, ties, ipiv
    return n, ties, ipiv


def _sy_step(A, k):
    """one step of oracle.sytf2_upper in A's dtype, in place: (kstep, the 1 x 1 pivot or None, a tie decided it)"""
    absakk = abs(A[k, k])
    imax, colmax = 0, 0.0
    if k > 0:
        imax = int(np.argmax(np.abs(A[:k, k])))
        colmax = abs(A[imax, k])
    if max(absakk, colmax) == 0.0:
        return 1, k, None, False
    tie = absakk < _ALPHA * colmax and _high_word_tie(A[:k, k])      # the first largest entry decides the interchange
    kstep, kp = 1, k
    if absakk < _ALPHA * colmax:
        rowmax = np.abs(A[imax, imax + 1:k + 1]).max()
        if imax > 0:
            rowmax = max(rowmax, np.abs(A[:imax, imax]).max())
        if absakk >= _ALPHA * colmax * (colmax / rowmax):
            kp = k
        elif abs(A[imax, imax]) >= _ALPHA * rowmax:
            kp = imax
        else:
            kp, kstep = imax, 2
    if kstep == 2:
        return 2, kp, None, tie              # the prefix ends with a 2 x 2 pivot (its update is not replayed)
    if kp != k:
        A[:kp, [k, kp]] = A[:kp, [kp, k]]
        t = A[kp + 1:k, k].copy()
        A[kp + 1:k, k] = A[kp, kp + 1:k]
        A[kp, kp + 1:k] = t
        A[k, k], A[kp, kp] = A[kp, kp], A[k, k]
    d = A[k, k]
    x = A[:k, k].copy()
    for j in range(k):
        if x[j] != 0.0:
            A[:j + 1, j] += x[:j + 1] * (-(1 / d) * x[j])
    A[:k, k] *= 1 / d
    return 1, kp, d, tie


def _sy_prefix(A):
    """(number of trailing ipiv entries decided from an exact state -- dsytf2 goes from the last column --, ties,
    the replay's ipiv, zero where not decided)"""
    a, b = np.triu(A).astype(np.float64), np.triu(A).astype(np.longdouble)
    n = a.shape[0]
    ties = 0
    ipiv = np.zeros(n, np.int32)
    for k in range(n - 1, -1, -1):
        kstep, kp, d, tie = _sy_step(a, k)
        _sy_step(b, k)
        ties += tie
        if kstep == 2:
            ipiv[k] = ipiv[k - 1] = -(kp + 1)
            return n - k + 1, ties, ipiv
        ipiv[k] = kp + 1
        if d is None or k == 0 or not _pow2(d) or not np.array_equal(np.triu(a).astype(np.longdouble), np.triu(b)):
            return n - k, ties, ipiv
    return n, ties, ipiv


def _coverage(tiers, seen, label):
    for lo, hi, name in tiers:
        nmax, ties = seen.get(name, (0, 0))
        print("%s %-20s largest n compared %2d, tied pivot decisions compared %d" % (label, name, nmax, ties))
        assert nmax == hi and ties > 0, (label, name, nmax, ties)


@pytest.mark.parametrize("kind", LU_KINDS)
def test_mgeneralfactor_pivot_ties(kind):
    from wlsqm_b200.utils import lapackdrivers as ld
    rng = np.random.default_rng(LU_KINDS.index(kind))
    seen = {}
    print()
    for n in range(1, 73):
        A = _tie_matrices(kind, n, 41, rng)
        LUo, ipo = A.copy(order="F"), np.zeros((n, 41), np.int32, order="F")
        orc.mgetrf(LUo, ipo)
        LU, ipiv = A.copy(order="F"), np.zeros_like(ipo)
        ld.mgeneralfactor(LU, ipiv)
        tier = next(name for lo, hi, name in LU_TIERS if lo <= n <= hi)
        for l in range(41):
            q, ties, replay = _lu_prefix(A[:, :, l])
            assert np.array_equal(replay, ipo[:q, l])           # the host replay follows the restatement
            assert np.array_equal(ipiv[:q, l], ipo[:q, l]), (kind, n, l, q, ipiv[:, l], ipo[:, l])
            if q == n:            # exact throughout: the factors agree as in test_batched_drivers_every_size
                assert np.allclose(LU[:, :, l], LUo[:, :, l], rtol=1e-8, atol=1e-10), (kind, n, l)
            s = seen.get(tier, (0, 0))
            seen[tier] = (max(s[0], n), s[1] + ties)
    _coverage(LU_TIERS, seen, "mgeneralfactor %s:" % kind)


@pytest.mark.parametrize("kind", SY_KINDS)
def test_msymmetricfactor_pivot_ties(kind):
    """sy_thread_kernel (n <= 12) and the warp kernel (larger n) against the dsytf2 restatement"""
    from wlsqm_b200.utils import lapackdrivers as ld
    rng = np.random.default_rng(3 + SY_KINDS.index(kind))
    seen = {}
    print()
    for n in range(1, 41):
        if kind == "sparse":      # +-1 off the diagonal, 0 / +-1 / +-2 on it: ties in the column maxima at most steps
            M = np.stack([_sparse_pm1(n, rng, False) * 1.0 for _ in range(37)])
            M[:, np.arange(n), np.arange(n)] = rng.choice([0.0, 0.0, 1.0, -1.0, 2.0, -2.0], (37, n))
        else:
            M = _tie_matrices(kind, n, 37, rng).transpose(2, 0, 1)
        A = np.asfortranarray((np.triu(M) + np.triu(M, 1).transpose(0, 2, 1)).transpose(1, 2, 0))
        Fo, ipo = A.copy(order="F"), np.zeros((n, 37), np.int32, order="F")
        orc.msytrf(Fo, ipo)
        F, ipiv = A.copy(order="F"), np.zeros_like(ipo)
        ld.msymmetricfactor(F, ipiv)
        tier = next(name for lo, hi, name in SY_TIERS if lo <= n <= hi)
        iu = np.triu_indices(n)
        for l in range(37):
            q, ties, replay = _sy_prefix(A[:, :, l])
            assert np.array_equal(replay[n - q:], ipo[n - q:, l])    # the host replay follows the restatement
            assert np.array_equal(ipiv[n - q:, l], ipo[n - q:, l]), (kind, n, l, q, ipiv[:, l], ipo[:, l])
            if q == n:
                assert np.allclose(F[:, :, l][iu], Fo[:, :, l][iu], rtol=1e-8, atol=1e-10), (kind, n, l)
            s = seen.get(tier, (0, 0))
            seen[tier] = (max(s[0], n), s[1] + ties)
    _coverage(SY_TIERS, seen, "msymmetricfactor %s:" % kind)
