"""CPU half of the extended-precision accuracy tests (tests/hp_reference.py states the criterion).

* self-checks of the reference: exact recovery of polynomials, the classical finite-difference stencils, the operator
  applied to the data reproduces the fit;
* the oracle (the C restatement of the original's algorithm) against the bound over the whole geometry matrix, with a
  table of the worst ratio and the worst kappa(S) per geometry x dimension x order -- the margin the constant was fixed
  with;
* translation by a power of two is bit for bit in the oracle (the GPU half relies on that relation).
"""
import numpy as np
import pytest
from mpmath import mp

import hp_reference as hp
import parity


def _hp_case(dim, order, knowns, wm, rel, h=1.0):
    xi = np.zeros(dim)
    return hp.HPCase(dim, order, knowns, wm, xi, h * rel)


@pytest.mark.parametrize("dim,order", [(1, 4), (2, 3), (2, 4), (3, 2), (3, 4)])
@pytest.mark.parametrize("wm", [hp.WEIGHT_UNIFORM, hp.WEIGHT_CENTER])
def test_reference_recovers_polynomials(dim, order, wm):
    """data from a polynomial of degree <= order, formed exactly: residual 0, the fit is the coefficients"""
    rng = np.random.default_rng(dim * 10 + order + wm)
    no = hp.number_of_dofs(dim, order)
    c = _hp_case(dim, order, 0, wm, hp.stencil("one_sided", dim, hp.default_nk(dim, order), rng), 2.0 ** -6)
    coef = rng.uniform(-1, 1, no)
    with mp.workdps(hp.DPS):
        fk = [mp.fsum(mp.mpf(coef[s]) * c.c[k][s] for s in range(no)) for k in range(c.nk)]
        sol = c.fit(fk)
        err = max(abs(sol["fi"][s] - mp.mpf(coef[s])) for s in range(no))
    assert err < 1e-30 * c.kappa, (err, c.kappa)
    # with knowns: the known slots hold the true coefficients, the rest is still recovered
    c2 = _hp_case(dim, order, 0b101, wm, hp.stencil("random", dim, hp.default_nk(dim, order), rng), 2.0 ** 3)
    with mp.workdps(hp.DPS):
        fk = [mp.fsum(mp.mpf(coef[s]) * c2.c[k][s] for s in range(no)) for k in range(c2.nk)]
        sol = c2.fit(fk, coef)
        assert max(abs(sol["fi"][s] - mp.mpf(coef[s])) for s in range(no)) < 1e-30 * c2.kappa


def test_reference_classical_stencils():
    """the stencils of test_gpu_golden.test_classical_stencils, exactly"""
    h = 2.0 ** -4
    f = np.sin
    c = hp.HPCase(1, 2, 0, hp.WEIGHT_UNIFORM, [0.0], np.array([-h, 0.0, h]))
    fk = f(np.array([-h, 0.0, h]))
    with mp.workdps(hp.DPS):
        sol = c.fit(fk)
        fm, f0, fp = (mp.mpf(v) for v in fk)
        assert abs(sol["fi"][0] - f0) < 1e-50
        assert abs(sol["fi"][1] - (fp - fm) / (2 * h)) < 1e-45
        assert abs(sol["fi"][2] - (fp - 2 * f0 + fm) / h ** 2) < 1e-45
    # 2D five-point plus with XY known (= 0): the four-neighbour Laplacian stencil, and its operator column
    gf = lambda x, y: np.exp(0.5 * x) * np.cos(y)
    xk = np.array([[0.0, 0.0], [h, 0.0], [-h, 0.0], [0.0, h], [0.0, -h]])
    iX2, iXY, iY2 = 3, 4, 5
    c2 = hp.HPCase(2, 2, 1 << iXY, hp.WEIGHT_UNIFORM, [0.0, 0.0], xk)
    g = gf(xk[:, 0], xk[:, 1])
    with mp.workdps(hp.DPS):
        sol = c2.fit(g, np.zeros(6))
        gk = [mp.mpf(v) for v in g]
        assert abs(sol["fi"][iX2] - (gk[1] - 2 * gk[0] + gk[2]) / h ** 2) < 1e-40
        assert abs(sol["fi"][iY2] - (gk[3] - 2 * gk[0] + gk[4]) / h ** 2) < 1e-40
        dfk, _ = c2.operator()
        want = [-2, 1, 1, 0, 0]
        assert all(abs(dfk[k][iX2] - mp.mpf(want[k]) / h ** 2) < 1e-40 for k in range(5))
        assert all(dfk[k][iXY] is None for k in range(5))


@pytest.mark.parametrize("dim,order,knowns,wm", [(1, 3, 0b10, 2), (2, 4, 0b1, 1), (2, 2, 0b110, 2), (3, 3, 0b1001, 1)])
def test_operator_reproduces_fit(dim, order, knowns, wm):
    rng = np.random.default_rng(order)
    nk = hp.default_nk(dim, order)
    c = _hp_case(dim, order, knowns, wm, hp.stencil("random", dim, nk, rng), 2.0 ** -3)
    fk = rng.standard_normal(nk)
    fkn = rng.standard_normal(c.no)
    with mp.workdps(hp.DPS):
        sol = c.fit(fk, fkn)
        dfk, dfkn = c.operator()
        for s in c.unknown:
            v = mp.fsum(dfk[k][s] * mp.mpf(fk[k]) for k in range(nk)) + mp.fsum(dfkn[m][s] * mp.mpf(fkn[m]) for m in c.known)
            assert abs(v - sol["fi"][s]) <= 1e-40 * (1 + abs(sol["fi"][s])) * c.kappa


def _oracle(b, T=0.0, algorithm=1, poly=False):
    xi, xk = b.place(T)
    fk, fi0 = (b.fkp, b.fi0p) if poly else (b.fk, b.fi0)
    fi, _, it, s = parity.oracle_solve(b.dim, *b.meta, xi, xk, fk, fi0, algorithm, False, 3)
    return fi, s


def test_oracle_within_bound_over_geometry_matrix():
    table = {}
    skipped = []
    worst = 0.0
    for b in hp.matrix_batches():
        ref = b.reference()
        r = np.fmax(b.ratios(_oracle(b)[0]), b.ratios(_oracle(b, poly=True)[0], poly=True))
        for i in range(b.n):
            key = (b.geom[i], b.dim, b.order)
            row = table.setdefault(key, [0.0, 0.0, 0, 0])
            if not b.judged(i):
                row[3] += 1
                skipped.append("%s %dD order %d h=%g kappa=%.1e" % (b.geom[i], b.dim, b.order, b.h[i], ref[i][0].kappa))
                continue
            row[0] = max(row[0], r[i])
            row[1] = max(row[1], ref[i][0].kappa)
            row[2] += 1
            worst = max(worst, r[i])
    print("\noracle vs extended precision: ratio = error / (g(nk) eps ||S^-1|| (nr ||y*|| + ||f||_w)), threshold %g" % hp.BOUND_C)
    print("%-16s %3s %5s %10s %10s %6s %7s" % ("geometry", "dim", "order", "worst", "kappa", "cases", "skipped"))
    for (gm, dim, order), (wr, kp, n, ns) in sorted(table.items(), key=lambda kv: (kv[0][1], kv[0][2], kv[0][0])):
        print("%-16s %3d %5d %10.2e %10.2e %6d %7d" % (gm, dim, order, wr, kp, n, ns))
    print("worst oracle ratio %.3g (%.3g of the threshold); %d cases skipped (kappa eps > %g)"
          % (worst, worst / hp.BOUND_C, len(skipped), hp.KAPPA_EPS_MAX))
    assert worst <= hp.BOUND_C / 4, worst
    # every geometry is judged somewhere, at every spacing
    for gm in hp.GEOMETRIES + ("square", "almost_square"):
        assert sum(v[2] for k, v in table.items() if k[0] == gm) > 0, gm


def test_oracle_interpolation_within_eval_bound():
    """the evaluation bound of hp_reference.eval_bound holds for the oracle's model evaluation"""
    import oracle as orc
    worst = 0.0
    for b in hp.matrix_batches():
        if b.geom[0] == "square":
            continue
        fi, _ = _oracle(b)
        xi, _ = b.place(0.0)
        xi = xi.reshape(b.n, b.dim)
        rng = np.random.default_rng(b.dim * 7 + b.order)
        xq = xi + b.h[:, None] * np.round(rng.uniform(-0.5, 0.5, (b.n, b.dim)) * 2 ** 20) / 2 ** 20
        for d in range(b.no):
            got = np.array([orc.interpolate_fit(xi[i] if b.dim > 1 else xi[i, 0], fi[i], b.dim, b.order, xq[i], d)[0]
                            for i in range(b.n)])
            for i in range(b.n):
                v, mag = hp.hp_eval(b.dim, xi[i], fi[i], xq[i], d)
                e = abs(float(mp.mpf(got[i]) - v))
                worst = max(worst, e / hp.eval_bound(b.dim, b.order, mag) if mag > 0 else 0.0)
    print("\nworst oracle evaluation ratio %.3g (threshold 1)" % worst)
    assert worst <= 0.25, worst


def test_oracle_translation_bit_for_bit():
    """shifting every coordinate by 2^12 (dyadic inputs: xk - xi is exact) changes nothing in the oracle"""
    for b in hp.matrix_batches():
        for algo in (1, 2):
            a, _ = _oracle(b, 0.0, algo)
            t, _ = _oracle(b, hp.T_SHIFT, algo)
            assert np.array_equal(a.view(np.uint64), t.view(np.uint64)), (b.dim, b.order, b.knowns, b.wm, algo)
