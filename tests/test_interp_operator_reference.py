"""CPU checks of the host reference for the interpolation operators (tests/interp_operator_reference.py): the Taylor
terms against exact rationals, and -- built from the oracle's `sens` -- rows at off-node query points that return the
exact derivatives of polynomial data the fit reproduces, with duplicate neighbours and centre folding, in 1D, 2D and
3D.  The identity bound that the GPU tests use is fixed here, on the oracle."""
from fractions import Fraction
from math import factorial

import numpy as np
import pytest
from scipy.spatial import cKDTree

import oracle as orc
import operator_reference as opref
import interp_operator_reference as ref
from hp_reference import EXPONENTS

IDENTITY_CONST = 16.0     # the bound's constant (interp_operator_reference.identity_bound): three times the worst oracle ratio (5.1), printed below

NO = {1: [1, 2, 3, 4, 5], 2: [1, 3, 6, 10, 15], 3: [1, 4, 10, 20, 35]}


def test_taylor_terms_are_one_hot_at_the_origin():
    for dim in (1, 2, 3):
        T = ref.T_matrix(dim, np.zeros(dim), NO[dim][4])
        assert np.array_equal(T, np.eye(NO[dim][4]))
        c = np.random.default_rng(dim).standard_normal((3, NO[dim][4]))
        c[:, ::3] = 0.0
        assert np.array_equal(ref.coefficient_rows_at(dim, c, np.zeros(dim)), c)


def test_taylor_terms_against_exact_rationals():
    rng = np.random.default_rng(7)
    worst = 0.0
    for dim in (1, 2, 3):
        no = NO[dim][4]
        ex = EXPONENTS[dim]
        for _ in range(20):
            h = rng.standard_normal(dim) * 10.0 ** rng.integers(-6, 3)
            T = ref.T_matrix(dim, h, no)
            hf = [Fraction(float(v)) for v in h] + [Fraction(0)] * 3
            for D in range(no):
                for s in range(no):
                    e = [ex[s][j] - ex[D][j] for j in range(3)]
                    if min(e) < 0:
                        assert T[D, s] == 0.0
                        continue
                    exact = Fraction(1)
                    for j in range(3):
                        exact *= hf[j] ** e[j] / factorial(e[j])
                    if exact == 0:
                        assert T[D, s] == 0.0
                        continue
                    err = abs(Fraction(float(T[D, s])) - exact) / abs(exact)
                    worst = max(worst, float(err) / np.finfo(np.float64).eps)
    print("Taylor terms: worst relative error %.2f ulp" % worst)
    assert worst <= 8.0


def _poly(dim, order, seed):
    """Taylor coefficients g at 0 of a polynomial of degree `order`, and d^D f at points x for every slot D"""
    no = NO[dim][order]
    g = np.random.default_rng(seed).standard_normal(no)
    ex = EXPONENTS[dim]

    def deriv(x, D):
        x = np.asarray(x, np.float64).reshape(-1, dim)
        out = np.zeros(len(x))
        p = ex[D]
        for s in range(no):
            e = [ex[s][j] - p[j] for j in range(3)]
            if min(e) < 0:
                continue
            term = g[s] * np.ones(len(x))
            for j in range(dim):
                term = term * x[:, j] ** e[j] / factorial(e[j])
            out += term
        return out
    return no, deriv


def _problem(dim, order, k, knowns_mask, center, n=120, seed=3):
    rng = np.random.default_rng(seed)
    npoints = n + center + 40
    x = rng.random((npoints, dim))
    xi = x[center:center + n]
    _, hoods = cKDTree(x).query(xi, k)
    hoods = hoods.astype(np.int32)
    hoods[::7, 3] = hoods[::7, 1]                   # duplicate neighbours
    nk = np.full(n, k, np.int32)
    nk[::5] = k - 2
    hoods[::5, k - 2:] = npoints + 999              # garbage padding, never read
    order_a = np.full(n, order, np.int32)
    knowns = np.full(n, knowns_mask, np.int64)
    wm = np.full(n, 2, np.int32)
    return x, xi, hoods, nk, order_a, knowns, wm


def _oracle(dim, x, xi, hoods, nk, order, knowns, wm, no):
    n, k = hoods.shape
    safe = np.where(np.arange(k)[None, :] < nk[:, None], hoods, 0)
    xk = x[safe] if dim > 1 else x[safe][:, :, 0]
    so = orc.OracleSolver(dim, nk, order, knowns, wm, do_sens=True)
    so.prepare(xi, xk)
    sens = np.zeros((n, k, no))
    so.solve(np.zeros((n, k)), np.zeros((n, no)), sens)

    def solve(fi_in):
        fi = fi_in.copy()
        so.solve(np.zeros((n, k)), fi, np.zeros((n, k, no)))
        return fi
    dfk = opref.known_weights_from_solves(solve, n, no, np.full(n, no), knowns)
    return so, sens, dfk, safe


def _queries(x, xi, nq, seed):
    rng = np.random.default_rng(seed)
    lo, hi = x.min(0), x.max(0)
    xq = lo + (hi - lo) * rng.random((nq, x.shape[1]))
    _, I = cKDTree(xi).query(xq, 1)
    return xq, I.astype(np.int64)


@pytest.mark.parametrize("dim,order,k", [(1, 3, 7), (2, 2, 12), (3, 2, 20)])
@pytest.mark.parametrize("knowns_mask,center", [(0, None), (1, 11)])
def test_rows_reproduce_exact_derivatives_at_off_node_queries(dim, order, k, knowns_mask, center):
    x, xi, hoods, nk, order_a, knowns, wm = _problem(dim, order, k, knowns_mask, center or 0, seed=dim)
    n, npoints = len(nk), len(x)
    no, deriv = _poly(dim, order, seed=10 + dim)
    _, sens, dfk, safe = _oracle(dim, x, xi, hoods, nk, order_a, knowns, wm, no)
    xq, I = _queries(x, xi, 60, seed=dim)
    I[5] = n                                         # no model found (a NaN query's index)
    c = np.eye(no)
    cq = ref.query_rows(dim, c, xq, xi, I, n)
    W, K = ref.stencils(sens, dfk, nk, np.full(n, no), knowns, cq, I)
    f = deriv(x, 0)
    fi_known = np.zeros((n, no))
    if knowns_mask:
        fi_known[:, 0] = deriv(xi, 0)
    rowptr, col, values, Kf = ref.csr(W, K, hoods, nk, knowns, npoints, I, n, center=center)
    E = opref.scipy_matrices(rowptr, col, values, len(I), npoints)
    ok = np.arange(len(I)) != 5
    assert rowptr[6] == rowptr[5] and np.isnan(K[:, 5]).all() and not W[:, 5].any()
    fk = np.where(np.arange(k)[None, :] < nk[:, None], f[safe], 0.0)
    r = np.median(np.linalg.norm(x[hoods[:, 1]] - xi, axis=-1))      # neighbour spacing: a |D|-th derivative of the
    for D in range(no):                                                   # fit loses (1/r)^|D| of the data's precision
        want = deriv(xq, D)
        got = (W[D] * fk[np.minimum(I, n - 1)]).sum(-1) + (K[D] * fi_known[np.minimum(I, n - 1)]).sum(-1)
        got_e = E[D] @ f + (Kf[D] * fi_known[np.minimum(I, n - 1)]).sum(-1)
        tol = 1e-11 * max(1.0, np.abs(want).max()) / r ** sum(EXPONENTS[dim][D])
        assert np.abs(got - want)[ok].max() < tol, D
        assert np.abs(got_e - want)[ok].max() < tol, D
        assert np.isnan(got[5]) and np.isnan(got_e[5])


def test_identity_bound_constant_on_the_oracle():
    """|E f + K . fi_known - interpolate(x, I, diff)| against the bound, after a solve of random data"""
    rng = np.random.default_rng(5)
    worst = 0.0
    for dim, order, k in [(1, 4, 9), (2, 4, 20), (3, 3, 26)]:
        for knowns_mask in (0, 1, 0b1001):
            x, xi, hoods, nk, order_a, knowns, wm = _problem(dim, order, k, knowns_mask, 9, seed=11 + knowns_mask + dim)
            n = len(nk)
            no = NO[dim][order]
            so, sens, dfk, safe = _oracle(dim, x, xi, hoods, nk, order_a, knowns, wm, no)
            f = rng.standard_normal(len(x))
            fk = np.where(np.arange(k)[None, :] < nk[:, None], f[safe], 0.0)
            fi_in = rng.standard_normal((n, no))
            fi_out = fi_in.copy()
            so.solve(fk, fi_out, np.zeros(sens.shape))
            xq, I = _queries(x, xi, 50, seed=dim + knowns_mask)
            c = np.vstack([np.eye(no), rng.standard_normal((2, no))])
            cq = ref.query_rows(dim, c, xq, xi, I, n)
            cq_abs = ref.query_rows(dim, np.abs(c), np.abs(xq - xi[I]), np.zeros_like(xi), I, n)
            W, K = ref.stencils(sens, dfk, nk, np.full(n, no), knowns, cq, I)
            lhs = (W * fk[I][None]).sum(-1) + (K * fi_in[I][None]).sum(-1)
            interp = np.stack([so.interpolate(xq if dim > 1 else xq[:, 0], I, D) for D in range(no)], -1)   # (nq, no)
            rhs = np.stack([(interp * c[o]).sum(-1) for o in range(len(c))])
            bound = ref.identity_bound(np.transpose(cq_abs, (1, 0, 2)), sens[I], dfk[I], fk[I], fi_in[I], fi_out[I], 1.0)
            worst = max(worst, float((np.abs(lhs - rhs) / bound).max()))
    print("interpolation identity: worst |error| / (L eps scale) on the oracle = %.3f (constant %.1f)" % (worst, IDENTITY_CONST))
    assert worst <= IDENTITY_CONST
