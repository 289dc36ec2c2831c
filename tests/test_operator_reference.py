"""CPU checks of the host reference for the operator export (tests/operator_reference.py), built from the oracle's
`sens`: applied to samples of a polynomial the fit reproduces exactly, the stencil weights, the known-value weights
and the assembled sparse operator return the exact slot combination -- with duplicate neighbours, the centre among its
own neighbours and centre folding.  The identity bound that the GPU tests use is fixed here, on the oracle."""
import numpy as np
import pytest
from scipy.spatial import cKDTree

import oracle as orc
import operator_reference as ref

IDENTITY_CONST = 4.0      # the bound's constant (operator_reference.identity_bound); worst oracle ratio printed below


def _poly2(x, y):
    """f = 1 + 2x - 3y + x^2/2 + xy - 2y^2 and its slots F, X, Y, X2, XY, Y2 at (x, y)"""
    f = 1 + 2 * x - 3 * y + 0.5 * x * x + x * y - 2 * y * y
    return f, np.stack([f, 2 + x + y, -3 + x - 4 * y, np.ones_like(x), np.ones_like(x), np.full_like(x, -4.0)], -1)


def _problem(knowns_mask, center, n=300, k=12, seed=3):
    rng = np.random.default_rng(seed)
    npoints = n + center + 40
    x = rng.random((npoints, 2))
    xi = x[center:center + n]
    _, hoods = cKDTree(x).query(xi, k)              # the centre is its own nearest neighbour
    hoods = hoods.astype(np.int32)
    hoods[::7, 3] = hoods[::7, 1]                   # duplicate neighbours
    nk = np.full(n, k, np.int32)
    nk[::5] = k - 2                                 # ragged rows ...
    hoods[::5, k - 2:] = npoints + 999              # ... with garbage padding
    order = np.full(n, 2, np.int32)
    knowns = np.full(n, knowns_mask, np.int64)
    wm = np.full(n, 1, np.int32)
    return x, xi, hoods, nk, order, knowns, wm


def _oracle_export(x, xi, hoods, nk, order, knowns, wm):
    n, k = hoods.shape
    safe = np.where(np.arange(k)[None, :] < nk[:, None], hoods, 0)
    xk = x[safe]
    so = orc.OracleSolver(2, nk, order, knowns, wm, do_sens=True)
    so.prepare(xi, xk)
    sens = np.zeros((n, k, 6))
    so.solve(np.zeros((n, k)), np.zeros((n, 6)), sens)

    def solve(fi_in):
        fi = fi_in.copy()
        so.solve(np.zeros((n, k)), fi, np.zeros((n, k, 6)))
        return fi
    dfk = ref.known_weights_from_solves(solve, n, 6, np.full(n, 6), knowns)
    return so, sens, dfk, safe


@pytest.mark.parametrize("knowns_mask,center", [(0, 0), (0, 17), (1, 0), (1, 17)])
def test_reference_reproduces_polynomial_slots(knowns_mask, center):
    x, xi, hoods, nk, order, knowns, wm = _problem(knowns_mask, center)
    n = len(nk)
    _, sens, dfk, _ = _oracle_export(x, xi, hoods, nk, order, knowns, wm)
    f, slots = _poly2(x[:, 0], x[:, 1])
    exact = slots[center:center + n]
    lap = np.zeros(6)
    lap[3] = lap[5] = 1.0
    c = np.vstack([np.eye(6), lap])
    W, K = ref.stencils(sens, dfk, nk, np.full(n, 6), knowns, c)
    rowptr, col, values, Kf = ref.csr(W, K, hoods, nk, knowns, len(x), center=center if knowns_mask else None)
    # the pattern is the canonical CSR of the used hood entries (+ the folded diagonal)
    rows = np.repeat(np.arange(n), nk)
    cols = np.concatenate([hoods[i, :nk[i]] for i in range(n)])
    if knowns_mask:
        rows, cols = np.concatenate([rows, np.arange(n)]), np.concatenate([cols, center + np.arange(n)])
    canon = ref.sp.csr_array((np.ones(len(rows)), (rows, cols)), shape=(n, len(x)))
    canon.sum_duplicates()
    canon.sort_indices()
    assert np.array_equal(canon.indptr, rowptr) and np.array_equal(canon.indices, col)
    fi_known = np.zeros((n, 6))
    fi_known[:, 0] = f[center:center + n] if knowns_mask else 0.0
    for o, D in enumerate(ref.scipy_matrices(rowptr, col, values, n, len(x))):
        got = D @ f + (Kf[o] * fi_known).sum(-1)
        want = (exact * c[o]).sum(-1)
        assert np.abs(got - want).max() < 1e-10 * max(1.0, np.abs(want).max()), o
        # without folding the same holds with K applied to the known values directly
        if knowns_mask:
            fk = np.where(np.arange(hoods.shape[1])[None, :] < nk[:, None], f[np.minimum(hoods, len(x) - 1)], 0.0)
            got2 = (W[o] * fk).sum(-1) + (K[o] * fi_known).sum(-1)
            assert np.abs(got2 - want).max() < 1e-10 * max(1.0, np.abs(want).max())


def test_identity_bound_constant_on_the_oracle():
    rng = np.random.default_rng(5)
    worst = 0.0
    for knowns_mask in (0, 1, 0b1001):
        x, xi, hoods, nk, order, knowns, wm = _problem(knowns_mask, 9, seed=11 + knowns_mask)
        n = len(nk)
        so, sens, dfk, safe = _oracle_export(x, xi, hoods, nk, order, knowns, wm)
        f = rng.standard_normal(len(x))
        fk = np.where(np.arange(hoods.shape[1])[None, :] < nk[:, None], f[safe], 0.0)
        fi_in = rng.standard_normal((n, 6))
        fi_out = fi_in.copy()
        so.solve(fk, fi_out, np.zeros(sens.shape))
        c = np.vstack([rng.standard_normal((3, 6)), np.eye(6)[[3]] + np.eye(6)[[5]]])
        W, K = ref.stencils(sens, dfk, nk, np.full(n, 6), knowns, c)
        lhs = (W * fk[None]).sum(-1) + (K * fi_in[None]).sum(-1)
        rhs = (fi_out[None] * c[:, None, :]).sum(-1)
        bound = ref.identity_bound(W, K, c, fk[None], fi_in[None], fi_out, 1.0)
        worst = max(worst, float((np.abs(lhs - rhs) / bound).max()))
    print("identity: worst |error| / (L eps scale) on the oracle = %.3f (constant %.1f)" % (worst, IDENTITY_CONST))
    assert worst <= IDENTITY_CONST
