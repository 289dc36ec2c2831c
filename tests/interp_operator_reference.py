"""Host reference for the interpolation operators (ExpertSolver.interp_stencils / .interp_operator): the definitions
of include/wlsqm_b200.h restated in numpy.

For query q with model m = I[q] and offset h = x[q] - xi[m] per axis, the Taylor terms t[0] = 1, t[n] = t[n-1] * st[n-1]
with st = (h, 0.5*h, (1.0/3.0)*h, 0.25*h); T_D(s) = (tx[a-p] * ty[b-r]) * tz[c-u] for slot s = (a, b, c) and derivative
slot D = (p, r, u) where a >= p, b >= r, c >= u, else 0; and the coefficient rows c_q[o][s] = sum over D ascending with
coeffs[o][D] != 0 of coeffs[o][D] * T_D(s).  Every product and sum is a separately rounded float64 operation (numpy and
Python floats do not contract), so these c_q are bitwise those of the GPU kernel.  A row of the operators is then the
node operator of model m (tests/operator_reference.py) with c_q in place of the coefficients.
"""
from __future__ import annotations

import numpy as np

from hp_reference import EXPONENTS
import operator_reference as opref


def taylor_terms(h):
    """t[0..4] of one axis"""
    h = float(h)
    st = (h, 0.5 * h, (1.0 / 3.0) * h, 0.25 * h)
    t = [1.0]
    for n in range(1, 5):
        t.append(t[-1] * st[n - 1])
    return t


def T_matrix(dim, h, maxno):
    """T[D][s] for D, s < maxno at the offset h (dim values)"""
    h = list(np.atleast_1d(np.asarray(h, np.float64))) + [0.0] * 3
    tx, ty, tz = taylor_terms(h[0]), taylor_terms(h[1]), taylor_terms(h[2])
    ex = EXPONENTS[dim]
    T = np.zeros((maxno, maxno))
    for D in range(maxno):
        p, r, u = ex[D]
        for s in range(maxno):
            a, b, c = ex[s]
            if a >= p and b >= r and c >= u:
                T[D, s] = (tx[a - p] * ty[b - r]) * tz[c - u]
    return T


def coefficient_rows_at(dim, coeffs, h):
    """c_q (nops, maxno) at offset h: sums over D ascending from +0, zero coefficients skipped"""
    c = np.atleast_2d(np.asarray(coeffs, np.float64))
    nops, maxno = c.shape
    T = T_matrix(dim, h, maxno)
    out = np.zeros((nops, maxno))
    for o in range(nops):
        for s in range(maxno):
            acc = 0.0
            for D in range(maxno):
                if c[o, D] != 0.0:
                    acc = acc + float(c[o, D]) * float(T[D, s])
            out[o, s] = acc
    return out


def query_rows(dim, coeffs, x, xi, I, ncases):
    """c_q for every query: (nx, nops, maxno); NaN rows where I is outside [0, ncases)"""
    c = np.atleast_2d(np.asarray(coeffs, np.float64))
    x = np.asarray(x, np.float64).reshape(len(I), dim)
    xi = np.asarray(xi, np.float64).reshape(-1, dim)
    out = np.full((len(I),) + c.shape, np.nan)
    for q, m in enumerate(np.asarray(I)):
        if 0 <= m < ncases:
            out[q] = coefficient_rows_at(dim, c, x[q] - xi[m])
    return out


def stencils(sens, dfk, nk, nos, knowns, cq, I):
    """W (nops, nx, maxnk), K (nops, nx, maxno) of the queries by the node reference with c_q per query (host sums:
    exact only where every product is, see operator_reference); queries without a model: W 0, K NaN"""
    nx, nops, maxno = cq.shape
    n = sens.shape[0]
    W = np.zeros((nops, nx, sens.shape[1]))
    K = np.full((nops, nx, maxno), np.nan)
    for q, m in enumerate(np.asarray(I)):
        if 0 <= m < n:
            w, k = opref.stencils(sens[m:m + 1], dfk[m:m + 1], nk[m:m + 1], nos[m:m + 1], knowns[m:m + 1], cq[q])
            W[:, q], K[:, q] = w[:, 0], k[:, 0]
    return W, K


def csr(W, K, hoods, nk, knowns, npoints, I, ncases, center=None):
    """(rowptr, col, values (nops, nnz), K with the folded column zeroed) of the interpolation operator: row q merges
    W[:, q] over the neighbour list of model I[q] in ascending k, the known-F weight added last to column center + I[q];
    a query without a model has an empty row."""
    nops, nx = W.shape[0], W.shape[1]
    K = K.copy()
    rowptr = [0]
    cols, vals = [], []
    for q in range(nx):
        m = int(I[q])
        row = {}
        if 0 <= m < ncases:
            for k in range(int(nk[m])):
                p = int(hoods[m][k])
                row[p] = (row[p] + W[:, q, k]) if p in row else W[:, q, k].copy()
            if center is not None and int(knowns[m]) & 1:
                f = center + m
                row[f] = (row[f] + K[:, q, 0]) if f in row else K[:, q, 0].copy()
                K[:, q, 0] = 0.0
        for p in sorted(row):
            cols.append(p)
            vals.append(row[p])
        rowptr.append(len(cols))
    values = np.array(vals).T.reshape(nops, len(cols)) if cols else np.zeros((nops, 0))
    return np.array(rowptr, np.int64), np.array(cols, np.int64), values, K


def identity_bound(cq_abs, sens_q, dfk_q, fk_q, fi_in_q, fi_out_q, const):
    """|sum_D c[D] d^D f(x_q) - (W . fk + K . fi_in)| <= const * L * eps * scale with L = max nk + 3 max no: the error of
    the solve (the magnitudes entering each fi[s], |sens| . |fk| + |dfk| . |fi_in| + |fi_in|), of the Taylor sum
    (|fi_out|) and of the contraction, weighted per slot by |c_q| (c_q of |coeffs| at |h|, no cancellation).
    cq_abs (nops, nx, no); the rest per query: sens_q (nx, nk, no), dfk_q (nx, no [known], no), fk_q (nx, nk),
    fi_in_q / fi_out_q (nx, no)."""
    eps = np.finfo(np.float64).eps
    L = sens_q.shape[1] + 3 * sens_q.shape[2]
    mag = np.einsum("qks,qk->qs", np.abs(sens_q), np.abs(fk_q)) + np.einsum("qts,qt->qs", np.abs(dfk_q), np.abs(fi_in_q)) \
        + np.abs(fi_in_q) + np.abs(fi_out_q)
    return const * L * eps * (cq_abs * mag[None]).sum(-1)
