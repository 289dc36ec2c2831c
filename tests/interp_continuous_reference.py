"""Host reference for the continuous-mode interpolation operators (ExpertSolver.interp_stencils / .interp_operator with
mode='continuous'): the definitions of include/wlsqm_b200.h restated in numpy.

Pairs: the origins xi[m] with d2 <= r*r, d2 the sum over the axes in axis order of (xi[m][d] - x[q][d])^2, every operation
a separately rounded float64 one (the ball rule of wlsqm_grid_ball_*); non-finite origins never, non-finite queries no
models.  Weights: w = (1 - sqrt(d2 / r2))^2, S = the sum of w in ascending m from +0, alpha = w / S.  A pair's coefficient
rows are alpha * c_q (tests/interp_operator_reference.py), one rounded multiply per entry.  Python floats and numpy
elementwise operations round every operation on its own, so these are bitwise the device's values.
"""
from __future__ import annotations

import math

import numpy as np

import interp_operator_reference as iref


def ball_d2(xi, xq):
    """d2 of one query against every origin by the ball rule: (n,)"""
    d2 = np.zeros(len(xi))
    for d in range(xi.shape[1]):
        dd = xi[:, d] - xq[d]
        d2 = d2 + dd * dd
    return d2


def pairs(xi, x, r):
    """(pair_ptr int64 (nx + 1,), J int64 (npairs,), d2 of each pair) by the ball rule"""
    xi = np.asarray(xi, np.float64).reshape(len(xi), -1)
    x = np.asarray(x, np.float64).reshape(len(x), xi.shape[1])
    finite = np.isfinite(xi).all(1)
    r2 = r * r
    ptr, J, D2 = [0], [], []
    for q in range(len(x)):
        if np.isfinite(x[q]).all():
            d2 = ball_d2(xi, x[q])
            m = np.flatnonzero(finite & (d2 <= r2))
            J.extend(m.tolist())
            D2.extend(d2[m].tolist())
        ptr.append(len(J))
    return np.array(ptr, np.int64), np.array(J, np.int64), np.array(D2, np.float64)


def weights(pair_ptr, d2, r):
    """(alpha (npairs,), w (npairs,), S (nx,)): separately rounded, S summed in pair order from +0"""
    r2 = r * r
    tmp = [1.0 - math.sqrt(v / r2) for v in d2.tolist()]
    w = np.array([t * t for t in tmp], np.float64)
    alpha = np.empty_like(w)
    S = np.zeros(len(pair_ptr) - 1)
    for q in range(len(pair_ptr) - 1):
        acc = 0.0
        for p in range(pair_ptr[q], pair_ptr[q + 1]):
            acc = acc + float(w[p])
        S[q] = acc
        for p in range(pair_ptr[q], pair_ptr[q + 1]):
            alpha[p] = float(w[p]) / acc if acc != 0.0 else math.nan
    return alpha, w, S


def pair_rows(dim, coeffs, x, xi, pair_ptr, J, alpha):
    """c_qm (npairs, nops, maxno) = alpha * c_q at the offset x[q] - xi[J[p]]"""
    c = np.atleast_2d(np.asarray(coeffs, np.float64))
    x = np.asarray(x, np.float64).reshape(-1, dim)
    xi = np.asarray(xi, np.float64).reshape(-1, dim)
    out = np.empty((len(J),) + c.shape)
    for q in range(len(pair_ptr) - 1):
        for p in range(pair_ptr[q], pair_ptr[q + 1]):
            out[p] = alpha[p] * iref.coefficient_rows_at(dim, c, x[q] - xi[J[p]])
    return out


def csr(W, K, hoods, nk, knowns, pair_ptr, J, center=None):
    """(rowptr, col, values (nops, nnz), K with the folded column zeroed): row q merges its pairs' candidates -- per pair
    (ascending m) the neighbours in ascending k, then the folded known-F weight at column center + m -- with each column
    summed in candidate order from +0"""
    nops = W.shape[0]
    K = K.copy()
    rowptr, cols, vals = [0], [], []
    for q in range(len(pair_ptr) - 1):
        row = {}
        for p in range(pair_ptr[q], pair_ptr[q + 1]):
            m = int(J[p])
            cand = [(int(hoods[m][k]), W[:, p, k]) for k in range(int(nk[m]))]
            if center is not None and int(knowns[m]) & 1:
                cand.append((center + m, K[:, p, 0].copy()))
                K[:, p, 0] = 0.0
            for col, v in cand:
                row[col] = (row[col] if col in row else np.zeros(nops)) + v
        for col in sorted(row):
            cols.append(col)
            vals.append(row[col])
        rowptr.append(len(cols))
    values = np.array(vals).T.reshape(nops, len(cols)) if cols else np.zeros((nops, 0))
    return np.array(rowptr, np.int64), np.array(cols, np.int64), values, K
