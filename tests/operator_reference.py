"""Host reference for the operator export (ExpertSolver.stencils / .operator): the definitions of
include/wlsqm_b200.h restated in numpy, from a solver's `sens` (d fi / d fk, impl.pyx:769-779) and its known-value
weights (d fi / d fi_known), plus the neighbour lists.

Sums run in the order the definitions fix: W over the slots in ascending order from 0, K the same plus c[m] last;
CSR values per column in ascending k starting from the first entry, the folded known-F weight added last.  With one-hot
coefficients every product is exact, so the GPU export must match these bit for bit.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp


def known_weights_from_solves(solve, ncases, maxno, nos, knowns):
    """d fi[s] / d fi_known[m] for every case: one solve with fk = 0 per known slot m, unit value there.
    ``solve(fi_in) -> fi_out`` runs the solver on fk = 0.  Returns (ncases, maxno [m], maxno [s])."""
    out = np.zeros((ncases, maxno, maxno))
    for m in range(maxno):
        has = np.array([m < nos[i] and (int(knowns[i]) >> m) & 1 for i in range(ncases)], dtype=bool)
        if not has.any():
            continue
        fi = np.zeros((ncases, maxno))
        fi[has, m] = 1.0
        fo = solve(fi)
        out[has, m, :] = fo[has, :]
    return out


def stencils(sens, dfk, nk, nos, knowns, c):
    """W (nops, n, maxnk), K (nops, n, maxno) from sens (n, maxnk, maxno) and dfk = known_weights_from_solves(...)."""
    c = np.atleast_2d(np.asarray(c, np.float64))
    nops, maxno = c.shape
    n, maxnk = sens.shape[0], sens.shape[1]
    W = np.zeros((nops, n, maxnk))
    K = np.zeros((nops, n, maxno))
    for i in range(n):
        no, kn = int(nos[i]), int(knowns[i])
        unk = [s for s in range(no) if not (kn >> s) & 1]
        for o in range(nops):
            used = [s for s in unk if c[o, s] != 0.0]
            acc = np.zeros(int(nk[i]))
            for s in used:
                acc = c[o, s] * sens[i, :nk[i], s] + acc
            W[o, i, :nk[i]] = acc
            for m in range(no):
                if (kn >> m) & 1:
                    a = 0.0
                    for s in used:
                        a = c[o, s] * dfk[i, m, s] + a
                    K[o, i, m] = a + c[o, m]
    return W, K


def csr(W, K, hoods, nk, knowns, npoints, center=None):
    """(rowptr, col, values (nops, nnz), K with the folded column zeroed) of the global operator."""
    nops, n = W.shape[0], W.shape[1]
    K = K.copy()
    rowptr = [0]
    cols, vals = [], []
    for i in range(n):
        row = {}
        for k in range(int(nk[i])):
            p = int(hoods[i][k])
            if p in row:
                row[p] = row[p] + W[:, i, k]
            else:
                row[p] = W[:, i, k].copy()
        if center is not None and int(knowns[i]) & 1:
            f = center + i
            row[f] = (row[f] + K[:, i, 0]) if f in row else K[:, i, 0].copy()
            K[:, i, 0] = 0.0
        for p in sorted(row):
            cols.append(p)
            vals.append(row[p])
        rowptr.append(len(cols))
    values = np.array(vals).T.reshape(nops, len(cols)) if cols else np.zeros((nops, 0))
    return np.array(rowptr, np.int64), np.array(cols, np.int64), values, K


def scipy_matrices(rowptr, col, values, n, npoints):
    return [sp.csr_array((values[o], col, rowptr), shape=(n, npoints)) for o in range(values.shape[0])]


def identity_bound(W, K, c, f_hoods, fi_in, fi_out, const):
    """|sum_s c fi_out - (W . fk + K . fi_in)| <= const * (nk + 2 no) * eps * (|W| . |fk| + |K| . |fi_in| + |c| . |fi_out|):
    the error of two summations of that length over the magnitudes that enter them (DESIGN.md section 6)."""
    eps = np.finfo(np.float64).eps
    n = W.shape[1]
    L = W.shape[2] + 2 * K.shape[2]
    scale = (np.abs(W) * np.abs(f_hoods)).sum(-1) + (np.abs(K) * np.abs(fi_in)).sum(-1) + \
        (np.abs(c)[:, None, :] * np.abs(fi_out)[None]).sum(-1)
    return const * L * eps * scale
