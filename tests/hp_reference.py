"""Extended-precision reference for the weighted least-squares fits, independent of the oracle and of the original code.

Every fit is solved from its definition: minimise sum_k w_k (f_k - sum_s fi_s c_ks)^2 over the unknown slots s, the known
slots fixed, with c_ks = dx^a dy^b dz^c / (a! b! c!), dx = xk - xi, and w_k = 1 (WEIGHT_UNIFORM) or
1e-4 + (1 - 1e-4) (1 - sqrt(d2_k / max d2))^2 (WEIGHT_CENTER; impl.pyx / infra.pyx of the original).  The slot -> exponent
table comes from the slot names of the original (tests/golden/golden_defs.json, e.g. i3_XY2Z -> (1, 2, 1)), not from
the product or the oracle.

Arithmetic: the float64 inputs are dyadic rationals, so dx and the monomials are exact integers times powers of two and
the Gram matrix sum_k w_k c_kj c_km is formed exactly in integers (WEIGHT_CENTER: w_k rounded to 256 fractional bits).
Everything after that -- equilibration, the elimination of the knowns, the solve -- runs in mpmath at 60 digits.  Only
the eigenvalues of the equilibrated matrix S, which enter the tolerance and nothing else, are taken in float64.

Criterion (per case, per unknown slot j), with D = diag(a_jj^(-1/2)), S = D A D, y* = D^-1 fi*:

    |fi_j - fi*_j| / D_j  <=  C * g(nk) * eps * ||S^-1||_2 * (nr ||y*||_inf + ||f||_w)

where eps = 2^-53, g(nk) = nk, C = 8 (BOUND_C) and ||f||_w = sqrt(sum_k w_k m_k^2) with m_k = |f_k| + sum_{m known}
|fi_m c_km|, the magnitude of the data that enters the elimination of the knowns.  (The norm of the data AFTER the
elimination, which can cancel to nearly nothing, under-states the rounding of the elimination itself: with it the
oracle missed the bound tenfold on well-conditioned fits whose knowns carry most of the data.)  `ratio()` returns the
left side over g(nk) eps ||S^-1|| (nr ||y*|| + ||f||_w), i.e. a case passes at ratio <= BOUND_C.

C and g were fixed on the CPU from the oracle (the C restatement of the original's algorithm: normal equations,
iterated Ruiz scaling, dgetf2 / dgetrs) before any GPU run.  Over the geometry matrix (matrix_batches(): random,
lattice, one-sided, anisotropic, near-degenerate, duplicate, square and almost-square stencils at spacings 2^-20, 1,
2^10; dims 1-3, orders 0-4, both weightings, knowns none / F / random; smooth-plus-noise and polynomial data) the
oracle's worst ratio is 0.99, 1/8 of the threshold (tests/test_accuracy_hp.py asserts <= BOUND_C / 4).  The worst
cases are order-0 fits with three neighbours and WEIGHT_CENTER, where the weight formula's own rounding (1 - sqrt(.)
cancels near the farthest neighbour) is of the size of the solve's.  A
GPU case above the threshold is a defect to find, not a reason to raise C.

Evaluation (`hp_eval`, `eval_bound`): |value - exact| <= (no + 2 order + 2) eps sum |terms|; the oracle's evaluation
reaches 0.23 of that.
"""
from __future__ import annotations

import functools
import json
import math
import re
from pathlib import Path

import mpmath
import numpy as np

mp = mpmath.mp
DPS = 60
EPS = 2.0 ** -53
BOUND_C = 8.0
CENTER_FLOOR = 1e-4            # the double literal of the original (impl.pyx / infra.pyx)
_WBITS = 256                   # fractional bits of the WEIGHT_CENTER weights in the exact Gram matrix

WEIGHT_UNIFORM, WEIGHT_CENTER = 1, 2


def g(nk):
    return float(nk)


def _slot_exponents():
    defs = json.loads((Path(__file__).resolve().parent / "golden" / "golden_defs.json").read_text())
    out = {}
    for dim in (1, 2, 3):
        table = {}
        for name, idx in defs.items():
            m = re.fullmatch(r"i%d_([A-Z0-9]+)" % dim, name)
            if not m:
                continue
            e = [0, 0, 0]
            if m.group(1) != "F":
                for ax, p in re.findall(r"([XYZ])(\d?)", m.group(1)):
                    e["XYZ".index(ax)] += int(p or 1)
            table[int(idx)] = tuple(e)
        out[dim] = [table[s] for s in range(len(table))]
    return out


EXPONENTS = _slot_exponents()           # EXPONENTS[dim][slot] = (a, b, c)


def number_of_dofs(dim, order):
    return sum(1 for e in EXPONENTS[dim] if sum(e) <= order)


def _ifact(e):
    return math.factorial(e[0]) * math.factorial(e[1]) * math.factorial(e[2])


def _exact_offsets(xi, xk):
    """dx = xk - xi exactly: integers X (nk, dim) and the common exponent L, dx = X * 2^-L"""
    vals = [float(v) for v in np.ravel(xi)] + [float(v) for v in np.ravel(xk)]
    ratios = [v.as_integer_ratio() for v in vals]
    L = max(d.bit_length() - 1 for _, d in ratios)
    ints = [n << (L - (d.bit_length() - 1)) for n, d in ratios]
    dim = np.size(xi)
    Xi = ints[:dim]
    Xk = ints[dim:]
    return [[Xk[k * dim + m] - Xi[m] for m in range(dim)] for k in range(len(Xk) // dim)], L


def _mono(X, e):
    r = 1
    for m, p in enumerate(e):
        if p:
            r *= X[m] ** p
    return r


class HPCase:
    """one local fit: geometry, weights and the equilibrated normal matrix, factored once in extended precision"""

    def __init__(self, dim, order, knowns, wm, xi, xk):
        with mp.workdps(DPS):
            self._setup(dim, order, knowns, wm, xi, xk)

    def _setup(self, dim, order, knowns, wm, xi, xk):
        self.dim, self.order, self.wm = dim, order, wm
        xi = np.asarray(xi, np.float64).reshape(dim)
        xk = np.asarray(xk, np.float64).reshape(-1, dim)
        self.nk = nk = xk.shape[0]
        self.no = no = number_of_dofs(dim, order)
        self.E = E = EXPONENTS[dim][:no]
        self.known = [s for s in range(no) if knowns >> s & 1]
        self.unknown = [s for s in range(no) if not knowns >> s & 1]
        self.nr = nr = len(self.unknown)
        X, L = _exact_offsets(xi, xk)
        P = np.empty((nk, no), dtype=object)
        for k in range(nk):
            for s, e in enumerate(E):
                P[k, s] = _mono(X[k], e)
        # c_ks = P_ks * scale_s  (exact value)
        self.scale = [mp.ldexp(mp.mpf(1), -L * sum(e)) / _ifact(e) for e in E]
        if wm == WEIGHT_UNIFORM:
            W = [1] * nk
            self.w = [mp.mpf(1)] * nk
            wshift = 0
        else:
            d2 = [sum(v * v for v in X[k]) for k in range(nk)]
            dmax = max(d2)
            self.w = []
            for k in range(nk):
                t = 1 - mp.sqrt(mp.mpf(d2[k]) / mp.mpf(dmax))
                self.w.append(mp.mpf(CENTER_FLOOR) + (1 - mp.mpf(CENTER_FLOOR)) * t * t)
            W = [int(mp.nint(mp.ldexp(v, _WBITS))) for v in self.w]
            wshift = _WBITS
        self.c = [[mp.mpf(P[k, s]) * self.scale[s] for s in range(no)] for k in range(nk)]
        if nr == 0:
            return
        Pu = P[:, self.unknown]
        G = Pu.T.dot(Pu * np.array(W, dtype=object)[:, None])          # exact integers
        A = [[mp.ldexp(mp.mpf(G[j, m]), -wshift) * self.scale[self.unknown[j]] * self.scale[self.unknown[m]]
              for m in range(nr)] for j in range(nr)]
        self.D = [1 / mp.sqrt(A[j][j]) for j in range(nr)]
        S = [[self.D[j] * A[j][m] * self.D[m] for m in range(nr)] for j in range(nr)]
        lam = np.linalg.eigvalsh(np.array([[float(v) for v in r] for r in S]))
        self.inv_s = 1.0 / lam[0] if lam[0] > 0 else math.inf
        self.kappa = lam[-1] / lam[0] if lam[0] > 0 else math.inf
        self._lu = _lu(S)

    # ---- solves ---------------------------------------------------------------------------------------------
    def _reduced_data(self, fk, fi_known):
        """f'_k = f_k - sum_{m known} fi_m c_km"""
        fk = [mp.mpf(v) for v in fk]
        for m in self.known:
            v = mp.mpf(fi_known[m])
            for k in range(self.nk):
                fk[k] -= v * self.c[k][m]
        return fk

    def _data_magnitude(self, fk, fi_known):
        """|f_k| + sum_{m known} |fi_m c_km|: what the elimination of the knowns rounds (its result may cancel)"""
        out = [abs(mp.mpf(v)) for v in fk]
        for m in self.known:
            v = abs(mp.mpf(fi_known[m]))
            for k in range(self.nk):
                out[k] += v * abs(self.c[k][m])
        return out

    def fit(self, fk, fi_known=None):
        with mp.workdps(DPS):
            fi = [mp.mpf(0)] * self.no
            if fi_known is not None:
                for m in self.known:
                    fi[m] = mp.mpf(fi_known[m])
            if self.nr == 0:
                return dict(fi=fi, y=[], fw=mp.mpf(0))
            fr = self._reduced_data(fk, fi_known)
            b = [self.D[j] * mp.fsum(self.w[k] * self.c[k][s] * fr[k] for k in range(self.nk))
                 for j, s in enumerate(self.unknown)]
            y = _lu_solve(self._lu, b)
            for j, s in enumerate(self.unknown):
                fi[s] = self.D[j] * y[j]
            fw = mp.sqrt(mp.fsum(self.w[k] * fm ** 2 for k, fm in enumerate(self._data_magnitude(fk, fi_known))))
            return dict(fi=fi, y=y, fw=fw)

    def operator(self):
        """(dfk, dfkn): dfk[k, s] = d fi_s / d fk_k, dfkn[m, s] = d fi_s / d fi_known_m (unknown s; mpf; None elsewhere)"""
        with mp.workdps(DPS):
            dfk = [[None] * self.no for _ in range(self.nk)]
            ys = []
            for k in range(self.nk):
                b = [self.D[j] * self.w[k] * self.c[k][s] for j, s in enumerate(self.unknown)]
                y = _lu_solve(self._lu, b) if self.nr else []
                ys.append(y)
                for j, s in enumerate(self.unknown):
                    dfk[k][s] = self.D[j] * y[j]
            dfkn = [[None] * self.no for _ in range(self.no)]
            for m in self.known:
                for s in self.unknown:
                    dfkn[m][s] = -mp.fsum(dfk[k][s] * self.c[k][m] for k in range(self.nk))
            self._op_y = ys
            return dfk, dfkn

    # ---- criterion ------------------------------------------------------------------------------------------
    def ratio(self, sol, fi_got):
        """max over the unknown slots of |fi_j - fi*_j| / D_j over g(nk) eps ||S^-1|| (nr ||y*|| + ||f||_w);
        the case passes at <= BOUND_C.  NaN / inf in fi_got give inf."""
        if self.nr == 0:
            return 0.0
        with mp.workdps(DPS):
            ymax = max(abs(v) for v in sol["y"])
            den = g(self.nk) * EPS * self.inv_s * float(self.nr * ymax + sol["fw"])
            worst = 0.0
            for j, s in enumerate(self.unknown):
                v = float(fi_got[s])
                if not math.isfinite(v):
                    return math.inf
                e = float(abs(mp.mpf(v) - sol["fi"][s]) / self.D[j])
                worst = max(worst, e / den if den > 0 else (0.0 if e == 0 else math.inf))
            return worst

    def operator_ratio(self, dfk, sens_got):
        """the same criterion for every entry of the operator: column k is the fit of the data e_k (||e_k||_w = sqrt(w_k))"""
        if self.nr == 0:
            return 0.0
        worst = 0.0
        with mp.workdps(DPS):
            for k in range(self.nk):
                ymax = max(abs(v) for v in self._op_y[k])
                den = g(self.nk) * EPS * self.inv_s * float(self.nr * ymax + mp.sqrt(self.w[k]))
                for j, s in enumerate(self.unknown):
                    v = float(sens_got[k, s])
                    if not math.isfinite(v):
                        return math.inf
                    e = float(abs(mp.mpf(v) - dfk[k][s]) / self.D[j])
                    worst = max(worst, e / den if den > 0 else (0.0 if e == 0 else math.inf))
        return worst


def _lu(S):
    """Gaussian elimination with partial pivoting (mpf)"""
    n = len(S)
    a = [list(r) for r in S]
    perm = list(range(n))
    for p in range(n):
        q = max(range(p, n), key=lambda i: abs(a[i][p]))
        if q != p:
            a[p], a[q] = a[q], a[p]
            perm[p], perm[q] = perm[q], perm[p]
        d = a[p][p]
        for i in range(p + 1, n):
            l = a[i][p] / d
            a[i][p] = l
            ri, rp = a[i], a[p]
            for m in range(p + 1, n):
                ri[m] -= l * rp[m]
    return a, perm


def _lu_solve(f, b):
    a, perm = f
    n = len(a)
    y = [b[perm[i]] for i in range(n)]
    for i in range(n):
        y[i] -= mp.fsum(a[i][m] * y[m] for m in range(i))
    for i in range(n - 1, -1, -1):
        y[i] = (y[i] - mp.fsum(a[i][m] * y[m] for m in range(i + 1, n))) / a[i][i]
    return y


def hp_fit(dim, order, knowns, wm, xi, xk, fk, fi_known=None):
    """exact solution of one fit: dict(fi, D, y, inv_s (||S^-1||_2), kappa, fw (||f||_w), nr, case)"""
    c = HPCase(dim, order, knowns, wm, xi, xk)
    sol = c.fit(fk, fi_known)
    return dict(sol, D=getattr(c, "D", []), inv_s=getattr(c, "inv_s", 0.0), kappa=getattr(c, "kappa", 1.0),
                nr=c.nr, case=c)


def hp_operator(dim, order, knowns, wm, xi, xk):
    """exact d fi / d fk (what `sens` returns) and d fi / d fi_known"""
    return HPCase(dim, order, knowns, wm, xi, xk).operator()


def bound(ref, nk):
    """per unknown slot: the largest admissible |fi_j - fi*_j| (BOUND_C g(nk) eps ||S^-1|| (nr ||y*|| + ||f||_w) D_j)"""
    if ref["nr"] == 0:
        return []
    with mp.workdps(DPS):
        ymax = max(abs(v) for v in ref["y"])
        t = BOUND_C * g(nk) * EPS * ref["inv_s"] * float(ref["nr"] * ymax + ref["fw"])
        return [t * float(d) for d in ref["D"]]


def hp_eval(dim, xi, fi, x, diff):
    """exact value of derivative `diff` (a slot index) of the model sum_s fi_s c_s(x - xi) at x, and sum |terms|"""
    with mp.workdps(DPS):
        no = len(fi)
        if diff >= no:
            return mp.mpf(0), 0.0
        E = EXPONENTS[dim]
        pd = E[diff]
        X, L = _exact_offsets(xi, x)
        acc, mag = mp.mpf(0), mp.mpf(0)
        for s in range(no):
            e = tuple(E[s][m] - pd[m] for m in range(3))
            if min(e) < 0:
                continue
            t = mp.mpf(float(fi[s])) * mp.ldexp(mp.mpf(_mono(X[0], e)), -L * sum(e)) / _ifact(e)
            acc += t
            mag += abs(t)
        return acc, float(mag)


EVAL_C = 1.0


def eval_bound(dim, order, mag):
    """admissible |interpolate - exact| for a model of the given order: EVAL_C (no + 2 order + 2) eps sum |terms|"""
    return EVAL_C * (number_of_dofs(dim, order) + 2 * order + 2) * EPS * mag


# ---- the geometry matrix ----------------------------------------------------------------------------------------
GEOMETRIES = ("random", "lattice", "one_sided", "anisotropic", "near_degenerate", "duplicates")
SCALES = (2.0 ** -20, 2.0 ** 10, 1.0)           # interleaved: neighbouring cases differ by 2^30, 2^10 and 2^20
T_SHIFT = 2.0 ** 12
FRAC_BITS = 20                                  # stencil offsets are multiples of 2^-20 in [-1, 1]
KAPPA_EPS_MAX = 1e-3                            # cases with kappa(S) eps above this are too close to singular to judge


def _dyadic(rng, shape, lo=-1.0, hi=1.0):
    q = 2 ** FRAC_BITS
    return rng.integers(int(lo * q), int(hi * q) + 1, shape) / q


def _lattice(dim, nk):
    r = 1
    while (2 * r + 1) ** dim < 4 * nk:
        r += 1
    g1 = np.arange(-r, r + 1)
    pts = np.array(np.meshgrid(*([g1] * dim), indexing="ij")).reshape(dim, -1).T
    key = [tuple([int((p * p).sum())] + list(p)) for p in pts]
    pts = pts[sorted(range(len(pts)), key=lambda i: key[i])][:nk].astype(np.float64)
    span = np.abs(pts).max()
    return pts / 2.0 ** math.ceil(math.log2(span)) if span > 0 else pts


def stencil(geom, dim, nk, rng):
    """neighbour offsets rel in [-1, 1]^dim, multiples of 2^-20"""
    if geom == "lattice":
        return _lattice(dim, nk)
    if geom == "one_sided":
        return _dyadic(rng, (nk, dim), 0.0, 1.0)
    rel = _dyadic(rng, (nk, dim))
    if geom == "anisotropic":
        rel[:, dim - 1] *= 2.0 ** -10
    elif geom == "near_degenerate":       # within 2^-14 (about 1e-4) of a line (2D) / plane (3D)
        t = _dyadic(rng, (nk,)) * 2.0 ** -14
        if dim == 2:
            rel[:, 1] = rel[:, 0] / 2 + t
        elif dim == 3:
            rel[:, 2] = (rel[:, 0] + rel[:, 1]) / 4 + t
    elif geom == "duplicates":             # two neighbours at the same place, one exactly at xi
        rel[1] = rel[0]
        rel[2] = 0.0
    # back onto the 2^-20 grid, so that xk = T + h rel stays exact at T = 2^12, h = 2^-20
    return np.round(rel * 2 ** FRAC_BITS) / 2 ** FRAC_BITS


def geometries_for(dim):
    return [gm for gm in GEOMETRIES if not (dim == 1 and gm in ("anisotropic", "near_degenerate"))]


def smooth(rel):
    r = np.zeros((rel.shape[0], 3))
    r[:, :rel.shape[1]] = rel
    return np.sin(1.3 * r[:, 0] + 0.4) * np.cos(0.7 * r[:, 1] - 0.2) * np.exp(0.3 * r[:, 2])


def random_mask(dim, order, rng):
    no = number_of_dofs(dim, order)
    if no < 2:
        return 0
    pick = rng.choice(np.arange(1, no), 1 if no == 2 else 2, replace=False) if no > 2 else [1]
    return int(sum(1 << int(s) for s in pick))


def default_nk(dim, order):
    no = number_of_dofs(dim, order)
    return {(3, 4): 60, (3, 3): 40, (2, 4): 30}.get((dim, order), max(no + 2, (8 * no + 4) // 5))


class Batch:
    """cases of one (dim, order, knowns, wm, nk) configuration, one per (geometry, spacing), with two data sets:
    smooth + noise (`fk`) and a polynomial of degree <= order (`fkp`, whose exact fit is close to `coef`)"""

    def __init__(self, dim, order, knowns, wm, nk=None, geoms=None, seed=0, reps=1, label=None):
        rng = np.random.default_rng(seed)
        self.dim, self.order, self.wm = dim, order, wm
        self.no = no = number_of_dofs(dim, order)
        self.nk = nk = nk or default_nk(dim, order)
        self.knowns = knowns & ((1 << no) - 1)
        geoms = geoms or geometries_for(dim)
        self.geom, self.h, rels = [], [], []
        for _ in range(reps):
            for gm in geoms:
                for h in SCALES:
                    self.geom.append(label or gm)
                    self.h.append(h)
                    rels.append(stencil(gm, dim, nk, rng))
        self.n = n = len(rels)
        self.rel = np.array(rels)
        self.h = np.array(self.h)
        deg = np.array([sum(e) for e in EXPONENTS[dim][:no]])
        self.fk = np.array([smooth(r) for r in rels]) + 1e-3 * rng.standard_normal((n, nk))
        self.coef = rng.uniform(-1, 1, (n, no)) / self.h[:, None] ** deg[None, :]
        mono = np.array([[[np.prod(r[k] ** np.array(e[:dim])) / _ifact(e) for e in EXPONENTS[dim][:no]]
                          for k in range(nk)] for r in rels])                 # monomials of rel (unit spacing)
        self.fkp = np.einsum("nks,ns->nk", mono, self.coef * self.h[:, None] ** deg[None, :])
        self.fi0 = 0.1 * rng.standard_normal((n, no)) / self.h[:, None] ** deg[None, :]
        self.fi0[:, 0] = smooth(np.zeros((1, dim)))[0]
        self.fi0p = self.coef.copy()
        self.meta = (np.full(n, nk, np.int32), np.full(n, order, np.int32), np.full(n, self.knowns, np.int64),
                     np.full(n, wm, np.int32))
        self._ref = None

    def place(self, T=0.0):
        """(xi, xk) with xi = T + 3 h i and xk = xi + h rel: dyadic, so that xk - xi = h rel exactly"""
        xi = T + 3.0 * self.h[:, None] * np.arange(self.n)[:, None] * np.ones((1, self.dim))
        xk = xi[:, None, :] + self.h[:, None, None] * self.rel
        assert np.array_equal(xk - xi[:, None, :], self.h[:, None, None] * self.rel)
        if self.dim == 1:
            return np.ascontiguousarray(xi[:, 0]), np.ascontiguousarray(xk[:, :, 0])
        return np.ascontiguousarray(xi), np.ascontiguousarray(xk)

    def reference(self):
        """per case: the HPCase and the exact fits of both data sets (computed once)"""
        if self._ref is None:
            xi, xk = self.place(0.0)
            xi2, xk2 = xi.reshape(self.n, self.dim), xk.reshape(self.n, self.nk, self.dim)
            self._ref = []
            for i in range(self.n):
                c = HPCase(self.dim, self.order, self.knowns, self.wm, xi2[i], xk2[i])
                self._ref.append((c, c.fit(self.fk[i], self.fi0[i]), c.fit(self.fkp[i], self.fi0p[i])))
        return self._ref

    def judged(self, i):
        c = self.reference()[i][0]
        return c.nr > 0 and c.kappa * EPS <= KAPPA_EPS_MAX

    def ratios(self, fi, poly=False):
        """per-case ratio (NaN for cases not judged)"""
        out = np.full(self.n, np.nan)
        for i, (c, s, sp) in enumerate(self.reference()):
            if self.judged(i):
                out[i] = c.ratio(sp if poly else s, fi[i])
        return out


def config_matrix(dims=(1, 2, 3), orders=(0, 1, 2, 3, 4)):
    """(dim, order, knowns, wm) of the geometry matrix: knowns none, F and a random mask (order 0: none)"""
    out = []
    rng = np.random.default_rng(11)
    for dim in dims:
        for order in orders:
            masks = [0] if order == 0 else sorted({0, 1, random_mask(dim, order, rng)})
            for wm in (WEIGHT_UNIFORM, WEIGHT_CENTER):
                for kn in masks:
                    out.append((dim, order, kn, wm))
    return out


def square_batches(dims=(1, 2, 3), orders=(1, 2, 3, 4), seed=0):
    """random stencils with nk = nr ("square") and nk = nr + 1 ("almost_square"), knowns none"""
    out = []
    for dim in dims:
        for order in orders:
            no = number_of_dofs(dim, order)
            for wm in (WEIGHT_UNIFORM, WEIGHT_CENTER):
                for extra, label in ((0, "square"), (1, "almost_square")):
                    out.append(Batch(dim, order, 0, wm, nk=no + extra, geoms=("random",), reps=2, label=label,
                                     seed=seed + 100 * dim + 10 * order + 2 * extra + wm))
    return out


@functools.lru_cache(maxsize=None)
def matrix_batches(dims=(1, 2, 3), orders=(0, 1, 2, 3, 4), seed=0):
    """the geometry matrix: one Batch per configuration of config_matrix(), then the square ones"""
    out = [Batch(*cfg, seed=seed + i) for i, cfg in enumerate(config_matrix(dims, orders))]
    return tuple(out + square_batches(dims, [o for o in orders if o > 0], seed))
