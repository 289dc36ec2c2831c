"""GPU tests of ExpertSolver.interpolate_fields (csrc/wlsqm_interp_fields.cu): caller-held solutions of several fields
evaluated at query points in one pass.

The contract is per-field equality: out[j] must be bit for bit what interpolate() returns on a solver whose last solve()
produced fi[j] -- here the same solver after solve(fk[j], fi[j]) -- while the field solutions come from solve_fields.
Beyond self-consistency, random fi that no solve produced (NaN in the slots a model does not have) are checked against
a numpy evaluation of the Taylor model and of the continuous-mode weighted average (expert.pyx:898-985).
"""
import ctypes as C

import numpy as np
import pytest
from scipy.spatial import cKDTree

import wlsqm_b200 as w
from wlsqm_b200 import _lib
from wlsqm_b200.fitter import defs
from interp_operator_reference import T_matrix
from test_gpu_operator import _batch, _solver
from test_gpu_solve_fields import _data, _dev, _eq

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _queries(b, nq=300, seed=0):
    """points inside and a little outside the cloud, a few exactly at origins"""
    rng = np.random.default_rng(seed)
    dim = b["dim"]
    x = rng.uniform(-0.05, 1.05, size=(nq, dim))
    x[:10] = b["xi"][:10]
    return x[:, 0].copy() if dim == 1 else x


def _nearest(b, x):
    return cKDTree(b["xi"]).query(x.reshape(len(x), -1), k=1)[1].astype(np.int64)


def _refs(s, fk, fi0, x, I, diffs, mode="nearest", r=None):
    """per field: solve(fk[j], fi[j]) then interpolate(x, ...) for every diff -> {diff: (nf, nx[, maxno])}, and the fi"""
    outs = {d: [] for d in diffs}
    fis = []
    for j in range(fi0.shape[0]):
        fi = fi0[j].copy()
        s.solve(fk[j], fi)
        fis.append(fi)
        for d in diffs:
            outs[d].append(s.interpolate(x, mode=mode, r=r, diff=d, I=I)[0])
    return {d: np.stack(v) for d, v in outs.items()}, np.stack(fis)


def _host(a):
    return a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)


CFGS = [(1, [4], 10), (2, [4], 20), (3, [4], 40), (2, [2, 3, 4], 20), (3, [0, 2, 3, 4], 40)]


@pytest.mark.parametrize("algo", [defs.ALGO_BASIC, defs.ALGO_ITERATIVE])
@pytest.mark.parametrize("knowns_mode", [0, "F", "rand"])
@pytest.mark.parametrize("dim,orders,k", CFGS)
def test_nearest_equals_single_fields(dim, orders, k, knowns_mode, algo):
    """every slot and 'all', nf = 1, 2, 3, 8 and 17 (more than one pass), fi from solve_fields"""
    b = _batch(dim, orders, k, knowns_mode)
    s = _solver(b, algorithm=algo, max_iter=3)
    s.prep_interpolate()
    nf = 17
    _, fk, fi0 = _data(b, s, nf)
    x = _queries(b)
    I = _nearest(b, x)
    I[::37] = -1                                                  # no model: NaN
    diffs = list(range(s._maxno)) + ['all']
    ref, fis = _refs(s, fk, fi0, x, I, diffs)
    fi = fi0.copy()
    s.solve_fields(fk, fi)
    assert _eq(fi, fis)
    dev = _dev()
    fi_t = torch.as_tensor(fi, device=dev)
    for n in (1, 2, 3, 8, 17):
        for d in diffs:
            out, I_out = s.interpolate_fields(x, fi[:n], diff=d, I=I)
            assert _eq(out, ref[d][:n]), (n, d)
            assert np.array_equal(I_out, I)
        out, _ = s.interpolate_fields(torch.as_tensor(x, device=dev), fi_t[:n], diff=n % s._maxno,
                                      I=torch.as_tensor(I, device=dev))
        assert _eq(out, ref[n % s._maxno][:n])
    # 'all' with device outputs: slots >= no_{I[q]} are zeros (interpolate leaves them unwritten on the device)
    out, _ = s.interpolate_fields(torch.as_tensor(x, device=dev), fi_t, diff='all', I=torch.as_tensor(I, device=dev))
    assert _eq(out, ref['all'])
    # fields-inner fi, device and host: dense rows are compacted pass by pass (17 fields: several passes)
    inner = np.ascontiguousarray(fi.transpose(1, 0, 2))
    inner_t = torch.as_tensor(inner, device=dev).permute(1, 0, 2)
    for d in (0, s._maxno - 1, 'all'):
        assert _eq(s.interpolate_fields(torch.as_tensor(x, device=dev), inner_t, diff=d, I=torch.as_tensor(I, device=dev))[0],
                   ref[d])
        assert _eq(s.interpolate_fields(x, inner.transpose(1, 0, 2), diff=d, I=I)[0], ref[d])


@pytest.mark.parametrize("dim,orders,k", [(1, [4], 10), (2, [4], 20), (3, [2, 3, 4], 40)])
def test_continuous_equals_single_fields(dim, orders, k):
    b = _batch(dim, orders, k, "rand", seed=3)
    s = _solver(b, algorithm=defs.ALGO_ITERATIVE, max_iter=3)
    s.prep_interpolate()
    nf = 11
    _, fk, fi0 = _data(b, s, nf, seed=4)
    x = _queries(b, seed=5)
    x[-5:] = 3.0                                                  # no model within r: NaN
    fi = fi0.copy()
    s.solve_fields(fk, fi)
    dev = _dev()
    diffs = [0, 1, s._maxno - 1]
    for r in (0.03, 0.08, 0.2):
        ref, _ = _refs(s, fk, fi0, x, None, diffs, mode="continuous", r=r)
        for d in diffs:
            out, I_out = s.interpolate_fields(x, fi, mode="continuous", r=r, diff=d)
            assert I_out.item() is None
            assert _eq(out, ref[d])
            assert np.isnan(out[:, -5:]).all()
            for n in (1, 2, 3, 8):
                out, _ = s.interpolate_fields(torch.as_tensor(x, device=dev), torch.as_tensor(fi[:n], device=dev),
                                              mode="continuous", r=r, diff=d)
                assert _eq(out, ref[d][:n])


def _taylor(dim, fi_m, no, h, D):
    T = T_matrix(dim, h, fi_m.shape[0])
    return float(np.dot(T[D, :no], fi_m[:no]))


@pytest.mark.parametrize("dim,orders,k", [(2, [2, 3, 4], 20), (3, [1, 4], 40)])
def test_arbitrary_fi_against_numpy(dim, orders, k):
    """random fi, NaN in slots >= no_i and in padding columns: the numpy Taylor model and the continuous average"""
    b = _batch(dim, orders, k, 0, seed=6)
    s = _solver(b)
    s.prep_interpolate()
    n, maxno, nf = len(b["nk"]), s._maxno, 3
    rng = np.random.default_rng(7)
    fi = np.full((nf, n, maxno + 2), np.nan)
    for i in range(n):
        fi[:, i, :b["nos"][i]] = rng.standard_normal((nf, b["nos"][i]))
    x = _queries(b, nq=120, seed=8)
    I = _nearest(b, x)
    for D in (0, 1, maxno - 1):
        out, _ = s.interpolate_fields(x, fi, diff=D, I=I)
        for q in range(len(x)):
            m = I[q]
            for j in range(nf):
                want = _taylor(dim, np.nan_to_num(fi[j, m, :maxno]), b["nos"][m], x[q] - b["xi"][m], D)
                assert abs(out[j, q] - want) <= 1e-12 * (1 + abs(want)), (D, q, j)
    # every slot at once: slots < no_m as the numpy model, zeros beyond
    out, _ = s.interpolate_fields(x, fi, diff='all', I=I)
    for q in range(len(x)):
        m, no = I[q], b["nos"][I[q]]
        T = T_matrix(dim, x[q] - b["xi"][m], maxno)
        for j in range(nf):
            want = T[:no, :no] @ fi[j, m, :no]
            assert np.all(np.abs(out[j, q, :no] - want) <= 1e-12 * (1 + np.abs(want))), (q, j)
            assert np.array_equal(out[j, q, no:], np.zeros(maxno - no)), (q, j)
    r = 0.1
    out, _ = s.interpolate_fields(x, fi, mode="continuous", r=r, diff=0)
    for q in range(len(x)):
        d2 = ((b["xi"] - x[q]) ** 2).sum(axis=1)
        inside = np.nonzero(d2 <= r * r)[0]
        for j in range(nf):
            if len(inside) == 0:
                assert np.isnan(out[j, q])
                continue
            wts = (1.0 - np.sqrt(d2[inside] / (r * r))) ** 2
            vals = [_taylor(dim, np.nan_to_num(fi[j, m, :maxno]), b["nos"][m], x[q] - b["xi"][m], 0) for m in inside]
            want = float(np.dot(wts, vals) / wts.sum())
            assert abs(out[j, q] - want) <= 1e-11 * (1 + abs(want)), (q, j)


def test_layouts_searches_and_ctypes():
    b = _batch(2, [2, 3, 4], 20, "rand", seed=9)
    s = _solver(b)
    s.prep_interpolate()
    nf = 5
    _, fk, fi0 = _data(b, s, nf, seed=10)
    x = _queries(b, seed=11)
    I = _nearest(b, x)
    ref, fi = _refs(s, fk, fi0, x, I, [0, 3, 'all'])
    dev = _dev()
    xt, It, fit = torch.as_tensor(x, device=dev), torch.as_tensor(I, device=dev), torch.as_tensor(fi, device=dev)
    for xa in (x, xt):
        for fa in (fi, fit):
            for Ia in (I, It, None):
                if Ia is It and not torch.is_tensor(xa):
                    continue                                      # interpolate() takes a CUDA I with CUDA x only
                out, I_out = s.interpolate_fields(xa, fa, diff=3, I=Ia)
                assert _eq(out, ref[3])
                assert torch.is_tensor(out) == torch.is_tensor(xa)
                if Ia is None:
                    assert np.array_equal(_host(I_out), I)
    # fields-inner and pitched fi
    inner = np.ascontiguousarray(fi.transpose(1, 0, 2)).transpose(1, 0, 2)
    assert _eq(s.interpolate_fields(x, inner, diff='all', I=I)[0], ref['all'])
    inner_t = torch.as_tensor(np.ascontiguousarray(fi.transpose(1, 0, 2)), device=dev).permute(1, 0, 2)
    assert _eq(s.interpolate_fields(xt, inner_t, diff=0, I=It)[0], ref[0])
    assert _eq(s.interpolate_fields(xt, fit[:1].expand(3, -1, -1), diff=0, I=It)[0], ref[0][[0, 0, 0]])   # fi_sf = 0
    pitched = np.full((nf, len(b["nk"]) + 3, s._maxno + 5), np.nan)
    pitched[:, :len(b["nk"]), :fi.shape[2]] = fi
    assert _eq(s.interpolate_fields(xt, torch.as_tensor(pitched, device=dev), diff=0, I=It)[0], ref[0])
    # the device search answers where the host one does
    s2 = _solver(b)
    s2.prep_interpolate(search='gpu')
    assert _eq(s2.interpolate_fields(x, fi, diff=0)[0], ref[0])
    # through ctypes: a fields-inner out, refused layouts and overlaps
    L = _lib.lib()
    nx, maxno = len(x), s._maxno
    buf = torch.full((nx, nf, maxno), float("nan"), dtype=torch.float64, device=dev)
    _lib.check(L.wlsqm_solver_interpolate_fields(s._handle, nf, int(fit.data_ptr()), fit.stride(0), fit.stride(1),
                                                 int(xt.data_ptr()), 2, int(It.data_ptr()), nx, _lib.DIFF_ALL,
                                                 int(buf.data_ptr()), maxno, nf * maxno))
    assert _eq(buf.permute(1, 0, 2), ref['all'])
    buf1 = torch.full((nx, nf), float("nan"), dtype=torch.float64, device=dev)     # one slot, fields-inner out
    _lib.check(L.wlsqm_solver_interpolate_fields(s._handle, nf, int(fit.data_ptr()), fit.stride(0), fit.stride(1),
                                                 int(xt.data_ptr()), 2, int(It.data_ptr()), nx, 3,
                                                 int(buf1.data_ptr()), 1, nf))
    assert _eq(buf1.T, ref[3])
    one = torch.zeros((nf, nx), dtype=torch.float64, device=dev)
    for sf, sq in ((1, 1), (0, 1), (nx - 1, 1)):
        with pytest.raises(ValueError, match="layout"):
            _lib.check(L.wlsqm_solver_interpolate_fields(s._handle, nf, int(fit.data_ptr()), fit.stride(0), fit.stride(1),
                                                         int(xt.data_ptr()), 2, int(It.data_ptr()), nx, 0,
                                                         int(one.data_ptr()), sf, sq))
    for victim in (fit, xt, It):
        with pytest.raises(ValueError, match="overlap"):
            _lib.check(L.wlsqm_solver_interpolate_fields(s._handle, nf, int(fit.data_ptr()), fit.stride(0), fit.stride(1),
                                                         int(xt.data_ptr()), 2, int(It.data_ptr()), nx, 0,
                                                         int(victim.data_ptr()), 1, nf))
    with pytest.raises(ValueError, match="r must be positive"):
        _lib.check(L.wlsqm_solver_interpolate_continuous_fields(s._handle, nf, int(fit.data_ptr()), fit.stride(0),
                                                                fit.stride(1), int(xt.data_ptr()), 2, nx, float("nan"), 0,
                                                                int(one.data_ptr()), nx, 1))
    with pytest.raises(ValueError, match="diff"):
        _lib.check(L.wlsqm_solver_interpolate_fields(s._handle, nf, int(fit.data_ptr()), fit.stride(0), fit.stride(1),
                                                     int(xt.data_ptr()), 2, int(It.data_ptr()), nx, maxno,
                                                     int(one.data_ptr()), nx, 1))
    torch.cuda.synchronize()


def test_solution_copy_guest_and_empty():
    b = _batch(2, [4], 20, "F", seed=12)
    s = _solver(b)
    s.prep_interpolate()
    nf = 3
    _, fk, fi0 = _data(b, s, nf, seed=13)
    x = _queries(b, seed=14)
    I = _nearest(b, x)
    ref, fis = _refs(s, fk, fi0, x, I, [0])
    fi = fi0.copy()
    s.solve_fields(fk, fi)
    with pytest.raises(RuntimeError):
        s.interpolate(x, diff=0, I=I)
    assert _eq(s.interpolate_fields(x, fi, diff=0, I=I)[0], ref[0])
    with pytest.raises(RuntimeError):                             # interpolate() still needs a solve()
        s.interpolate(x, diff=0, I=I)
    s.keep_solution(False)
    dev = _dev()
    fit = torch.as_tensor(fi0.copy(), device=dev)
    s.solve(torch.as_tensor(fk[0], device=dev), fit[0])
    assert _eq(s.interpolate_fields(x, fi, diff=0, I=I)[0], ref[0])
    s.keep_solution(True)
    # a guest answers with its host's origins, as its own interpolate() does
    g = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"], host=s)
    g.prepare(None, None)
    g.prep_interpolate()
    gi = fi0[1].copy()
    g.solve(fk[1], gi)
    assert _eq(g.interpolate_fields(x, fi[1:2], diff=0, I=I)[0][0], g.interpolate(x, diff=0, I=I)[0])
    # no fields, no queries
    assert s.interpolate_fields(x, np.zeros((0, len(b["nk"]), s._maxno)), diff=0, I=I)[0].shape == (0, len(x))
    assert s.interpolate_fields(x[:0], fi, diff='all', I=I[:0])[0].shape == (nf, 0, s._maxno)
    assert s.interpolate_fields(x[:0], fi, mode='continuous', r=0.1)[0].shape == (nf, 0)
    # a NaN query (the device search reports it as model ncases) poisons the whole host output, as in interpolate()
    s.prep_interpolate(search='gpu')
    xn = x.copy()
    xn[4] = np.nan
    out, I_out = s.interpolate_fields(xn, fi, diff=0)
    assert np.isnan(out).all() and I_out[4] == len(b["nk"])
    torch.cuda.synchronize()
