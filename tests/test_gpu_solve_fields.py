"""GPU tests of the field-batched solve: ExpertSolver.solve_fields / .solve_hoods_fields (csrc/wlsqm_solve_fields.cu).

The contract is per-field equality: for every field j the result must be bit for bit what solve(fk[j], fi[j]) (or
solve_hoods(f[j], fi[j])) writes on the same solver, with known slots and padding untouched, the return value the
maximum of the single solves' and iterations() their per-case maximum.  fi starts from random values everywhere, so
that a write to a known slot or to padding shows, and every field has its own data and known values.
"""
import numpy as np
import pytest
from scipy.spatial import cKDTree

import wlsqm_b200 as w
from wlsqm_b200 import _lib
from wlsqm_b200.fitter import defs
from test_gpu_operator import _batch, _solver

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

DEV = None


def _dev():
    global DEV
    if DEV is None:
        DEV = torch.device("cuda", _lib.default_device())
    return DEV


def _uniform_batch(dim, order, k, knowns_mode, n=400, seed=0):
    """every case with the same sizes (geometry-uniform: the packed kernel for small blocks); knowns pattern may vary"""
    # (the mixed-size builder duplicates neighbour columns up to 5: its cloud is drawn with at least 6 neighbours)
    b = _batch(dim, [order], max(k, 6), knowns_mode, n=n, seed=seed)
    _, hoods = cKDTree(b["x"]).query(b["xi"], k)
    hoods = hoods.astype(np.int32)
    hoods[::7, 2 % k] = hoods[::7, 0]                  # duplicated neighbours
    b["hoods"] = hoods
    b["nk"][:] = k
    b["wm"][:] = 1
    if knowns_mode == "rand":
        rng = np.random.default_rng(seed + 1)
        no = defs.NUMBER_OF_DOFS[dim][order]
        # the same NUMBER of knowns in every case (geometry-uniform), in varying slots
        nkn = 1 if no > 1 else 0
        kn = np.zeros(n, np.int64)
        for i in range(n):
            if nkn:
                kn[i] = 1 << int(rng.integers(0, no))
        b["knowns"] = kn
    return b


def _data(b, s, nf, seed=1):
    """fk (nf, n, max nk + 3) with smooth and rough fields, fi0 (nf, n, max no + 2) random everywhere"""
    rng = np.random.default_rng(seed)
    n = len(b["nk"])
    x = b["x"]
    fpt = np.stack([np.sin((j + 1) * x.sum(axis=1)) + (0.1 * j) * rng.standard_normal(len(x)) for j in range(nf)])
    hk = np.clip(b["hoods"], 0, len(x) - 1)
    fk = np.full((nf, n, s._maxnk + 3), np.nan)
    for j in range(nf):
        fk[j, :, :s._maxnk] = fpt[j][hk[:, :s._maxnk]]
    fi0 = rng.standard_normal((nf, n, s._maxno + 2))
    return fpt, fk, fi0


def _single(s, fk, fi0, hoods_f=None):
    """per-field single solves: results, return values, per-case iteration counts"""
    outs, its, iters = [], [], []
    for j in range(fi0.shape[0]):
        fi = fi0[j].copy()
        its.append(s.solve_hoods(hoods_f[j], fi) if hoods_f is not None else s.solve(fk[j], fi))
        iters.append(s.iterations())
        outs.append(fi)
    return np.stack(outs), max(its), np.max(np.stack(iters), axis=0)


def _eq(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    return a.shape == b.shape and np.array_equal(a.view(np.int64), b.view(np.int64))


def _check(s, fk, fi0, ref, it_ref, iters_ref, cuda=True):
    dev = _dev()
    fi = torch.as_tensor(fi0.copy(), device=dev) if cuda else fi0.copy()
    fkx = torch.as_tensor(fk, device=dev) if cuda else fk
    it = s.solve_fields(fkx, fi)
    assert _eq(fi, ref)
    assert it == it_ref
    assert np.array_equal(s.iterations(), iters_ref)


CFGS = [(1, [0], 6), (1, [4], 10), (2, [2], 12), (2, [4], 20), (3, [1], 10), (3, [3], 26), (3, [4], 40),
        (2, [2, 3, 4], 20), (3, [0, 2, 3, 4], 40)]


@pytest.mark.parametrize("algo", [defs.ALGO_BASIC, defs.ALGO_ITERATIVE])
@pytest.mark.parametrize("knowns_mode", [0, "F", "rand"])
@pytest.mark.parametrize("dim,orders,k", CFGS)
def test_fields_equal_single_solves_mixed(dim, orders, k, knowns_mode, algo):
    """mixed-size batches (ragged nk, duplicated hoods), every order, known patterns; nf = 1, 2, 3, 8 and 40 (more
    fields than one pass holds for the larger blocks)"""
    b = _batch(dim, orders, k, knowns_mode)
    s = _solver(b, algorithm=algo, max_iter=4)
    _, fk, fi0 = _data(b, s, 40)
    ref, _, _ = _single(s, fk, fi0)
    for nf in (1, 2, 3, 8, 40):
        # the maxima over the first nf fields
        _, it_ref, iters_ref = _single(s, fk[:nf], fi0[:nf])
        _check(s, fk[:nf], fi0[:nf], ref[:nf], it_ref, iters_ref)


@pytest.mark.parametrize("algo", [defs.ALGO_BASIC, defs.ALGO_ITERATIVE])
@pytest.mark.parametrize("knowns_mode", [0, "F", "rand"])
@pytest.mark.parametrize("dim,order,k", [(1, 2, 5), (2, 2, 12), (2, 4, 30), (3, 2, 16), (3, 4, 60), (3, 4, 36)])
def test_fields_equal_single_solves_uniform(dim, order, k, knowns_mode, algo):
    """geometry-uniform batches: the packed kernel (small ALGO_BASIC blocks) and the uniform-record kernel; 3D order 4
    without knowns has 35 > 32 unknowns"""
    b = _uniform_batch(dim, order, k, knowns_mode, n=333)
    s = _solver(b, algorithm=algo, max_iter=3)
    _, fk, fi0 = _data(b, s, 24, seed=2)
    for nf in (1, 2, 3, 8, 24):
        ref, it_ref, iters_ref = _single(s, fk[:nf], fi0[:nf])
        _check(s, fk[:nf], fi0[:nf], ref, it_ref, iters_ref)


@pytest.mark.parametrize("algo", [defs.ALGO_BASIC, defs.ALGO_ITERATIVE])
def test_several_passes(algo):
    """3D order 4 with k = 60: a pass holds only a few fields, so 13 fields take several passes"""
    b = _uniform_batch(3, 4, 60, "rand", n=500, seed=3)
    s = _solver(b, algorithm=algo, max_iter=4)
    _, fk, fi0 = _data(b, s, 13, seed=4)
    ref, it_ref, iters_ref = _single(s, fk, fi0)
    _check(s, fk, fi0, ref, it_ref, iters_ref)
    _check(s, fk, fi0, ref, it_ref, iters_ref, cuda=False)


@pytest.mark.parametrize("algo", [defs.ALGO_BASIC, defs.ALGO_ITERATIVE])
@pytest.mark.parametrize("dim,orders,k,uniform", [(2, [4], 20, False), (3, [2, 3, 4], 40, False), (2, [2], 12, True)])
def test_hoods_fields_equal_solve_hoods(dim, orders, k, uniform, algo):
    b = _uniform_batch(dim, orders[0], k, "rand") if uniform else _batch(dim, orders, k, "rand")
    s = _solver(b, algorithm=algo, max_iter=3)
    fpt, _, fi0 = _data(b, s, 9, seed=5)
    ref, it_ref, iters_ref = _single(s, None, fi0, hoods_f=fpt)
    dev = _dev()
    for f in (torch.as_tensor(fpt, device=dev), torch.as_tensor(np.ascontiguousarray(fpt.T), device=dev).T, fpt,
              np.ascontiguousarray(fpt.T).T):
        fi = torch.as_tensor(fi0.copy(), device=dev)
        assert s.solve_hoods_fields(f, fi) == it_ref
        assert _eq(fi, ref)
        assert np.array_equal(s.iterations(), iters_ref)
    fi = fi0.copy()                                           # numpy fi
    s.solve_hoods_fields(fpt, fi)
    assert _eq(fi, ref)


def test_layouts_numpy_guest():
    b = _batch(2, [2, 3, 4], 20, "rand", seed=6)
    s = _solver(b, algorithm=defs.ALGO_ITERATIVE, max_iter=3)
    nf = 5
    _, fk, fi0 = _data(b, s, nf, seed=7)
    ref, it_ref, iters_ref = _single(s, fk, fi0)
    dev = _dev()
    # numpy against CUDA
    _check(s, fk, fi0, ref, it_ref, iters_ref, cuda=False)
    _check(s, fk, fi0, ref, it_ref, iters_ref, cuda=True)
    # fields-inner fi: (ncases, nf, no) storage
    inner = torch.as_tensor(np.ascontiguousarray(fi0.transpose(1, 0, 2)), device=dev)
    fiv = inner.permute(1, 0, 2)
    assert s.solve_fields(torch.as_tensor(fk, device=dev), fiv) == it_ref
    assert _eq(fiv, ref)
    inner_np = np.ascontiguousarray(fi0.transpose(1, 0, 2))
    s.solve_fields(fk, inner_np.transpose(1, 0, 2))
    assert _eq(inner_np.transpose(1, 0, 2), ref)
    # a fully strided device fk: (n, maxnk, nf) storage, every row pitched
    big = torch.full((fk.shape[1], fk.shape[2] * 2, nf + 1), float("nan"), dtype=torch.float64, device=dev)
    big[:, ::2, :nf] = torch.as_tensor(fk, device=dev).permute(1, 2, 0)
    fks = big[:, ::2, :nf].permute(2, 0, 1)
    assert fks.stride(2) != 1
    fi = torch.as_tensor(fi0.copy(), device=dev)
    s.solve_fields(fks, fi)
    assert _eq(fi, ref)
    # a guest answers with its host's operators
    g = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"], algorithm=defs.ALGO_ITERATIVE, max_iter=3, host=s)
    g.prepare(None, None)
    fi = torch.as_tensor(fi0.copy(), device=dev)
    assert g.solve_fields(torch.as_tensor(fk, device=dev), fi) == it_ref
    assert _eq(fi, ref)
    assert np.array_equal(g.iterations(), iters_ref)


def test_sens_solver_and_zero_sizes():
    b = _batch(2, [4], 20, "F", seed=8)
    s = _solver(b, do_sens=True)
    _, fk, fi0 = _data(b, s, 3, seed=9)
    n = len(b["nk"])
    refs = []
    for j in range(3):
        fi = fi0[j].copy()
        s.solve(fk[j], fi, np.zeros((n, s._maxnk, s._maxno)))
        refs.append(fi)
    fi = fi0.copy()
    assert s.solve_fields(fk, fi) == 0
    assert _eq(fi, np.stack(refs))
    empty = np.zeros((0, n, s._maxno))
    assert s.solve_fields(np.zeros((0, n, s._maxnk)), empty) == 0
    assert s.solve_hoods_fields(np.zeros((0, len(b["x"]))), empty) == 0


def test_errors_and_solution_copy():
    b = _batch(2, [2, 3], 12, "rand", seed=10)
    s = _solver(b)
    _, fk, fi0 = _data(b, s, 3, seed=11)
    dev = _dev()
    n = len(b["nk"])
    s.prep_interpolate()
    s.solve(fk[0], fi0[0].copy())
    s.interpolate(b["xi"][:5], diff=0)
    fi = torch.as_tensor(fi0.copy(), device=dev)
    s.solve_fields(torch.as_tensor(fk, device=dev), fi)
    with pytest.raises(RuntimeError):
        s.interpolate(b["xi"][:5], diff=0)
    s.solve(fk[0], fi0[0].copy())
    s.interpolate(b["xi"][:5], diff=0)
    # device fk overlapping device fi
    buf = torch.zeros((3, n, s._maxnk + s._maxno + 4), dtype=torch.float64, device=dev)
    with pytest.raises(ValueError, match="overlap"):
        s.solve_fields(buf[:, :, :s._maxnk], buf[:, :, 2:2 + s._maxno])
    # fi layouts that map two entries to one element
    flat = torch.zeros(n * s._maxno + 10, dtype=torch.float64, device=dev)
    alias = flat.as_strided((3, n, s._maxno), (1, s._maxno, 1))
    with pytest.raises(ValueError):
        s.solve_fields(torch.as_tensor(fk, device=dev), alias)
    same = flat.as_strided((3, n, s._maxno), (0, s._maxno, 1))
    with pytest.raises(ValueError):
        s.solve_fields(torch.as_tensor(fk, device=dev), same)
    with pytest.raises(ValueError):
        s.solve_fields(fk[:2], fi0.copy())                  # field counts differ
    # an active fused gather
    s2 = _solver(b)
    tgt = torch.zeros((n, 16), dtype=torch.float64, device=dev)
    import ctypes as C
    bases = (C.c_void_p * 1)(tgt.data_ptr())
    _lib.check(_lib.lib().wlsqm_solver_set_gather(s2._handle, 1, bases, 0, 16))
    with pytest.raises(ValueError, match="gather"):
        s2.solve_fields(fk, fi0.copy())
    # no prepare_hoods
    s3 = w.ExpertSolver(2, b["nk"], b["order"], b["knowns"], b["wm"])
    xk = b["x"][np.clip(b["hoods"], 0, len(b["x"]) - 1)]
    s3.prepare(b["xi"], xk)
    with pytest.raises(RuntimeError):
        s3.solve_hoods_fields(np.zeros((3, len(b["x"]))), fi0.copy())
    torch.cuda.synchronize()


def test_full_size_cfg2_eight_fields():
    n, k, nf = 1_000_000, 30, 8
    dev = _dev()
    g = torch.Generator(device="cpu").manual_seed(0)
    x = (torch.randint(0, 2 ** 24, (n, 2), generator=g) / 2.0 ** 24).double().to(dev)
    hoods = w.knn_hoods(x, k)
    s = w.ExpertSolver(2, np.full(n, k, np.int32), np.full(n, 4, np.int32), np.zeros(n, np.int64),
                       np.full(n, 1, np.int32))
    s.prepare_hoods(x, hoods)
    f = torch.stack([torch.sin((j + 1) * x.sum(dim=1)) for j in range(nf)])
    ref = torch.zeros((nf, n, 15), dtype=torch.float64, device=dev)
    for j in range(nf):
        s.solve_hoods(f[j], ref[j])
    fi = torch.zeros((nf, n, 15), dtype=torch.float64, device=dev)
    s.solve_hoods_fields(f, fi)
    assert bool((fi.view(torch.int64) == ref.view(torch.int64)).all())
    fk = torch.stack([f[j][hoods.long()] for j in range(nf)])
    fi2 = torch.zeros((nf, n, 15), dtype=torch.float64, device=dev)
    s.solve_fields(fk, fi2)
    assert bool((fi2.view(torch.int64) == ref.view(torch.int64)).all())
    torch.cuda.synchronize()
