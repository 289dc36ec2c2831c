"""CPU checks of the argument resolution of ExpertSolver.interpolate_fields (wlsqm_b200.fitter.fields), in both
bindings: modes, diff, I, the shape and dtype of fi, and the output a query without a model gives.  No device is needed:
the method is called on a stand-in solver without a handle, so accepted arguments go through to the C ABI, which answers
"NULL solver" (and every refusal must come before that)."""
import os
import subprocess
import sys
import types
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent

N, MAXNO, NX = 7, 6, 5


def _fake(tree=True):
    return types.SimpleNamespace(ready=True, ncases=N, dimension=2, _maxno=MAXNO, _handle=None, _use_stream=lambda: None,
                                 tree=object() if tree else None,
                                 _nearest_models=lambda x, xp, x_s0, nx, x_cuda, I: (I, I))   # I is always given here


def _cases():
    """(expected, x, fi, kwargs): 'ok' reaches the C ABI, 'nan' returns all-NaN output without it, others must raise
    before it with a message containing the expected text"""
    x = np.zeros((NX, 2))
    fi = np.zeros((3, N, MAXNO))
    I = np.arange(NX, dtype=np.int64)
    inner = np.zeros((N, 3, MAXNO)).transpose(1, 0, 2)
    same = np.broadcast_to(np.zeros((N, MAXNO)), (3, N, MAXNO))        # fi_sf = 0: one field three times (read only)
    return [
        ("ok", x, fi, dict(I=I)),
        ("ok", x, fi, dict(I=I, diff='all')),
        ("ok", x, fi, dict(I=I, diff=3)),
        ("ok", x, inner, dict(I=I)),
        ("ok", x, same, dict(I=I)),
        ("ok", x, np.zeros((3, N + 2, MAXNO + 3)), dict(I=I)),
        ("ok", x, fi[:1], dict(I=I)),
        ("ok", x, fi, dict(mode='continuous', r=0.5)),
        ("ok", x, np.zeros((0, N, MAXNO)), dict(I=I)),
        ("nan", x, fi, dict(I=np.array([0, 1, N, 2, 3], np.int64))),
        ("nan", x, fi, dict(I=np.array([0, 1, N, 2, 3], np.int64), diff='all')),
        ("mode must be", x, fi, dict(I=I, mode='linear')),
        ("r must be specified", x, fi, dict(mode='continuous')),
        ("diff cannot be None", x, fi, dict(I=I, diff=None)),
        ("same length", x, fi, dict(I=I[:NX - 1])),
        ("not available in mode='continuous'", x, fi, dict(mode='continuous', r=0.5, diff='all')),
        ("dtype", x, fi.astype(np.float32), dict(I=I)),
        ("dimensions", x, fi[0], dict(I=I)),
        ("shape", x, fi[:, :N - 1], dict(I=I)),
        ("shape", x, fi[:, :, :MAXNO - 1], dict(I=I)),
        ("contiguous", x, np.zeros((3, N, 2 * MAXNO))[:, :, ::2], dict(I=I)),
        ("dtype", x.astype(np.float32), fi, dict(I=I)),
    ]


def _run(cls):
    """-> list of (expected, outcome) for the cases"""
    res = []
    for exp, x, fi, kw in _cases():
        try:
            out, _ = cls.interpolate_fields(_fake(), x, fi, **kw)
            want = (fi.shape[0], NX, MAXNO) if kw.get("diff") == 'all' else (fi.shape[0], NX)
            got = "nan" if out.shape == want and np.isnan(out).all() else "returned %s" % (out.shape,)
        except ValueError as e:
            got = "ok" if "NULL solver" in str(e) else str(e)
        except TypeError as e:
            got = "TypeError: %s" % e
        res.append((exp, got))
    return res


def _verdict(res):
    bad = []
    for exp, got in res:
        if exp in ("ok", "nan"):
            if got != exp:
                bad.append((exp, got))
        elif got == "ok" or exp.lower() not in got.lower():
            bad.append((exp, got))
    return bad


def test_cython_binding():
    import wlsqm_b200 as w
    from wlsqm_b200.fitter import expert
    assert expert.BINDING == "cython", "build the shim: python python-wlsqm_b200/build_shim.py"
    assert not _verdict(_run(w.ExpertSolver)), _verdict(_run(w.ExpertSolver))


def test_ctypes_binding():
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import wlsqm_b200 as w, test_interp_fields_args as t\n"
            "from wlsqm_b200.fitter import expert\n"
            "assert expert.BINDING == 'ctypes' and w.ExpertSolver.__module__.endswith('expert')\n"
            "bad = t._verdict(t._run(w.ExpertSolver))\n"
            "print('ok' if not bad else bad)\n" % (str(ROOT / "python-wlsqm_b200"), str(ROOT / "tests")))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       env=dict(os.environ, WLSQM_BINDING="ctypes"))
    assert r.stdout.strip() == "ok", (r.stdout[-600:], r.stderr[-600:])


def test_not_indexed():
    import wlsqm_b200 as w
    for kw in (dict(I=np.arange(NX, dtype=np.int64)), dict(mode='continuous', r=0.5)):
        with pytest.raises(RuntimeError, match="prep_interpolate"):
            w.ExpertSolver.interpolate_fields(_fake(tree=False), np.zeros((NX, 2)), np.zeros((2, N, MAXNO)), **kw)
