"""CPU checks of the argument resolution of ExpertSolver.interp_stencils / .interp_operator with mode='continuous'
(wlsqm_b200.fitter.opexport), in both bindings.  No device is needed: the methods are called on a stand-in solver
without a handle, so accepted arguments go through to the C ABI, which answers "NULL solver" (and every refusal must
come before that)."""
import os
import subprocess
import sys
import types
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent

N, MAXNO, MAXNK, NX = 7, 6, 9, 5


def _fake(tree=True):
    return types.SimpleNamespace(ready=True, ncases=N, dimension=2, _maxno=MAXNO, _maxnk=MAXNK, _handle=None, device=0,
                                 host=None, _use_stream=lambda: None, tree=object() if tree else None,
                                 _nearest_models=lambda x, xp, x_s0, nx, x_cuda, I: (I, I))


def _cases():
    """(expected, method, kwargs): 'ok' reaches the C ABI, others must raise before it with the expected text"""
    I = np.arange(NX, dtype=np.int64)
    out = []
    for meth in ("interp_stencils", "interp_operator"):
        out += [
            ("ok", meth, dict(mode='continuous', r=0.5)),
            ("ok", meth, dict(mode='continuous', r=np.float64(0.25), coeffs=np.ones((3, MAXNO)))),
            ("ok", meth, dict(mode='continuous', r=np.inf)),
            ("ok", meth, dict(I=I)),
            ("mode must be", meth, dict(mode='linear', r=0.5)),
            ("r must be specified", meth, dict(mode='continuous')),
            ("r must be positive", meth, dict(mode='continuous', r=0.0)),
            ("r must be positive", meth, dict(mode='continuous', r=-1.0)),
            ("r must be positive", meth, dict(mode='continuous', r=np.nan)),
            ("I cannot be given", meth, dict(mode='continuous', r=0.5, I=I)),
            ("coeffs must", meth, dict(mode='continuous', r=0.5, coeffs=np.zeros(MAXNO + 1))),
            ("finite", meth, dict(mode='continuous', r=0.5, coeffs=np.full(MAXNO, np.nan))),
        ]
    out.append(("center must be", "interp_operator", dict(mode='continuous', r=0.5, center=-2)))
    return out


def _run(cls):
    res = []
    for exp, meth, kw in _cases():
        kw = dict(kw)
        coeffs = kw.pop("coeffs", 0)
        try:
            getattr(cls, meth)(_fake(), np.zeros((NX, 2)), coeffs, **kw)
            got = "returned"
        except ValueError as e:
            got = "ok" if "NULL solver" in str(e) else str(e)
        except TypeError as e:
            got = "TypeError: %s" % e
        res.append((exp, got))
    return res


def _verdict(res):
    bad = []
    for exp, got in res:
        if exp == "ok":
            if got != "ok":
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
            "import wlsqm_b200 as w, test_interp_continuous_operator_args as t\n"
            "from wlsqm_b200.fitter import expert\n"
            "assert expert.BINDING == 'ctypes' and w.ExpertSolver.__module__.endswith('expert')\n"
            "bad = t._verdict(t._run(w.ExpertSolver))\n"
            "print('ok' if not bad else bad)\n" % (str(ROOT / "python-wlsqm_b200"), str(ROOT / "tests")))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       env=dict(os.environ, WLSQM_BINDING="ctypes"))
    assert r.stdout.strip() == "ok", (r.stdout[-600:], r.stderr[-600:])


def test_not_indexed():
    import wlsqm_b200 as w
    for meth in ("interp_stencils", "interp_operator"):
        with pytest.raises(RuntimeError, match="prep_interpolate"):
            getattr(w.ExpertSolver, meth)(_fake(tree=False), np.zeros((NX, 2)), 0, mode='continuous', r=0.5)
