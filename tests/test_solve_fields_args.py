"""CPU checks of the argument resolution of ExpertSolver.solve_fields / .solve_hoods_fields (wlsqm_b200.fitter.fields),
in both bindings: shapes, dtypes, the two accepted fi layouts and refused ones.  No device is needed: the methods are
called on a stand-in solver without a handle, so accepted arguments go through to the C ABI, which answers "NULL solver"
(and every refusal must come before that)."""
import os
import subprocess
import sys
import types
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parent.parent

N, MAXNK, MAXNO, NPTS = 7, 5, 6, 11


def _fake():
    return types.SimpleNamespace(ready=True, ncases=N, _maxnk=MAXNK, _maxno=MAXNO, _hood_points=NPTS, _handle=None,
                                 _use_stream=lambda: None)


def _cases():
    """(name, call) pairs: ('ok', ...) reach the C ABI, others must raise ValueError before it"""
    fk = np.zeros((3, N, MAXNK))
    fi = np.zeros((3, N, MAXNO))
    inner = np.zeros((N, 3, MAXNO)).transpose(1, 0, 2)
    pitched = np.zeros((3, N, MAXNO + 4))[:, :, :MAXNO]
    f = np.zeros((3, NPTS))
    return [
        ("ok", "solve_fields", fk, fi),
        ("ok", "solve_fields", fk, inner),                                   # fields-inner rows
        ("ok", "solve_fields", fk, pitched),                                 # pitched fields-outer rows
        ("ok", "solve_fields", np.zeros((3, N + 2, MAXNK + 1)), np.zeros((3, N + 1, MAXNO + 1))),
        ("ok", "solve_fields", np.zeros((3, MAXNK + 2, N)).transpose(0, 2, 1)[:, :, :MAXNK], fi),   # strided host fk
        ("ok", "solve_hoods_fields", f, fi),
        ("ok", "solve_hoods_fields", np.zeros((NPTS, 3)).T, inner),          # f.T of (npoints, nf)
        ("no fields", "solve_fields", np.zeros((0, N, MAXNK)), np.zeros((0, N, MAXNO))),
        ("no fields", "solve_hoods_fields", np.zeros((0, NPTS)), np.zeros((0, N, MAXNO))),
        ("dtype", "solve_fields", fk.astype(np.float32), fi),
        ("dtype", "solve_fields", fk, fi.astype(np.float32)),
        ("dimensions", "solve_fields", fk[0], fi),
        ("dimensions", "solve_fields", fk, fi[0]),
        ("fields", "solve_fields", fk[:2], fi),                              # field counts differ
        ("shape", "solve_fields", fk[:, :N - 1], fi),
        ("shape", "solve_fields", fk[:, :, :MAXNK - 1], fi),
        ("shape", "solve_fields", fk, fi[:, :, :MAXNO - 1]),
        ("contiguous", "solve_fields", fk, np.zeros((3, N, 2 * MAXNO))[:, :, ::2]),
        ("read-only", "solve_fields", fk, np.broadcast_to(np.zeros(MAXNO), (3, N, MAXNO))),
        ("map two", "solve_fields", fk, np.lib.stride_tricks.as_strided(np.zeros(N * MAXNO + 2), (3, N, MAXNO),
                                                                       (8, MAXNO * 8, 8))),
        ("map two", "solve_fields", fk, np.lib.stride_tricks.as_strided(np.zeros(2 * N * MAXNO), (3, N, MAXNO),
                                                                       (MAXNO * 8 // 2, 2 * MAXNO * 8, 8))),
        ("fields", "solve_hoods_fields", f[:2], fi),
        ("one value per point", "solve_hoods_fields", f[:, :NPTS - 1], fi),
        ("dimensions", "solve_hoods_fields", f[0], fi),
    ]


def _run(cls):
    """-> list of (expected, outcome) for the cases"""
    res = []
    for exp, meth, a, b in _cases():
        try:
            got = "no fields" if getattr(cls, meth)(_fake(), a, b) == 0 else "returned"
        except ValueError as e:
            got = "ok" if "NULL solver" in str(e) else str(e)
        except TypeError as e:
            got = "TypeError: %s" % e
        res.append((exp, got))
    return res


def _verdict(res):
    bad = []
    for exp, got in res:
        if exp in ("ok", "no fields"):
            if got != exp:
                bad.append((exp, got))
        elif got == "ok" or exp.lower() not in got.lower():
            bad.append((exp, got))
    return bad


def test_layout_rule():
    from wlsqm_b200.fitter.fields import fi_layout_ok
    assert fi_layout_ok(3, N, MAXNO, N * MAXNO, MAXNO)                  # fields-outer, dense
    assert fi_layout_ok(3, N, MAXNO, MAXNO, 3 * MAXNO)                  # fields-inner, dense
    assert not fi_layout_ok(3, N, MAXNO, MAXNO, MAXNO)                  # fields overlap cases
    assert not fi_layout_ok(3, N, MAXNO, 0, MAXNO)
    assert not fi_layout_ok(3, N, MAXNO, -N * MAXNO, MAXNO)
    assert not fi_layout_ok(3, N, MAXNO, (N - 1) * MAXNO + MAXNO - 1, MAXNO)
    assert fi_layout_ok(1, N, MAXNO, 0, MAXNO)                          # one field: its stride is never used
    assert fi_layout_ok(3, 1, MAXNO, MAXNO, 0)                          # one case: its stride is never used


def test_cython_binding():
    import wlsqm_b200 as w
    from wlsqm_b200.fitter import expert
    assert expert.BINDING == "cython", "build the shim: python python-wlsqm_b200/build_shim.py"
    assert not _verdict(_run(w.ExpertSolver)), _verdict(_run(w.ExpertSolver))


def test_ctypes_binding():
    code = ("import sys; sys.path.insert(0, %r); sys.path.insert(0, %r)\n"
            "import wlsqm_b200 as w, test_solve_fields_args as t\n"
            "from wlsqm_b200.fitter import expert\n"
            "assert expert.BINDING == 'ctypes' and w.ExpertSolver.__module__.endswith('expert')\n"
            "bad = t._verdict(t._run(w.ExpertSolver))\n"
            "print('ok' if not bad else bad)\n" % (str(ROOT / "python-wlsqm_b200"), str(ROOT / "tests")))
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       env=dict(os.environ, WLSQM_BINDING="ctypes"))
    assert r.stdout.strip() == "ok", (r.stdout[-600:], r.stderr[-600:])


def test_not_ready():
    import wlsqm_b200 as w
    s = _fake()
    s.ready = False
    with pytest.raises(RuntimeError, match="ready"):
        w.ExpertSolver.solve_fields(s, np.zeros((1, N, MAXNK)), np.zeros((1, N, MAXNO)))
