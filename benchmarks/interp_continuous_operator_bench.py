"""Continuous-mode interpolation operators on one GPU: interp_stencils / interp_operator(mode='continuous') against the
route solve_hoods + interpolate(mode='continuous').

    python benchmarks/interp_continuous_operator_bench.py [--out FILE] [--reps R] [--n N]

Solver: cfg2 (1M points, 2D order 4, k = 30, uniform weights, no knowns) from prepare_hoods on a device kNN.  Queries:
the 1M transfer points of benchmarks/interp_operator_bench.py (the same seeded draws), as device tensors.  Radii r =
1.5 h0 and 2.5 h0 with h0 = 1 / sqrt(n) (about 7 and 20 models per query).  Operators: the value and the Laplacian.
Timed per case: the count call (pairs and nnz), interp_stencils, interp_operator, the route, and one step E @ f (torch
CSR matvec).  The count and interp_operator are also timed with every row on the sort route (WLSQM_CONT_ROW_CAP=0)
instead of the shared-memory row merge, alternated with the default in the same repeats.  Each is called once per repeat and the repeats alternate between them; medians over --reps repeats with
their interquartile range, after one warm-up call of each.  The working sets are larger than L2.  Bytes: the least the
algorithm moves (below), over the median time, against the project's measured HBM bandwidth of 6558 GB/s.  What does
not fit the device or fails is reported as not measured.  The GPU's name and power limit are read in this process.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "python-wlsqm_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import wlsqm_b200 as w  # noqa: E402
from wlsqm_b200 import _lib  # noqa: E402
from wlsqm_b200.fitter import defs  # noqa: E402

HBM_GBS = 6558.0


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # noqa: BLE001
        pl = "unavailable (%s)" % e
    return name, pl


def once(fn):
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def bytes_formula(nx, npairs, nnz, n, nk, no, nops, dim, csr):
    """interp_stencils: every operator block once (8 nk nr), the queries (8 dim) and the pair arrays (pair_ptr, J, the
    query and weight of a pair: 8 + 8 + 4 + 8), W and K written (8 nops (nk + no) per pair).  interp_operator adds W read
    back and the CSR written (col 4 and values 8 nops per entry); the merge itself stays in shared memory (the sort
    route's scratch traffic is not counted)."""
    b = 8.0 * n * nk * no + 8.0 * nx * dim + 28.0 * npairs + 8.0 * npairs * nops * (nk + no)
    if csr:
        b += 8.0 * npairs * nops * nk + nnz * (4 + 8.0 * nops) + 4.0 * nx
    return b


def stats(v):
    v = np.asarray(v)
    q1, med, q3 = np.percentile(v, [25, 50, 75])
    return float(med), float((q3 - q1) / med) if med else 0.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--n", type=int, default=1_000_000)
    args = ap.parse_args()
    name, pl = card()
    dev = torch.device("cuda", 0)
    n, k, dim, order = args.n, 30, 2, 4
    no = defs.NUMBER_OF_DOFS[dim][order]
    g = torch.Generator(device="cpu").manual_seed(1)
    x = torch.rand((n, dim), generator=g, dtype=torch.float64).to(dev)
    xq = torch.rand((n, dim), generator=g, dtype=torch.float64).to(dev)       # the transfer queries
    f = torch.rand(n, generator=torch.Generator(device="cpu").manual_seed(2), dtype=torch.float64).to(dev)
    hoods = w.knn_hoods(x, k)
    s = w.ExpertSolver(dim, np.full(n, k, np.int32), np.full(n, order, np.int32), np.zeros(n, np.int64),
                       np.full(n, defs.WEIGHT_UNIFORM, np.int32))
    s.prepare_hoods(x, hoods)
    s.prep_interpolate()
    fi = torch.zeros((n, no), dtype=torch.float64, device=dev)
    lap = np.zeros(no)
    lap[[defs.i2_X2, defs.i2_Y2]] = 1.0
    ops = {"value": (np.eye(no)[[0]], [0]), "laplacian": (lap[None], [defs.i2_X2, defs.i2_Y2])}
    L = _lib.lib()
    h0 = 1.0 / math.sqrt(n)
    lines = []
    for rmul in (1.5, 2.5):
        r = rmul * h0
        for oname, (c, diffs) in ops.items():
            out = {"run": "cfg2", "queries": "transfer", "nx": n, "r_over_h0": rmul, "op": oname, "n": n, "k": k,
                   "order": order, "gpu": name, "power_limit": pl, "reps": args.reps}
            pp = torch.empty(n + 1, dtype=torch.int64, device=dev)
            npairs, nnz = C.c_int64(), C.c_int64()

            def count():
                _lib.check(L.wlsqm_solver_interp_continuous_count(s._handle, xq.data_ptr(), dim, n, r, -1, pp.data_ptr(),
                                                                  C.byref(npairs), C.byref(nnz)))
            E = []

            def operator():
                E[:] = [s.interp_operator(xq, c, mode="continuous", r=r)[0]]

            def route():
                s.solve_hoods(f, fi)
                return [s.interpolate(xq, mode="continuous", r=r, diff=int(d))[0] for d in diffs]
            def sort_route(fn):
                def run():
                    os.environ["WLSQM_CONT_ROW_CAP"] = "0"
                    try:
                        fn()
                    finally:
                        del os.environ["WLSQM_CONT_ROW_CAP"]
                return run
            fns = {"count": count, "count_sort_route": sort_route(count),
                   "interp_stencils": lambda: s.interp_stencils(xq, c, mode="continuous", r=r),
                   "interp_operator": operator, "interp_operator_sort_route": sort_route(operator),
                   "route_solve_interpolate": route, "step_E_at_f": lambda: E[0][0] @ f}
            times = {key: [] for key in fns}
            for key, fn in fns.items():
                try:
                    fn()
                except (torch.cuda.OutOfMemoryError, RuntimeError, MemoryError, IndexError) as e:
                    times[key] = "not measured (%s)" % str(e).splitlines()[0][:80]
                torch.cuda.empty_cache()
            for _ in range(args.reps):
                for key, fn in fns.items():
                    if isinstance(times[key], list):
                        times[key].append(once(fn))
            out["mean_pairs_per_query"] = npairs.value / n
            out["nnz_per_row"] = nnz.value / n
            for key, t in times.items():
                if isinstance(t, list):
                    out[key + "_ms"], out[key + "_iqr_rel"] = stats(t)
                else:
                    out[key + "_ms"] = t
            for key, csr in (("interp_stencils", False), ("interp_operator", True), ("interp_operator_sort_route", True)):
                b = bytes_formula(n, npairs.value, nnz.value, n, k, no, len(c), dim, csr)
                out["bytes_" + key] = b
                if isinstance(out[key + "_ms"], float):
                    out[key + "_hbm_fraction"] = b / (out[key + "_ms"] * 1e-3) / (HBM_GBS * 1e9)
            if isinstance(out.get("step_E_at_f_ms"), float) and isinstance(out.get("route_solve_interpolate_ms"), float):
                out["step_speedup_vs_route"] = out["route_solve_interpolate_ms"] / out["step_E_at_f_ms"]
            E.clear()
            torch.cuda.empty_cache()
            line = json.dumps(out)
            print(line, flush=True)
            lines.append(line)
    s.close()
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
