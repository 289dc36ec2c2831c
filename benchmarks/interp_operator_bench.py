"""Interpolation operators on one GPU: ExpertSolver.interp_stencils / .interp_operator against solve + interpolate.

    python benchmarks/interp_operator_bench.py [--out FILE] [--reps R] [--n N]

Solver: cfg2 (1M points, 2D order 4, k = 30, uniform weights) from prepare_hoods on a device kNN, with knowns = 0
(cfg2) and with b2_F known and centre folding (cfg2_F, center = 0).  Queries (device tensors, their models found by
the device grid once, I passed explicitly to every timed call):
  transfer  1M points of a second seeded cloud
  cfg5      16M points of a second seeded cloud
Operators: the value, the gradient (2 rows), the Laplacian and all 15 slots.  Per (run, queries, operator): the time of
interp_stencils and of interp_operator, the bytes they move by the formula below and the fraction of the measured HBM
bandwidth that is; the route solve_hoods + interpolate for the same outputs; one applied step E @ f (torch CSR matvec)
against that route.  Times are CUDA-event means over --reps calls after one warm-up call; the working sets are larger
than L2.  A case that does not fit the device memory is reported as not measured.  One JSON line per case; the GPU's
name and power limit are read in the same process.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "python-wlsqm_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import wlsqm_b200 as w  # noqa: E402
from wlsqm_b200.fitter import defs  # noqa: E402

HBM_GBS = 6558.0      # the project's measured HBM bandwidth of a B200 (benchmarks/operator_bench.py)


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # noqa: BLE001
        pl = "unavailable (%s)" % e
    return name, pl


def bytes_formula(nx, models, nk, no, nkn, nops, dim, csr=False):
    """interp_stencils: the blocks of the distinct models touched, 8 (nk + nkn) nr each, plus 8 (dim + 1) per query
    (coordinates and index) read; 8 nops (nk + no) per query written.  interp_operator adds the CSR passes of the node
    operator with one row per query: hoods 4 nk read twice, W written and read back, col 4 and values 8 nops per entry."""
    nr = no - nkn
    read = 8.0 * models * (nk + nkn) * nr + 8.0 * nx * (dim + 1)
    write = 8.0 * nx * nops * (nk + no)
    if not csr:
        return read + write
    nnz = nx * nk + (nx if nkn else 0)
    return read + write + 8.0 * nx * nops * nk + 2 * 4.0 * nx * nk + nnz * (4 + 8.0 * nops)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--n", type=int, default=1_000_000)
    args = ap.parse_args()
    name, pl = card()
    dev = torch.device("cuda", 0)
    n, k, dim, order = args.n, 30, 2, 4
    no = defs.NUMBER_OF_DOFS[dim][order]
    g = torch.Generator(device="cpu").manual_seed(1)
    x = torch.rand((n, dim), generator=g, dtype=torch.float64).to(dev)
    hoods = w.knn_hoods(x, k)
    queries = {"transfer": torch.rand((n, dim), generator=g, dtype=torch.float64).to(dev),
               "cfg5": torch.rand((16 * n, dim), generator=g, dtype=torch.float64).to(dev)}
    lap = np.zeros(no)
    lap[[defs.i2_X2, defs.i2_Y2]] = 1.0
    ops = {"value": (np.eye(no)[[0]], [0]), "gradient": (np.eye(no)[[defs.i2_X, defs.i2_Y]], [defs.i2_X, defs.i2_Y]),
           "laplacian": (lap[None], [defs.i2_X2, defs.i2_Y2]), "all": (np.eye(no), "all")}
    f = torch.rand(n, generator=g, dtype=torch.float64).to(dev)
    lines = []
    for run, knowns in (("cfg2", 0), ("cfg2_F", 1)):
        nkn = bin(knowns).count("1")
        center = 0 if knowns else None
        s = w.ExpertSolver(dim, np.full(n, k, np.int32), np.full(n, order, np.int32), np.full(n, knowns, np.int64),
                           np.full(n, defs.WEIGHT_UNIFORM, np.int32))
        s.prepare_hoods(x, hoods)
        s.prep_interpolate()
        fi = torch.zeros((n, no), dtype=torch.float64, device=dev)
        fi[:, 0] = f
        for qname, xq in queries.items():
            nx = xq.shape[0]
            _, I = s.tree.query(xq)
            models = int(torch.unique(I).numel())
            for oname, (c, diffs) in ops.items():
                out = {"run": run, "queries": qname, "nx": nx, "models_touched": models, "op": oname, "nops": len(c),
                       "n": n, "k": k, "order": order, "knowns": knowns, "fold": center is not None,
                       "gpu": name, "power_limit": pl, "reps": args.reps}
                b_st = bytes_formula(nx, models, k, no, nkn, len(c), dim)
                b_op = bytes_formula(nx, models, k, no, nkn, len(c), dim, csr=True)
                out["bytes_interp_stencils"], out["bytes_interp_operator"] = b_st, b_op
                try:
                    out["interp_stencils_ms"] = timed(lambda: s.interp_stencils(xq, c, I), args.reps)
                    out["interp_stencils_hbm_fraction"] = b_st / (out["interp_stencils_ms"] * 1e-3) / (HBM_GBS * 1e9)
                except (torch.cuda.OutOfMemoryError, RuntimeError, MemoryError) as e:
                    out["interp_stencils_ms"] = "not measured (%s)" % str(e).splitlines()[0][:80]
                torch.cuda.empty_cache()
                E = None
                try:
                    out["interp_operator_ms"] = timed(lambda: s.interp_operator(xq, c, I, center=center), args.reps)
                    out["interp_operator_hbm_fraction"] = b_op / (out["interp_operator_ms"] * 1e-3) / (HBM_GBS * 1e9)
                    E, K, _ = s.interp_operator(xq, c, I, center=center)
                    E = E if isinstance(E, list) else [E]
                except (torch.cuda.OutOfMemoryError, RuntimeError, MemoryError) as e:
                    out["interp_operator_ms"] = "not measured (%s)" % str(e).splitlines()[0][:80]
                torch.cuda.empty_cache()

                def route():
                    s.solve_hoods(f, fi)
                    if diffs == "all":
                        return s.interpolate(xq, diff="all", I=I)[0]
                    return [s.interpolate(xq, diff=int(d), I=I)[0] for d in diffs]
                try:
                    out["route_solve_interpolate_ms"] = timed(route, args.reps)
                except (torch.cuda.OutOfMemoryError, RuntimeError, MemoryError) as e:
                    out["route_solve_interpolate_ms"] = "not measured (%s)" % str(e).splitlines()[0][:80]
                torch.cuda.empty_cache()
                if E is not None:
                    out["step_E_at_f_ms"] = timed(lambda: [e @ f for e in E], args.reps)
                    if isinstance(out["route_solve_interpolate_ms"], float):
                        out["step_speedup_vs_route"] = out["route_solve_interpolate_ms"] / out["step_E_at_f_ms"]
                del E
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
