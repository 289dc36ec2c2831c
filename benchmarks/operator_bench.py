"""Operator export on one GPU: ExpertSolver.stencils / .operator against the route through `sens`.

    python benchmarks/operator_bench.py [--out FILE] [--reps R] [--n N]

Runs (device-resident inputs, solvers from prepare_hoods on a device kNN):
  cfg2        1M points, 2D order 4, k = 30, knowns = 0
  cfg2_F      the same with b2_F known and centre folding (center = 0)
  cfg3        1M points, 3D order 4, k = 60, knowns = 0 (the geometry of the project's config 3)
First the split of operator(all slots) for cfg3 into device time per kernel (torch.profiler) and wall time.
Per run: the time of stencils(Laplacian) and stencils(all slots), operator_nnz, operator (count + contraction + fill),
the bytes these move by the formula below and their fraction of the measured 6558 GB/s; the "sens route" (solve_hoods
with sens, then CSR assembly in torch) for the Laplacian and for all slots; one applied step D @ f (torch CSR matvec)
against solve_hoods.  Times are CUDA-event means over --reps calls after one warm-up call; the working sets are far
larger than L2.  One JSON line per run; the GPU's name and power limit are read in the same process.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
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

HBM_GBS = 6558.0      # the project's measured HBM bandwidth of this B200 pool


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


def bytes_formula(n, nk, no, nkn, nops, fold):
    """bytes moved: operator blocks read 8 (nk + nkn) nr per case; stencils write W 8 nops nk and K 8 nops no per case;
    the CSR build reads hoods 4 nk twice (count, fill) plus rowptr, writes W and reads it back, writes col 4 and
    values 8 nops per entry (nnz = n nk for distinct kNN lists, + n when folding)"""
    nr = no - nkn
    op = 8.0 * n * (nk + nkn) * nr
    st = op + 8.0 * n * nops * (nk + no)
    nnz = n * nk + (n if fold else 0)
    csr = op + 8.0 * n * nops * (2 * nk + no) + 2 * 4.0 * n * nk + 8.0 * 2 * (n + 1) + nnz * (4 + 8.0 * nops)
    return op, st, csr, nnz


def run(tag, dim, order, k, n, knowns, fold, reps):
    dev = torch.device("cuda", 0)
    g = torch.Generator(device="cpu").manual_seed(1)
    x = torch.rand((n, dim), generator=g, dtype=torch.float64).to(dev)
    hoods = w.knn_hoods(x, k)
    no = defs.NUMBER_OF_DOFS[dim][order]
    nkn = bin(knowns & ((1 << no) - 1)).count("1")
    s = w.ExpertSolver(dim, np.full(n, k, np.int32), np.full(n, order, np.int32), np.full(n, knowns, np.int64),
                       np.full(n, defs.WEIGHT_UNIFORM, np.int32), do_sens=True)
    s.prepare_hoods(x, hoods)
    torch.cuda.synchronize()
    lap = np.zeros(no)
    lap[[defs.i2_X2, defs.i2_Y2] if dim == 2 else [defs.i3_X2, defs.i3_Y2, defs.i3_Z2]] = 1.0
    center = 0 if fold else None
    L = _lib.lib()
    nnz = C.c_int64()
    out = {"run": tag, "n": n, "dim": dim, "order": order, "k": k, "knowns": knowns, "fold": fold}

    # the export
    out["stencils_lap_ms"] = timed(lambda: s.stencils(lap), reps)
    out["stencils_all_ms"] = timed(lambda: s.stencils(np.eye(no)), reps)
    out["operator_nnz_ms"] = timed(lambda: _lib.check(L.wlsqm_solver_operator_nnz(s._handle, -1 if center is None else center,
                                                                                    C.byref(nnz))), reps)
    out["operator_lap_ms"] = timed(lambda: s.operator(lap, center=center), reps)
    out["operator_all_ms"] = timed(lambda: s.operator(np.eye(no), center=center), reps)
    op_b, st_b, csr_b, nnz_f = bytes_formula(n, k, no, nkn, 1, fold)
    _, st_all, csr_all, _ = bytes_formula(n, k, no, nkn, no, fold)
    out["nnz"] = int(nnz.value)
    out["nnz_formula"] = nnz_f
    out["bytes"] = {"operator_blocks": op_b, "stencils_lap": st_b, "stencils_all": st_all, "operator_lap": csr_b,
                    "operator_all": csr_all}
    for key, b in (("stencils_lap", st_b), ("stencils_all", st_all), ("operator_lap", csr_b), ("operator_all", csr_all)):
        out[key + "_hbm_fraction"] = b / (out[key + "_ms"] * 1e-3) / (HBM_GBS * 1e9)

    # the route through sens: solve_hoods with sens, then a CSR over (rows, hoods) in torch
    f = torch.rand(n, generator=g, dtype=torch.float64).to(dev)
    fi = torch.zeros((n, no), dtype=torch.float64, device=dev)
    sens = torch.empty((n, k, no), dtype=torch.float64, device=dev)
    rows = torch.arange(n, device=dev).repeat_interleave(k)
    cols = hoods.reshape(-1).long()

    def sens_route(slots):
        s.solve_hoods(f, fi, sens)
        mats = []
        for sl in slots:
            v = sum(sens[:, :, j] for j in sl).reshape(-1)
            mats.append(torch.sparse_coo_tensor(torch.stack([rows, cols]), v, (n, n)).coalesce().to_sparse_csr())
        return mats
    lap_slots = [[j for j in range(no) if lap[j]]]
    out["sens_route_lap_ms"] = timed(lambda: sens_route(lap_slots), max(1, reps // 2))
    out["sens_route_all_ms"] = timed(lambda: sens_route([[j] for j in range(no)]), max(1, reps // 4))
    del sens
    torch.cuda.empty_cache()

    # one applied step of the Laplacian: torch CSR matvec against a solve_hoods step (device fi, no sens)
    D, _ = s.operator(lap, center=center)
    fcol = f.reshape(-1, 1)
    out["step_csr_matvec_ms"] = timed(lambda: D @ fcol, reps)
    s2 = w.ExpertSolver(dim, np.full(n, k, np.int32), np.full(n, order, np.int32), np.full(n, knowns, np.int64),
                        np.full(n, defs.WEIGHT_UNIFORM, np.int32))
    s2.prepare_hoods(x, hoods)
    out["step_solve_hoods_ms"] = timed(lambda: s2.solve_hoods(f, fi), reps)
    s.close()
    s2.close()
    torch.cuda.empty_cache()
    return out


def profile_split(dim, order, k, n, reps=3):
    """where the time of operator(all slots) goes: device time per kernel name (torch.profiler, CUDA activities) against
    the wall time of the same calls; what is left over is host work, allocation and synchronisation"""
    from torch.profiler import ProfilerActivity, profile
    dev = torch.device("cuda", 0)
    g = torch.Generator(device="cpu").manual_seed(1)
    x = torch.rand((n, dim), generator=g, dtype=torch.float64).to(dev)
    hoods = w.knn_hoods(x, k)
    no = defs.NUMBER_OF_DOFS[dim][order]
    s = w.ExpertSolver(dim, np.full(n, k, np.int32), np.full(n, order, np.int32), np.zeros(n, np.int64),
                       np.full(n, defs.WEIGHT_UNIFORM, np.int32))
    s.prepare_hoods(x, hoods)
    c = np.eye(no)
    s.operator(c)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(reps):
            s.operator(c)
        b.record()
        torch.cuda.synchronize()
    per = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None)
        if t is None:
            t = e.cuda_time_total
        if t > 0:
            per[e.key[:80]] = t / 1e3 / reps
    s.close()
    torch.cuda.empty_cache()
    return {"run": "split_operator_all", "dim": dim, "order": order, "k": k, "n": n, "wall_ms": a.elapsed_time(b) / reps,
            "device_ms_by_name": dict(sorted(per.items(), key=lambda kv: -kv[1]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--n", type=int, default=1_000_000)
    ap.add_argument("--split-only", action="store_true", help="only the per-kernel split of operator(all slots), cfg3")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("operator_bench.py needs a CUDA device")
    name, pl = card()
    lines = []
    split = profile_split(3, 4, 60, a.n)
    split["gpu"], split["power_limit"] = name, pl
    print(json.dumps(split), flush=True)
    lines.append(split)
    for args in () if a.split_only else (("cfg2", 2, 4, 30, a.n, 0, False), ("cfg2_F", 2, 4, 30, a.n, 1, True), ("cfg3", 3, 4, 60, a.n, 0, False)):
        r = run(*args, reps=a.reps)
        r["gpu"], r["power_limit"] = name, pl
        print(json.dumps(r), flush=True)
        lines.append(r)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        with open(a.out, "w") as fh:
            for r in lines:
                fh.write(json.dumps(r) + "\n")


if __name__ == "__main__":
    os.environ.setdefault("PYTHONDONTWRITEBYTECODE", "1")
    main()
