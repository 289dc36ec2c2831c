"""Several fields on one geometry: ExpertSolver.solve_fields / .solve_hoods_fields against one solve per field.

    python benchmarks/solve_fields_bench.py [--out FILE] [--reps R]

Workloads (device-resident arrays, solvers from prepare_hoods on a device kNN, no knowns):
  cfg2        1M points, 2D order 4, k = 30, ALGO_BASIC and ALGO_ITERATIVE(3), F in {1, 2, 4, 8, 16}
  cfg3        500k points, 3D order 4, k = 60 (the geometry of the project's config 3), ALGO_BASIC, F in {1, 8}
  pack        1M points, 2D order 2, k = 12 (small blocks: the packed kernel), ALGO_BASIC, F in {1, 8}
For each F: solve_fields(fk, fi) against F calls of solve(fk[j], fi[j]) with keep_solution(False) (the single solves
then move the same bytes per field: no solution copy), and solve_hoods_fields(f, fi) against F calls of solve_hoods.
The byte model of an ALGO_BASIC pass is 8 (nr nq + F (nk + no)) bytes per point (operator once, data and results per
field); it is reported with the time it takes at the copy bandwidth measured in the same run (a device-to-device copy
of 4 GB, bytes read + written).  Times are CUDA-event means over --reps calls after one warm-up call; every working set
is far larger than L2.  The outputs of solve_fields are checked bit for bit against the single solves.  One JSON line
per measurement; the GPU's name and power limit are read in the same process.
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


def copy_peak_gbs(dev):
    a = torch.empty(512 * 1024 * 1024, dtype=torch.float64, device=dev)
    b = torch.empty_like(a)
    ms = timed(lambda: b.copy_(a), 20)
    del a, b
    return 2 * 4 * 2 ** 30 / (ms * 1e-3) / 1e9


def run(label, dim, order, k, n, algo, Fs, reps, peak, dev, emit):
    g = torch.Generator(device="cpu").manual_seed(0)
    x = (torch.randint(0, 2 ** 24, (n, dim), generator=g) / 2.0 ** 24).double().to(dev)
    hoods = w.knn_hoods(x, k)
    no = defs.NUMBER_OF_DOFS[dim][order]
    args = (dim, np.full(n, k, np.int32), np.full(n, order, np.int32), np.zeros(n, np.int64), np.full(n, 1, np.int32))
    s = w.ExpertSolver(*args, algorithm=algo, max_iter=3)
    s.prepare_hoods(x, hoods)
    s.keep_solution(False)
    Fmax = max(Fs)
    f = torch.stack([torch.sin((j + 1) * x.sum(dim=1)) for j in range(Fmax)])
    fk_all = torch.stack([f[j][hoods.long()] for j in range(Fmax)])
    fi_ref = torch.zeros((Fmax, n, no), dtype=torch.float64, device=dev)
    fi = torch.zeros_like(fi_ref)
    for F in Fs:
        fk, fr, fo, ff = fk_all[:F], fi_ref[:F], fi[:F], f[:F]

        def single():
            for j in range(F):
                s.solve(fk[j], fr[j])

        def single_hoods():
            for j in range(F):
                s.solve_hoods(ff[j], fr[j])

        t_single = timed(single, reps)
        t_fields = timed(lambda: s.solve_fields(fk, fo), reps)
        same = bool((fo.view(torch.int64) == fr.view(torch.int64)).all())
        t_single_h = timed(single_hoods, reps)
        t_fields_h = timed(lambda: s.solve_hoods_fields(ff, fo), reps)
        same_h = bool((fo.view(torch.int64) == fr.view(torch.int64)).all())
        nq, nr = k, no
        bytes_fields = 8 * (nr * nq + F * (k + no)) * n
        bytes_single = F * 8 * (nr * nq + k + no) * n
        rec = dict(workload=label, algorithm="ITERATIVE(3)" if algo == defs.ALGO_ITERATIVE else "BASIC", F=F, n=n,
                   t_solve_fields_ms=round(t_fields, 4), t_F_solves_ms=round(t_single, 4),
                   speedup=round(t_single / t_fields, 3),
                   t_solve_hoods_fields_ms=round(t_fields_h, 4), t_F_solve_hoods_ms=round(t_single_h, 4),
                   speedup_hoods=round(t_single_h / t_fields_h, 3),
                   model_bytes_per_point_fields=bytes_fields // n, model_bytes_per_point_F_solves=bytes_single // n,
                   model_bound_fields_ms=round(bytes_fields / (peak * 1e9) * 1e3, 4),
                   share_of_bound_fields=round(bytes_fields / (peak * 1e9) * 1e3 / t_fields, 3),
                   share_of_bound_F_solves=round(bytes_single / (peak * 1e9) * 1e3 / t_single, 3),
                   bitwise_equal=same, bitwise_equal_hoods=same_h)
        emit(rec)
    del s
    del fk_all, fi_ref, fi, f, x, hoods
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--quick", action="store_true", help="small sizes (a rehearsal of the script, not a measurement)")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    name, pl = card()
    peak = copy_peak_gbs(dev)
    out = open(a.out, "w") if a.out else None

    def emit(rec):
        rec = dict(rec, gpu=name, power_limit=pl, copy_peak_gbs=round(peak, 1))
        line = json.dumps(rec)
        print(line, flush=True)
        if out:
            out.write(line + "\n")
            out.flush()

    emit(dict(workload="copy_peak", bytes=2 * 4 * 2 ** 30))
    scale = 100 if a.quick else 1
    run("cfg2", 2, 4, 30, 1_000_000 // scale, defs.ALGO_BASIC, [1, 2, 4, 8, 16], a.reps, peak, dev, emit)
    run("cfg2", 2, 4, 30, 1_000_000 // scale, defs.ALGO_ITERATIVE, [1, 2, 4, 8, 16], a.reps, peak, dev, emit)
    run("cfg3", 3, 4, 60, 500_000 // scale, defs.ALGO_BASIC, [1, 8], a.reps, peak, dev, emit)
    run("pack", 2, 2, 12, 1_000_000 // scale, defs.ALGO_BASIC, [1, 8], a.reps, peak, dev, emit)


if __name__ == "__main__":
    main()
