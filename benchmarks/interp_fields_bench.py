"""Several fields at query points: ExpertSolver.interpolate_fields against one interpolate() per field.

    python benchmarks/interp_fields_bench.py [--out FILE] [--reps R] [--quick]

The baseline is the reference's multi-field route: nf guest solvers, guest j holding field j (its last solve() produced
fi[j]), each answering interpolate(); the fields route is one interpolate_fields(x, fi) on the host solver.  Workloads
(device-resident arrays, 2D order 4, k = 30, solvers from prepare_hoods on a device kNN, random queries, models found
once by the device search):
  1. cfg2: 1M models, 16M queries, nearest, one slot and 'all', fi fields-outer and fields-inner, nf in {1, 3, 8}
  2. the same with 100k models (the rows of 8 fields fit in L2)
  3. continuous mode, 1M models, 1M queries, r with ~15 models per ball, nf in {1, 3, 8}
  4. one step at nf = 8, 1M queries: solve_hoods_fields + interpolate_fields against 8 x (solve_hoods + interpolate)
Every shape is warmed up; each measurement is the median over --reps alternated repeats (fields, guests, fields, ...)
of a CUDA-event time, with the minimum and the interquartile range over the median.  Every timed output is compared bit for bit with the
baseline.  Next to each time: the byte model of wlsqm_interp_fields.cu (DRAM bytes of the call) for one field per pass
(the guests) and for the plan it picks.  The GPU's name and power limit are read in the same process.
"""
from __future__ import annotations

import argparse
import math
import subprocess
import sys
from pathlib import Path

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT / "python-wlsqm_b200"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import wlsqm_b200 as w  # noqa: E402


def card():
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:          # noqa: BLE001
        pl = "unavailable (%s)" % e
    return name, pl


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def compare(f_fields, f_guests, reps):
    """alternated repeats after one warm-up of each -> (median fields, stats text, median guests, stats text, outputs).
    A route's previous output is released before its next call, so that the caching allocator serves the next output
    from the same block instead of allocating a second one of up to 15 GB inside the timed window."""
    of, og = f_fields(), f_guests()
    torch.cuda.synchronize()
    tf, tg = [], []
    for _ in range(reps):
        of = None
        t, of = event_ms(f_fields)
        tf.append(t)
        og = None
        t, og = event_ms(f_guests)
        tg.append(t)

    def stats(v):
        q1, med, q3 = np.percentile(v, [25, 50, 75])
        return float(med), "%8.3f ms (min %.3f, IQR %.1f%%)" % (med, min(v), 100 * (q3 - q1) / med)
    (mf, sf), (mg, sg) = stats(tf), stats(tg)
    return mf, sf, mg, sg, of, og


def same_bits(a, b):
    if isinstance(b, list):
        b = torch.stack(b)
    return a.shape == b.shape and bool((a.view(torch.int64) == b.view(torch.int64)).all())


def byte_model(nf, ncases, maxno, nx, rows_per_query, query_bytes, out_bytes, l2, f):
    """DRAM bytes of a call with f fields per pass (interp_fields_per_pass in csrc/wlsqm_interp_fields.cu)"""
    rb = sum(32.0 * math.ceil((off + 8.0 * maxno) / 32.0) for off in (0, 8, 16, 24)) / 4.0
    A = nx * rows_per_query
    U = ncases * -math.expm1(-A / ncases)
    live = min(f, nf) * U * rb
    hit = 1.0 if live <= l2 else l2 / live
    rows = U * rb + (A - U) * rb * (1.0 - hit)
    return nf * (rows + nx * out_bytes) + math.ceil(nf / f) * nx * query_bytes


def plan(nf, *a):
    best_f, best = 1, None
    for f in (1, 2, 4, 8):
        if f > 1 and f // 2 >= nf:
            break
        b = byte_model(nf, *a, f)
        if best is None or b <= best:
            best_f, best = f, b
    return best_f, best


def cloud(n, k, dev, seed=0):
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = (torch.randint(0, 2 ** 24, (n, 2), generator=g) / 2.0 ** 24).double().to(dev)
    hoods = w.knn_hoods(x, k)
    args = (2, np.full(n, k, np.int32), np.full(n, 4, np.int32), np.zeros(n, np.int64), np.full(n, 1, np.int32))
    s = w.ExpertSolver(*args)
    s.prepare_hoods(x, hoods)
    s.prep_interpolate(search='gpu')
    return x, hoods, args, s


def fields_and_guests(s, x, hoods, args, nf):
    """nf fields (solve_fields), and nf guests each solved on its own field"""
    f = torch.stack([torch.sin((j + 1) * x.sum(dim=1)) + 0.1 * torch.cos(7.0 * x[:, 0] * (j + 1)) for j in range(nf)])
    n = x.shape[0]
    fi = torch.zeros((nf, n, 15), dtype=torch.float64, device=x.device)
    s.solve_hoods_fields(f, fi)
    guests = []
    for j in range(nf):
        g = w.ExpertSolver(*args, host=s)
        g.prepare(None, None)
        g.prep_interpolate()
        gi = torch.zeros((n, 15), dtype=torch.float64, device=x.device)
        g.solve(f[j][hoods.long()], gi)
        guests.append(g)
    return f, fi, guests


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r08_interp_fields_bench.txt"))
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--quick", action="store_true", help="small sizes, to rehearse the script")
    a = ap.parse_args()
    dev = torch.device("cuda", 0)
    name, pl = card()
    l2 = torch.cuda.get_device_properties(0).L2_cache_size
    lines = ["# interp_fields_bench on %s, power limit %s, L2 %d MB; medians of %d alternated repeats, IQR = "
             "interquartile range / median; bytes = byte model (GB) with 1 field per pass (guests) / the planned fields per pass"
             % (name, pl, l2 >> 20, a.reps)]

    def emit(s_):
        print(s_, flush=True)
        lines.append(s_)

    scale = 100 if a.quick else 1
    nq = 16_000_000 // scale
    for label, n in (("cfg2 1M models", 1_000_000 // scale), ("100k models", 100_000 // scale)):
        x, hoods, args, s = cloud(n, 30, dev)
        f, fi_all, guests = fields_and_guests(s, x, hoods, args, 8)
        gq = torch.Generator(device="cpu").manual_seed(1)
        xq = torch.rand((nq, 2), generator=gq, dtype=torch.float64).to(dev)
        I = s.tree.query(xq)[1]
        inner_store = fi_all.permute(1, 0, 2).contiguous()
        for nf in (1, 3, 8):
            for diff in (0, 'all'):
                for layout in ("outer", "inner"):
                    fi = fi_all[:nf] if layout == "outer" else inner_store[:, :nf].permute(1, 0, 2)
                    ff = lambda: s.interpolate_fields(xq, fi, diff=diff, I=I)[0]                      # noqa: E731
                    fg = lambda: [guests[j].interpolate(xq, diff=diff, I=I)[0] for j in range(nf)]  # noqa: E731
                    tf, sf, tg, sg, of, og = compare(ff, fg, a.reps)
                    ob = 8.0 * (15 if diff == 'all' else 1)
                    m = (nf, n, 15, nq, 1.0, 24.0, ob, l2)
                    fb, bp = plan(*m)
                    emit("%s  %2d fields  diff=%-3s  fi %-5s  fields %s  guests %s  "
                         "ratio %.3f  bytes %.2f / %.2f GB at %d per pass  bitwise %s"
                         % (label, nf, diff, layout, sf, sg, tf / tg, byte_model(*m, 1) / 1e9,
                            bp / 1e9, fb, same_bits(of, og)))
                    del of, og
                    torch.cuda.empty_cache()
        del guests, xq, I
        torch.cuda.empty_cache()

    # 3. continuous mode and 4. one step, on the cfg2 cloud
    n = 1_000_000 // scale
    x, hoods, args, s = cloud(n, 30, dev)
    f, fi_all, guests = fields_and_guests(s, x, hoods, args, 8)
    nq = 1_000_000 // scale
    xq = torch.rand((nq, 2), generator=torch.Generator(device="cpu").manual_seed(2), dtype=torch.float64).to(dev)
    r = math.sqrt(15.0 / (math.pi * n))
    for nf in (1, 3, 8):
        ff = lambda: s.interpolate_fields(xq, fi_all[:nf], mode='continuous', r=r)[0]                       # noqa: E731
        fg = lambda: [guests[j].interpolate(xq, mode='continuous', r=r)[0] for j in range(nf)]  # noqa: E731
        tf, sf, tg, sg, of, og = compare(ff, fg, a.reps)
        cells = n * (2 * r + 1.0 / math.sqrt(n)) ** 2        # candidates of the cell box (grid cell ~ point spacing)
        m = (nf, n, 15, nq, 15.0, 16.0 + cells * 20.0, 8.0, l2)
        fb, bp = plan(*m)
        emit("continuous 1M models 1M queries r=%.5f  %d fields  fields %s  guests %s  "
             "ratio %.3f  bytes %.2f / %.2f GB at %d per pass  bitwise %s"
             % (r, nf, sf, sg, tf / tg, byte_model(*m, 1) / 1e9, bp / 1e9, fb, same_bits(of, og)))
    I = s.tree.query(xq)[1]
    fi_step = torch.zeros_like(fi_all)
    fi_one = torch.zeros((n, 15), dtype=torch.float64, device=dev)

    def step_fields():
        s.solve_hoods_fields(f, fi_step)
        return s.interpolate_fields(xq, fi_step, I=I)[0]

    def step_single():
        outs = []
        for j in range(8):
            s.solve_hoods(f[j], fi_one)
            outs.append(s.interpolate(xq, I=I)[0])
        return outs

    tf, sf, tg, sg, of, og = compare(step_fields, step_single, a.reps)
    emit("step 1M models 1M queries 8 fields: solve_hoods_fields + interpolate_fields %s  "
         "8 x (solve_hoods + interpolate) %s  ratio %.3f  bitwise %s"
         % (sf, sg, tf / tg, same_bits(of, og)))
    Path(a.out).parent.mkdir(parents=True, exist_ok=True)
    Path(a.out).write_text("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
