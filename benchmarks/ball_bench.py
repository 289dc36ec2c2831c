"""Fixed-radius neighbourhoods on the device (PointGrid.ball / ball_hoods) against knn_hoods at the same mean k and
cKDTree.query_ball_point on the host.

Workloads: 1M uniform points in 2D with r for a mean of about 30 neighbours, 500k in 3D with a mean of about 60.
For each: grid build, count pass, fill + sort pass, ball_hoods end to end, knn_hoods at the mean k (CUDA events, after
warm-up, inputs resident on the device), and one host cKDTree query (workers=-1).  Candidates visited per member come
from the cell size: the walk reads every point of the cell box [cell(q - r), cell(q + r)], whose expected volume is
(2r + h)^dim, against the ball's volume.  Prints one JSON line per workload, headed by the card and its power limit.

    python benchmarks/ball_bench.py [--reps 20]
"""
import argparse
import ctypes as C
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "python-wlsqm_b200"))


def card():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return out[0] if out else "unknown"
    except Exception:
        return "unknown"


def timed(torch, fn, reps):
    fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    import torch
    from scipy.spatial import cKDTree
    import wlsqm_b200 as wlsqm
    from wlsqm_b200 import _lib
    print(json.dumps({"card": card()}))
    L = _lib.lib()
    for dim, n, mean in ((2, 1_000_000, 30), (3, 500_000, 60)):
        x = np.random.default_rng(0).random((n, dim))
        vol_unit = math.pi if dim == 2 else 4.0 / 3.0 * math.pi
        r = (mean / (vol_unit * n)) ** (1.0 / dim)
        xt = torch.from_numpy(x).cuda()
        t_build = timed(torch, lambda: wlsqm.PointGrid(xt).close(), args.reps)
        g = wlsqm.PointGrid(xt)
        h = g.info()[1]
        rt = torch.tensor([r], dtype=torch.float64, device="cuda")
        rowptr = torch.empty(n + 1, dtype=torch.int64, device="cuda")
        nnz = C.c_int64()

        def count():
            _lib.announce_stream(0)
            _lib.check(L.wlsqm_grid_ball_count(g._handle, None, 0, n, int(rt.data_ptr()), 0, 1, 0,
                                               int(rowptr.data_ptr()), None, C.byref(nnz)))
        t_count = timed(torch, count, args.reps)
        col = torch.empty(nnz.value, dtype=torch.int32, device="cuda")

        def fill(order):
            _lib.announce_stream(0)
            _lib.check(L.wlsqm_grid_ball_csr(g._handle, None, 0, n, int(rt.data_ptr()), 0, 1, 0, order,
                                             int(rowptr.data_ptr()), int(col.data_ptr())))
        t_fill = timed(torch, lambda: fill(0), args.reps)
        t_fill_d = timed(torch, lambda: fill(1), args.reps)
        t_hoods = timed(torch, lambda: wlsqm.ball_hoods(xt, r), args.reps)
        t_knn = timed(torch, lambda: wlsqm.knn_hoods(xt, mean), args.reps)
        tree = cKDTree(x)
        t0 = time.perf_counter()
        ref = tree.query_ball_point(x, r, workers=-1, return_length=True)
        t_ck = time.perf_counter() - t0
        t0 = time.perf_counter()
        tree.query_ball_point(x, r, workers=-1)
        t_ck_lists = time.perf_counter() - t0
        members = nnz.value / n                               # self excluded
        cand = (2 * r + h) ** dim * n                          # expected points in the visited cell box
        out = {"dim": dim, "n": n, "r": r, "mean_members": members, "cell": h,
               "candidates_per_member": cand / (members + 1), "nnz": nnz.value,
               "matches_ckdtree_counts": bool(np.array_equal(np.diff(rowptr.cpu().numpy()), ref - 1)),
               "ms_grid_build": t_build, "ms_count": t_count, "ms_fill_sort_index": t_fill,
               "ms_fill_sort_distance": t_fill_d, "ms_ball_hoods": t_hoods, "ms_knn_hoods_same_k": t_knn,
               "ms_ckdtree_counts_host": t_ck * 1e3, "ms_ckdtree_lists_host": t_ck_lists * 1e3,
               "col_bytes_per_point": 4 * members}
        print(json.dumps(out))
        g.close()


if __name__ == "__main__":
    main()
