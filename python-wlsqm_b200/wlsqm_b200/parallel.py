"""Multi-GPU plumbing: one process per GPU, contiguous case ranges of ONE global batch per rank.

Every case of a batch is independent and all per-case inputs are row-sliced (SURVEY.md 8e), so rank r owns an
``ExpertSolver`` over its contiguous slice ``[lo_r, hi_r)`` of the cases -- the reference's ``prange`` over all cases of
one solver (``expert.pyx:536-557``) cut into ranges -- and ``prepare`` / ``solve`` / ``interpolate`` need no exchange
at all.  The only communication is assembling the global ``fi`` for callers that want the whole field on every rank:

* **fused gather** (CUDA, default when enabled with :meth:`ShardedExpertSolver.enable_fused_gather`): every rank holds
  a copy of the global array in peer-accessible memory (CUDA IPC); the solve kernel stores each row it computes into
  ALL copies over NVLink while it streams the operators, so there is no collective pass at all -- only one tiny
  stream-ordered synchronisation per step (a 4-byte NCCL all-reduce) before rows written by peers are read;
* **collective gather** (:func:`all_gather_rows`): one ``all_gather_into_tensor`` straight into the output for even
  shards (one uneven ``all_gather`` otherwise); shard sizes are known from ``(n, world)`` alone, so the step contains
  no host synchronisation and no Python copy loop.  NCCL over NVLink / NVSwitch on GPUs, gloo in the CPU tests.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

from .fitter.expert import ExpertSolver
from .fitter import defs, opexport
from . import _lib

__all__ = ["shard_range", "shard_ranges", "balanced_shards", "all_gather_rows", "ShardedExpertSolver"]


def shard_range(n: int, rank: int, world: int):
    """contiguous, near-equal split of n cases: rank r owns [lo, hi)"""
    if not (0 <= rank < world):
        raise ValueError("rank must be in [0, world)")
    base, rem = divmod(int(n), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_ranges(n: int, world: int):
    """[(lo, hi)] of every rank (what each rank can compute for itself: no exchange of sizes is ever needed)"""
    return [shard_range(n, r, world) for r in range(world)]


def balanced_shards(cost, world: int):
    """contiguous split of heterogeneous cases balancing sum(cost) per rank (cost ~ nr^2 nk per case)
    -> list of (lo, hi).  SURVEY.md 8e: balance shards by work, not by case count."""
    cost = np.asarray(cost, dtype=np.float64)
    n = len(cost)
    cum = np.concatenate([[0.0], np.cumsum(cost)])
    cuts = [0]
    for r in range(1, world):
        target = cum[-1] * r / world
        cuts.append(int(min(max(np.searchsorted(cum, target), cuts[-1]), n)))
    cuts.append(n)
    return [(cuts[r], cuts[r + 1]) for r in range(world)]


def case_cost(dimension, nk, order, knowns):
    """work estimate per case for balanced_shards: nr^2 * nk"""
    no = np.asarray(defs.NUMBER_OF_DOFS[dimension], dtype=np.int64)[np.asarray(order, dtype=np.int64)]
    kn = np.asarray(knowns, dtype=np.int64) & ((np.int64(1) << no) - 1)
    nkn = np.zeros(len(no), dtype=np.int64)
    for b in range(int(no.max()) if len(no) else 0):
        nkn += (kn >> b) & 1
    nr = no - nkn
    return (nr.astype(np.float64) ** 2) * np.asarray(nk, dtype=np.float64)


def all_gather_rows(local, ranges, out=None, group=None):
    """Gather the row slices of every rank into the full (n_total, ...) tensor on every rank.

    ``local``: this rank's rows; ``ranges``: the ``[(lo, hi)]`` of all ranks (``shard_ranges`` or ``balanced_shards`` --
    known on every rank without communication); ``out``: optional preallocated result.  Even shards: one
    ``all_gather_into_tensor`` straight into ``out``.  Uneven shards: one ``all_gather`` into views of ``out`` (NCCL), or
    a padded gather where the backend needs equal sizes (gloo).  No ``.item()``, no host synchronisation."""
    import torch
    import torch.distributed as dist
    world = dist.get_world_size(group)
    if len(ranges) != world:
        raise ValueError("ranges must list one (lo, hi) per rank")
    n_total = ranges[-1][1]
    counts = [hi - lo for lo, hi in ranges]
    me = dist.get_rank(group)
    if local.shape[0] != counts[me]:
        raise ValueError("this rank holds %d rows, its range has %d" % (local.shape[0], counts[me]))
    tail = tuple(local.shape[1:])
    if out is None:
        out = torch.empty((n_total,) + tail, dtype=local.dtype, device=local.device)
    local = local.contiguous()
    if len(set(counts)) == 1:
        dist.all_gather_into_tensor(out, local, group=group)
        return out
    views = [out[lo:hi] for lo, hi in ranges]
    if dist.get_backend(group) == "nccl":
        dist.all_gather(views, local, group=group)          # uneven sizes: grouped broadcasts inside one NCCL group call
        return out
    longest = max(counts)
    pad = torch.zeros((longest,) + tail, dtype=local.dtype, device=local.device)
    pad[:local.shape[0]] = local
    buf = torch.empty((world * longest,) + tail, dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(buf, pad, group=group)
    for r, (lo, hi) in enumerate(ranges):
        out[lo:hi] = buf[r * longest:r * longest + (hi - lo)]
    return out


class _CudaBuffer:
    """a raw device allocation seen by torch through ``__cuda_array_interface__`` (the fused gather's global array)"""

    def __init__(self, ptr, shape, row_stride=None):
        self.ptr, self.shape = int(ptr), tuple(int(s) for s in shape)
        self.strides = None if row_stride is None or row_stride == self.shape[1] else (8 * int(row_stride), 8)

    @property
    def __cuda_array_interface__(self):
        return {"shape": self.shape, "typestr": "<f8", "data": (self.ptr, False), "version": 2, "strides": self.strides}


class ShardedExpertSolver:
    """An ``ExpertSolver`` over this rank's contiguous slice of a global batch.

    Takes the GLOBAL metadata arrays; ``prepare`` / ``solve`` / ``interpolate`` take either global arrays
    (sliced here, no copy) or arrays that already hold just the local rows (``local=True``)."""

    def __init__(self, dimension, nk, order, knowns, weighting_method, *, rank, world, device=None, balance=False,
                 **kwargs):
        nk, order = np.asarray(nk), np.asarray(order)
        knowns, weighting_method = np.asarray(knowns), np.asarray(weighting_method)
        self.n_total = len(nk)
        if balance:
            self.ranges = balanced_shards(case_cost(dimension, nk, order, knowns), world)
        else:
            self.ranges = shard_ranges(self.n_total, world)
        self.lo, self.hi = self.ranges[rank]
        sl = slice(self.lo, self.hi)
        self.rank, self.world = rank, world
        self.solver = ExpertSolver(dimension, np.ascontiguousarray(nk[sl]), np.ascontiguousarray(order[sl]),
                                   np.ascontiguousarray(knowns[sl]), np.ascontiguousarray(weighting_method[sl]),
                                   device=device, **kwargs)
        self.maxno = int(defs.NUMBER_OF_DOFS[int(dimension)][int(order.max())]) if self.n_total else 1     # of the GLOBAL batch
        self.fi_global = None          # fused gather: torch view of this rank's copy of the global solution
        self._own = None
        self._peers = []
        self._sync = None

    def _rows(self, a, local):
        return a if (local or a is None) else a[self.lo:self.hi]

    def prepare(self, xi, xk, local=False):
        return self.solver.prepare(self._rows(xi, local), self._rows(xk, local))

    def solve(self, fk, fi, sens=None, local=False):
        return self.solver.solve(self._rows(fk, local), self._rows(fi, local), self._rows(sens, local))

    # -- neighbourhoods as index lists: replicated points, one all-gather of the per-point data per step (SURVEY 8e) --
    def prepare_hoods(self, x, hoods, local=False):
        """``x``: the FULL point cloud, replicated on every rank (16 MB per million 2D points; the neighbours of a
        contiguous case range may lie anywhere in index space unless the points are spatially sorted -- the "halo");
        ``hoods``: the global (n_total, k) int32 index lists into ``x`` (or this rank's rows with ``local=True``).
        The origins of this rank's cases are ``x[lo:hi]``."""
        return self.solver.prepare_hoods(x, self._rows(hoods, local), xi=x[self.lo:self.hi])

    def solve_hoods(self, f, fi, sens=None, local=False, f_is_local=False, group=None):
        """``f``: one value per point of the full cloud (replicated), or -- ``f_is_local=True`` -- only this rank's
        slice ``f[lo:hi]`` (what a time-stepping code owns), which is all-gathered first: the one exchange of a step,
        8 bytes per point over NCCL.  ``fi`` / ``sens``: global arrays (sliced here) or local rows (``local=True``)."""
        if f_is_local:
            f = all_gather_rows(f, self.ranges, group=group)
        return self.solver.solve_hoods(f, self._rows(fi, local), self._rows(sens, local))

    def operator(self, coeffs, fold_center=False):
        """This rank's row block ``[lo, hi)`` of the global sparse operator (``ExpertSolver.operator``) after
        ``prepare_hoods``, with global column indices: stacking the blocks of all ranks gives the unsharded matrix.
        ``coeffs`` are rows over the GLOBAL batch's max no; K comes back with that width.  ``fold_center``: the
        origins of this rank's cases are ``x[lo:hi]``, so the known-F weight of case lo + i goes to column lo + i."""
        c, squeeze = opexport.coefficient_rows(coeffs, self.maxno)
        c = c[:, :self.solver._maxno]       # slots beyond this rank's largest model are ignored by all its cases
        D, K = self.solver.operator(c[0] if squeeze else c, center=self.lo if fold_center else None)
        pad = self.maxno - K.shape[-1]
        if pad:
            if _lib._is_torch_tensor(K):
                import torch
                K = torch.nn.functional.pad(K, (0, pad))
            else:
                K = np.pad(K, [(0, 0)] * (K.ndim - 1) + [(0, pad)])
        return D, K

    def gather(self, local_rows, out=None, group=None):
        """collective all-gather of a per-rank result (e.g. the local fi tensor) into the global array"""
        return all_gather_rows(local_rows, self.ranges, out=out, group=group)

    # -- fused gather: the solve kernel stores its rows into every GPU's copy of the global fi over NVLink ---------------
    def enable_fused_gather(self, group=None):
        """Allocate this rank's copy of the global ``fi`` (n_total x max no) in peer-accessible memory, exchange the IPC
        handles, and make ``solve`` / ``solve_hoods`` store every row into all copies.  Returns ``self.fi_global``
        (a CUDA tensor).  After a solve call :meth:`sync_gather` before reading rows owned by other ranks."""
        import torch
        import torch.distributed as dist
        if self.world > 8:
            raise ValueError("the fused gather serves the GPUs of one NVSwitch domain (<= 8)")
        L = _lib.lib()
        dev = self.solver.device
        # rows padded to whole 128 B lines where that costs <= 10 % (2D order 4: 15 -> 16 doubles): full-line NVLink writes
        stride = -(-self.maxno // 16) * 16
        if stride > 32 or stride > 1.1 * self.maxno or os.environ.get("WLSQM_GATHER_PAD", "1") == "0":
            stride = self.maxno
        self.gather_stride = stride
        nbytes = max(1, self.n_total * stride * 8)
        ptr, handle = C.c_void_p(), (C.c_char * 64)()
        _lib.check(L.wlsqm_peer_alloc(dev, nbytes, C.byref(ptr), handle))
        self._own = ptr
        handles = [None] * self.world
        if self.world > 1:
            dist.all_gather_object(handles, bytes(handle.raw), group=group)
        else:
            handles[0] = bytes(handle.raw)
        bases = (C.c_void_p * self.world)()
        for r in range(self.world):
            if r == self.rank:
                bases[r] = ptr.value
            else:
                p = C.c_void_p()
                _lib.check(L.wlsqm_peer_open(dev, handles[r], C.byref(p)))
                self._peers.append(p)
                bases[r] = p.value
        _lib.check(L.wlsqm_solver_set_gather(self.solver._handle, self.world, bases, self.lo, stride))
        self.fi_global = torch.as_tensor(_CudaBuffer(ptr.value, (self.n_total, self.maxno), stride), device=torch.device("cuda", dev))
        self._sync = torch.zeros(1, dtype=torch.int32, device=self.fi_global.device)
        self._group = group
        if self.world > 1:
            dist.barrier(group=group)      # every rank has mapped every copy before the first store
        return self.fi_global

    def sync_gather(self):
        """stream-ordered synchronisation of the ranks after a step of the fused gather (one 4-byte all-reduce): rows
        stored by peers are visible to work queued on the current stream afterwards"""
        if self.world > 1:
            import torch.distributed as dist
            dist.all_reduce(self._sync, group=self._group)

    def disable_fused_gather(self):
        L = _lib.lib()
        if self._own is None:
            return
        if self.solver._handle is not None:
            L.wlsqm_solver_set_gather(self.solver._handle, 0, None, 0, 0)
            self.solver.synchronize()
        if self.world > 1:
            import torch.distributed as dist
            try:
                dist.barrier(group=self._group)     # nobody is still storing into a copy that is about to go away
            except Exception:
                pass
        for p in self._peers:
            L.wlsqm_peer_close(p)
        self._peers = []
        self.fi_global = None
        L.wlsqm_peer_free(self._own)
        self._own = None

    def close(self):
        try:
            self.disable_fused_gather()
        finally:
            self.solver.close()
