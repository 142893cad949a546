"""The reference's Python-level dispatch surface on top of libtaxidispatch.so (B200, sm_100a).

Host functions mirror the reference's names, argument order and return layouts
(SURVEY.md section 8(b)):

  calculate_cost(distances, demand, cabs)          split.py:123-136, simulate.py:17-33
  solve(n, cost) -> x                              solver.py:11-27   (x[n*cab+cust] in {0,1})
  solve_dispatch(distances, demand, cabs)          split.py:139-155  -> (n, x, cost)
  LCM(n, c, ...)                                   heuristic.py:24-33, split.py:161-175,
                                                   greedy_opt.py:61-82, simulate.py:76-97
  LCM_java(cost)                                   Simulator.java:523-549
  solve_batch(costs) / LCM_batch(costs, ...)       heuristic.py:20-40, python.py:6-25 over many instances
  find_pool(...) / find_pool_all(...) / pool_merge(...)   pool_n.c / findpool.c
  find_pool_pairs_batch(...)                       Simulator.findPool over many instances in one launch
  find_pool_all_batch(...)                         the whole findpool job over many small demand sets in one launch
  find_pool_pairs_exact(...) / find_pool_pairs_exact_batch(...)   the optimum of pool_optimum.py / pool_opt_min.py
  solve_stands_batch(...) / solve_assignment_stands(...)    exact stand-derived solves as S x S transportation problems

PyTorch is used only for device buffers, pinned staging and streams.  All arithmetic runs in the
hand-written CUDA kernels behind the C ABI (include/taxidispatch.h).  There is no CPU fallback:
without the built library or without a CUDA device these functions raise.
"""
from __future__ import annotations

import ctypes
import os
from typing import Optional, Sequence

import numpy as np
import torch

from . import _lib
from ._lib import BIG_COST, INT32_MAX, PAIRS_EXACT_MAX_N, POOL_REC_W, AssignStats, LcmParams, PoolStats, TaxiDispatchError, check

__all__ = ["BIG_COST", "Engine", "calculate_cost", "solve", "solve_dispatch", "solve_full", "solve_assignment", "solve_assignment_stands", "solve_stands_batch", "pack_stands_batch", "LCM", "LCM_heuristic",
           "LCM_split", "LCM_greedy_opt", "LCM_simulate", "LCM_java", "find_pool", "find_pool_all", "find_pool_block",
           "find_pool_pairs", "find_pool_pairs_batch", "find_pool_pairs_exact", "find_pool_pairs_exact_batch", "find_pool_all_batch", "pack_pool_batch", "pool_merge", "pack_batch", "pack_cost_matrices", "run_packed", "run_batch", "solve_batch", "LCM_batch",
           "TaxiDispatchError"]


def _require_cuda():
    if not torch.cuda.is_available():
        raise TaxiDispatchError(_lib.TD_ERR_NO_DEVICE, "taxidispatcher_b200",
                                "torch sees no CUDA device; this engine has no CPU fallback")


def _ptr(t: Optional[torch.Tensor]):
    return ctypes.c_void_p(0 if t is None else t.data_ptr())


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


_PINNED = {}   # numel -> reusable pinned staging buffer (cudaHostAlloc per call costs more than small copies)
COPIED = {"h2d": 0, "d2h": 0}   # bytes the host-facing functions moved over PCIe so far (bench.py reports the per-call difference)


def _d2h(t: torch.Tensor) -> np.ndarray:
    """Device tensor -> numpy, counted."""
    arr = t.cpu().numpy()
    COPIED["d2h"] += arr.nbytes
    return arr


def _d2h_int(t: torch.Tensor) -> int:
    COPIED["d2h"] += t.element_size()
    return int(t.item())


def _h2d_i32(a, pinned: bool = True) -> torch.Tensor:
    """Host array-like -> int32 CUDA tensor through pinned staging (asynchronous copy on the current stream).
    Staging buffers are reused; the stream is synchronised before a buffer is overwritten again."""
    arr = np.ascontiguousarray(np.asarray(a, dtype=np.int32))
    COPIED["h2d"] += arr.nbytes
    if not pinned or arr.size == 0:
        return torch.from_numpy(arr).to("cuda")
    if arr.size > (1 << 22):                       # big matrices: one-off pinned copy
        return torch.from_numpy(arr).pin_memory().to("cuda", non_blocking=True)
    bucket = 1 << max(8, int(arr.size - 1).bit_length())        # power-of-two buckets: few allocations
    slot = _PINNED.get(bucket)
    if slot is None:
        slot = {"buf": torch.empty(bucket, dtype=torch.int32).pin_memory(), "ev": None}
        _PINNED[bucket] = slot
    if slot["ev"] is not None:
        slot["ev"].synchronize()                   # the previous copy out of this buffer has finished
    stage = slot["buf"][: arr.size]
    stage.numpy()[:] = arr.reshape(-1)
    t = stage.to("cuda", non_blocking=True).reshape(arr.shape)
    ev = torch.cuda.Event()
    ev.record()
    slot["ev"] = ev
    return t


def _h2d_i32_many(arrays) -> list:
    """Several small host arrays -> int32 CUDA tensors through ONE pinned staging buffer and ONE asynchronous copy (each
    array starts on a 16-byte boundary: the pool kernels stage their tables with bulk copies).  The per-copy cost of a
    few-KB transfer is its fixed latency, not its bytes."""
    arrs = [np.ascontiguousarray(np.asarray(a, dtype=np.int32)) for a in arrays]
    offs, total = [], 0
    for arr in arrs:
        offs.append(total)
        total += (arr.size + 3) & ~3
    if total == 0 or total > (1 << 22) or any(arr.size == 0 for arr in arrs):
        return [_h2d_i32(arr) for arr in arrs]
    COPIED["h2d"] += sum(arr.nbytes for arr in arrs)
    bucket = 1 << max(8, int(total - 1).bit_length())
    slot = _PINNED.get(("many", bucket))
    if slot is None:
        slot = {"buf": torch.empty(bucket, dtype=torch.int32).pin_memory(), "ev": None}
        _PINNED[("many", bucket)] = slot
    if slot["ev"] is not None:
        slot["ev"].synchronize()
    host = slot["buf"].numpy()
    for arr, off in zip(arrs, offs):
        host[off: off + arr.size] = arr.reshape(-1)
    dev = slot["buf"][:total].to("cuda", non_blocking=True)
    ev = torch.cuda.Event()
    ev.record()
    slot["ev"] = ev
    return [dev[off: off + arr.size].reshape(arr.shape) for arr, off in zip(arrs, offs)]


BATCH_MAX_N = 232   # TD_BATCH_MAX_N: the largest instance the batched kernels hold in one CTA's shared memory
BATCH_CLUSTER_MAX_N = 640   # TD_BATCH_CLUSTER_MAX_N: the largest instance one 8-CTA cluster holds in its shared memory
# run_batch sends the LCMs of fewer mid-size instances than this through single td_lcm calls.  One cluster LCM pays about
# 2 us of cluster barrier and reductions per iteration (1.2 ms for a 600 x 600 instance, flat up to many instances per
# launch), while a single td_lcm call takes 0.39 ms at 600 x 600.  Measured on one NVIDIA B200 at 1000 W
# (profiles/cluster_batch_b200.json): at 600 x 600 the loop wins up to 3 instances (1.11 against 1.20 ms) and the cluster
# from 4 (1.21 against 1.51 ms); at 240 x 240 both take 0.4 ms for 3.  The cluster assignment wins from one instance on.
LCM_CLUSTER_MIN_BATCH = 4
STANDS_MAX_S = _lib.STANDS_MAX_S   # TD_STANDS_MAX_S: the largest stand table td_assign_stands_batch holds
BATCH_LARGE_MAX_N = _lib.BATCH_LARGE_MAX_N   # TD_BATCH_LARGE_MAX_N: one cluster per instance, the matrix in global memory
# run_batch sends the assignments / LCMs of fewer large instances (641 to 2048 rows) than these through single calls.
# Measured on one NVIDIA B200 at 1000 W (profiles/large_batch_b200.json, 1 to 128 instances of 700 / 1300 / 2000 rows,
# U[1,39] and stand-derived).  Assignment: from 2 instances the batch wins on stand-derived costs at every size (2 x
# 2000: 46.7 against 48.1 ms; 8 x 2000: 48.1 against 175 ms), while a lone 2000-row instance loses (46.7 against 25.2
# ms).  U[1,39] instances are cheap for the whole-GPU solver: the batch wins from 8 (700 rows), 16 (1300) and 32 (2000)
# instances and loses at most 6 ms below that, so the stand-derived crossover decides.  LCM: a cluster iteration costs
# about 4.5 us (3.1 ms for 700 rows), a whole-GPU td_lcm call 0.3 ms at 700 and 0.9 ms at 2000 rows, so the batch wins
# from 64 instances at every size and kind (64 x 2000: 46.7 against 55.7 ms) and loses below (32 x 2000: 43.4
# against 28.0 ms).
ASSIGN_LARGE_MIN_BATCH = 2
LCM_LARGE_MIN_BATCH = 64


def pack_batch(costs: Sequence):
    """Square host matrices -> (packed, sizes, offsets, n_max) on the device for Engine.assign_batch / lcm_batch.
    Instance b is stored row-major at packed[offsets[b]:], padded to a multiple of 4 elements; sizes (int32) and offsets
    (int64) travel in the same pinned buffer, so the whole batch is ONE host->device copy."""
    mats = []
    for c in costs:
        a = np.asarray(c)
        if a.ndim != 2 or a.shape[0] != a.shape[1]:
            raise ValueError("pack_batch takes square matrices, got shape %s" % (a.shape,))
        mats.append(a)
    B = len(mats)
    sizes = np.array([a.shape[0] for a in mats], dtype=np.int32)
    offsets = np.zeros(B, dtype=np.int64)
    total = 0
    for b, a in enumerate(mats):
        offsets[b] = total
        total += (a.size + 3) & ~3
    meta = (total + 1) & ~1                               # sizes start here; offsets at an even int32 index (int64 view)
    off_at = (meta + B + 1) & ~1
    words = max(off_at + 2 * B, 4)
    COPIED["h2d"] += words * 4
    bucket = 1 << max(8, int(words - 1).bit_length())
    slot = _PINNED.get(("batch", bucket)) if bucket <= (1 << 24) else None
    if slot is None:
        slot = {"buf": torch.empty(bucket, dtype=torch.int32).pin_memory(), "ev": None}
        if bucket <= (1 << 24):
            _PINNED[("batch", bucket)] = slot
    if slot["ev"] is not None:
        slot["ev"].synchronize()
    host = slot["buf"].numpy()
    for a, o in zip(mats, offsets):
        host[o: o + a.size] = a.reshape(-1)
    host[meta: meta + B] = sizes
    host[off_at: off_at + 2 * B] = offsets.view(np.int32)
    dev = slot["buf"][:words].to("cuda", non_blocking=True)
    ev = torch.cuda.Event()
    ev.record()
    slot["ev"] = ev
    n_max = int(sizes.max()) if B else 0
    return dev[:max(total, 4)], dev[meta: meta + B], dev[off_at: off_at + 2 * B].view(torch.int64), n_max


_NP_OF = {torch.int32: np.int32, torch.int64: np.int64}


class _Arena:
    """Several output tensors carved from ONE device buffer, so that a batch comes back in one device->host copy."""

    def __init__(self, device, parts):
        self.spec, off = [], 0
        for numel, dtype in parts:
            nbytes = int(numel) * np.dtype(_NP_OF[dtype]).itemsize
            self.spec.append((off, nbytes, dtype))
            off += (nbytes + 7) & ~7
        self.buf = torch.empty(max(off, 8), dtype=torch.uint8, device=device)
        self.views = [self.buf[o: o + nb].view(dt) for o, nb, dt in self.spec]

    def host(self):
        h = _d2h(self.buf)
        return [h[o: o + nb].view(_NP_OF[dt]) for o, nb, dt in self.spec]


class Engine:
    """Device-pointer front end: torch CUDA tensors in, torch CUDA tensors out, workspaces cached
    per (operation, size) so that steady-state calls allocate nothing."""

    def __init__(self, device: Optional[int] = None):
        _require_cuda()
        self.lib = _lib.lib()
        self.device = torch.device("cuda", torch.cuda.current_device() if device is None else device)
        self._ws = {}

    # -- scratch --------------------------------------------------------------------------------
    def _workspace(self, key, nbytes: int) -> torch.Tensor:
        """One grow-only scratch buffer per operation (calls are stream-ordered, so reuse across sizes is safe)."""
        ws = self._ws.get(key)
        if ws is None or ws.numel() < nbytes:
            ws = None
            self._ws.pop(key, None)                                   # release before growing
            ws = torch.empty(max(int(nbytes * 5 // 4), 256), dtype=torch.uint8, device=self.device)
            self._ws[key] = ws
        return ws

    # -- K1 ---------------------------------------------------------------------------------------
    def cost_matrix(self, dist: torch.Tensor, cab_to: torch.Tensor, cust_from: torch.Tensor, fill: int = BIG_COST,
                    cutoff: Optional[int] = None, out: Optional[torch.Tensor] = None,
                    rows: Optional[tuple] = None) -> torch.Tensor:
        """Padded n x n matrix, or -- rows=(lo, hi) -- its cab-row block [lo, hi) as a (hi - lo) x n tensor."""
        n_cabs, n_cust = int(cab_to.numel()), int(cust_from.numel())
        n = max(n_cabs, n_cust)
        n_stands = int(dist.shape[0]) if dist.numel() else 0
        lo, hi = (0, n) if rows is None else (int(rows[0]), int(rows[1]))
        if out is None:
            out = torch.empty((hi - lo, n), dtype=torch.int32, device=self.device)
        rc = self.lib.td_cost_matrix_rows(_ptr(dist), n_stands, _ptr(cab_to), n_cabs, _ptr(cust_from), n_cust, int(fill),
                                          -1 if cutoff is None else int(cutoff), lo, hi - lo, _ptr(out), _stream())
        check(rc, "td_cost_matrix_rows")
        return out

    # -- K3 ---------------------------------------------------------------------------------------
    def lcm(self, cost: torch.Tensor, mask_value: int, stop_above: int = INT32_MAX, stop_at_value: int = INT32_MAX,
            sum_below: int = INT32_MAX, residual_size: int = 0, max_iters: int = -1):
        """Returns device tensors (rows[n], cols[n], scal) where scal = int64[2] {total, n_pairs | last_min << 32}.
        Use lcm_host_view() to decode after a synchronisation."""
        n = int(cost.shape[0])
        rows = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)
        cols = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)
        scal = torch.zeros(4, dtype=torch.int32, device=self.device)  # [total lo, total hi, n_pairs, last_min]
        prm = LcmParams(int(mask_value), int(stop_above), int(stop_at_value), int(sum_below), int(residual_size),
                        int(max_iters))
        nbytes = self.lib.td_lcm_workspace_bytes(n)
        ws = self._workspace("lcm", nbytes)
        base = scal.data_ptr()
        rc = self.lib.td_lcm(_ptr(cost), n, ctypes.byref(prm), _ptr(rows), _ptr(cols), ctypes.c_void_p(base + 8),
                             ctypes.c_void_p(base), ctypes.c_void_p(base + 12), _ptr(ws), ws.numel(), _stream())
        check(rc, "td_lcm")
        return rows, cols, scal

    @staticmethod
    def lcm_host_view(rows, cols, scal):
        s = scal.cpu().numpy()
        total = int(np.frombuffer(s[:2].tobytes(), dtype=np.int64)[0])
        k = int(s[2])
        return {"total": total, "n_pairs": k, "last_min": int(s[3]), "rows": rows[:k].cpu().numpy(),
                "cols": cols[:k].cpu().numpy()}

    # -- K2 ---------------------------------------------------------------------------------------
    def assign(self, cost: torch.Tensor, want_x: bool = False, want_stats: bool = False,
               n_real_rows: Optional[int] = None, n_real_cols: Optional[int] = None):
        """Exact optimum of the padded n x n matrix.  n_real_rows / n_real_cols (one of them == n) name the real block of
        an unbalanced instance: the constant padding rows / columns are then not searched (td_assign_exact_rect); the
        objective and the padded output layout are the same either way."""
        n = int(cost.shape[0])
        nr = n if n_real_rows is None else int(n_real_rows)
        nc = n if n_real_cols is None else int(n_real_cols)
        col = torch.empty(max(n, 1), dtype=torch.int32, device=self.device)
        obj = torch.zeros(1, dtype=torch.int64, device=self.device)
        x = torch.empty(n * n, dtype=torch.uint8, device=self.device) if want_x else None
        nbytes = self.lib.td_assign_rect_workspace_bytes(n, nr, nc)
        ws = self._workspace("assign", nbytes)
        st = AssignStats() if want_stats else None
        rc = self.lib.td_assign_exact_rect(_ptr(cost), n, nr, nc, _ptr(col), _ptr(obj), _ptr(x),
                                           ctypes.byref(st) if st is not None else None, _ptr(ws), ws.numel(), _stream())
        check(rc, "td_assign_exact_rect")
        return col[:n], obj, x, st

    def assign_duals(self, n: int, n_real_rows: Optional[int] = None, n_real_cols: Optional[int] = None):
        """Dual potentials (u per cab row, v per customer column; int64 device tensors) of the LAST assign() call."""
        nr = n if n_real_rows is None else int(n_real_rows)
        nc = n if n_real_cols is None else int(n_real_cols)
        u = torch.empty(max(n, 1), dtype=torch.int64, device=self.device)
        v = torch.empty(max(n, 1), dtype=torch.int64, device=self.device)
        ws = self._ws["assign"]
        check(self.lib.td_assign_read_duals(_ptr(ws), n, nr, nc, _ptr(u), _ptr(v), _stream()), "td_assign_read_duals")
        return u[:n], v[:n]

    def assign_certify(self, cost: torch.Tensor, col: torch.Tensor, u: torch.Tensor, v: torch.Tensor,
                       n_real_rows: Optional[int] = None, n_real_cols: Optional[int] = None) -> dict:
        """One sweep over the cost matrix: the complementary-slackness certificate of (col, u, v).  Returns the
        td_assign_certificate fields plus `optimal` (all conditions hold)."""
        n = int(cost.shape[0])
        nr = n if n_real_rows is None else int(n_real_rows)
        nc = n if n_real_cols is None else int(n_real_cols)
        cert = torch.zeros(ctypes.sizeof(_lib.AssignCertificate), dtype=torch.uint8, device=self.device)
        ws = self._workspace("certify", self.lib.td_assign_certify_workspace_bytes(n))
        check(self.lib.td_assign_certify(_ptr(cost), n, nr, nc, _ptr(col), _ptr(u), _ptr(v), _ptr(cert), _ptr(ws), ws.numel(),
                                         _stream()), "td_assign_certify")
        c = _lib.AssignCertificate.from_buffer_copy(cert.cpu().numpy().tobytes())
        out = {f: getattr(c, f) for f, _ in _lib.AssignCertificate._fields_ if f != "reserved"}
        out["optimal"] = (c.min_reduced_cost >= 0 and c.max_matched_slack == 0 and c.sign_violations == 0 and
                          c.dual_objective == c.matched_real_cost)
        return out

    # -- batches (td_assign_exact_batch / td_lcm_batch up to 232, the *_cluster kernels up to 640, *_large up to 2048) --
    def _batch_out(self, out, name, shape, dtype):
        if out is not None and out.get(name) is not None:
            return out[name]
        return torch.empty(shape, dtype=dtype, device=self.device)

    @staticmethod
    def _batch_kernel(n_max: int, name: str) -> str:
        """One CTA per instance up to BATCH_MAX_N, one thread-block cluster per instance with the matrix in its shared
        memory up to BATCH_CLUSTER_MAX_N, and in global memory up to BATCH_LARGE_MAX_N."""
        if n_max <= BATCH_MAX_N:
            return name
        if n_max <= BATCH_CLUSTER_MAX_N:
            return name + "_cluster"
        if n_max <= BATCH_LARGE_MAX_N:
            return name + "_large"
        raise ValueError("batched %s holds instances up to %d rows, got n_max %d" % (name, BATCH_LARGE_MAX_N, n_max))

    def assign_batch(self, packed: torch.Tensor, sizes: torch.Tensor, offsets: torch.Tensor, n_max: int,
                     want_duals: bool = False, out: Optional[dict] = None):
        """Exact optimum of every instance of a pack_batch() buffer, one launch (n_max <= BATCH_LARGE_MAX_N).  Returns
        device tensors (col [B, n_max] int32, objective [B] int64, u, v) -- u / v are [B, n_max] int64 potentials or
        None.  `out` may supply any of them by name ("col", "objective", "u", "v")."""
        name = self._batch_kernel(int(n_max), "td_assign_exact_batch")
        B = int(sizes.numel())
        col = self._batch_out(out, "col", (B, n_max), torch.int32)
        obj = self._batch_out(out, "objective", (B,), torch.int64)
        u = self._batch_out(out, "u", (B, n_max), torch.int64) if want_duals else None
        v = self._batch_out(out, "v", (B, n_max), torch.int64) if want_duals else None
        rc = getattr(self.lib, name)(_ptr(packed), _ptr(sizes), _ptr(offsets), B, int(n_max), _ptr(col), _ptr(obj),
                                     _ptr(u), _ptr(v), _stream())
        check(rc, name)
        return col, obj, u, v

    def lcm_batch(self, packed: torch.Tensor, sizes: torch.Tensor, offsets: torch.Tensor, n_max: int, mask_value: int,
                  stop_above: int = INT32_MAX, stop_at_value: int = INT32_MAX, sum_below: int = INT32_MAX,
                  residual_size: int = 0, max_iters: int = -1, out: Optional[dict] = None):
        """LCM of every instance of a pack_batch() buffer, one launch, the same params for all (n_max <=
        BATCH_LARGE_MAX_N).  Returns device tensors (rows [B, n_max], cols [B, n_max], n_pairs [B] int32, total [B]
        int64, last_min [B] int32); `out` may supply any of them by name."""
        name = self._batch_kernel(int(n_max), "td_lcm_batch")
        B = int(sizes.numel())
        rows = self._batch_out(out, "rows", (B, n_max), torch.int32)
        cols = self._batch_out(out, "cols", (B, n_max), torch.int32)
        npairs = self._batch_out(out, "n_pairs", (B,), torch.int32)
        total = self._batch_out(out, "total", (B,), torch.int64)
        last = self._batch_out(out, "last_min", (B,), torch.int32)
        prm = LcmParams(int(mask_value), int(stop_above), int(stop_at_value), int(sum_below), int(residual_size),
                        int(max_iters))
        rc = getattr(self.lib, name)(_ptr(packed), _ptr(sizes), _ptr(offsets), B, int(n_max), ctypes.byref(prm), _ptr(rows),
                                     _ptr(cols), _ptr(npairs), _ptr(total), _ptr(last), _stream())
        check(rc, name)
        return rows, cols, npairs, total, last

    # -- stand-derived assignment as S x S transportation problems (td_assign_stands_batch) ---------------------------
    def assign_stands_batch(self, dist: torch.Tensor, cab_to: torch.Tensor, cab_off: torch.Tensor, n_c: torch.Tensor,
                            cust_from: torch.Tensor, cust_off: torch.Tensor, n_d: torch.Tensor, n_max: int,
                            fill: int = BIG_COST, cutoff: Optional[int] = None, want_cost: bool = False,
                            want_duals: bool = False, want_stats: bool = False, out: Optional[dict] = None):
        """Exact optimum of every stand-derived instance (include/taxidispatch.h, td_assign_stands_batch), device tensors
        in and out: (col [B, n_max] int32, cost [B, n_max] int32 or None, objective [B] int64, u [B, S], v [B, S] int64
        or None, stats [B, 2] int32 or None).  `out` may supply any of them by name."""
        B, S = int(n_c.numel()), int(dist.shape[0])
        col = self._batch_out(out, "col", (B, n_max), torch.int32)
        cost = self._batch_out(out, "cost", (B, n_max), torch.int32) if want_cost else None
        obj = self._batch_out(out, "objective", (B,), torch.int64)
        u = self._batch_out(out, "u", (B, S), torch.int64) if want_duals else None
        v = self._batch_out(out, "v", (B, S), torch.int64) if want_duals else None
        stats = self._batch_out(out, "stats", (B, 2), torch.int32) if want_stats else None
        nbytes = self.lib.td_assign_stands_workspace_bytes(B, S, int(n_max))
        ws = self._workspace("stands", nbytes)
        rc = self.lib.td_assign_stands_batch(_ptr(dist), S, int(fill), -1 if cutoff is None else int(cutoff), _ptr(cab_to),
                                             _ptr(cab_off), _ptr(n_c), _ptr(cust_from), _ptr(cust_off), _ptr(n_d), B,
                                             int(n_max), _ptr(col), _ptr(cost), _ptr(obj), _ptr(u), _ptr(v), _ptr(stats),
                                             _ptr(ws), ws.numel(), _stream())
        check(rc, "td_assign_stands_batch")
        return col, cost, obj, u, v, stats

    # -- K4 ---------------------------------------------------------------------------------------
    def pool_find(self, demand: torch.Tensor, dist: torch.Tensor, pool_size: int, shard: int = 0, n_shards: int = 8,
                  max_feasible: Optional[int] = None, out: Optional[torch.Tensor] = None, want_stats: bool = True,
                  cnt_out: Optional[torch.Tensor] = None):
        """out: [cap, 9] int32 device rows (cap >= n // pool_size); cnt_out: 1-element int32 device view that
        receives the number of surviving plans (-1: the record list overflowed, only when want_stats=False)."""
        n = int(demand.shape[0])
        n_stands = int(dist.shape[0])
        cap = n // 2 + 1
        if out is None:
            out = torch.empty((cap, POOL_REC_W), dtype=torch.int32, device=self.device)
        cnt = cnt_out if cnt_out is not None else torch.zeros(1, dtype=torch.int32, device=self.device)
        mf = int(max_feasible) if max_feasible is not None else self._ws.get(("pool_mf", n, pool_size), 1 << 21)
        for _ in range(8):
            nbytes = self.lib.td_pool_workspace_bytes(n, n_stands, pool_size, mf)
            ws = self._workspace("pool", nbytes)
            st = PoolStats()
            rc = self.lib.td_pool_find(_ptr(demand), n, _ptr(dist), n_stands, pool_size, shard, n_shards, _ptr(out),
                                       int(out.shape[0]), _ptr(cnt), ctypes.byref(st) if want_stats else None,
                                       _ptr(ws), ws.numel(), mf, _stream())
            if rc == _lib.TD_ERR_CAPACITY and want_stats and st.feasible > mf:
                mf = int(st.feasible) + 1024          # grow the materialised list and retry
                self._ws[("pool_mf", n, pool_size)] = mf
                continue
            check(rc, "td_pool_find")
            return out, cnt, (st if want_stats else None)
        raise TaxiDispatchError(_lib.TD_ERR_CAPACITY, "td_pool_find")

    def pool_find_shards(self, demand: torch.Tensor, dist: torch.Tensor, pool_size: int, shard_begin: int = 0,
                         shard_count: int = 8, n_shards: int = 8, max_feasible: Optional[int] = None,
                         out: Optional[torch.Tensor] = None, counts_out: Optional[torch.Tensor] = None,
                         want_stats: bool = True, defer_stats: bool = False):
        """Consecutive logical shards in one call (one enumeration + one selection launch for all of them).
        out: [shard_count, cap, 9]; counts_out: [shard_count] int32 (device).  Returns (out, counts, stats list).
        defer_stats=True launches asynchronously (single pass, no host round trip) and returns a token for
        pool_read_stats() instead of the stats."""
        n = int(demand.shape[0])
        n_stands = int(dist.shape[0])
        cap = n // 2 + 1
        if out is None:
            out = torch.empty((shard_count, cap, POOL_REC_W), dtype=torch.int32, device=self.device)
        cnt = counts_out if counts_out is not None else torch.zeros(shard_count, dtype=torch.int32, device=self.device)
        key = ("pool_mf", n, pool_size, shard_count)
        mf = int(max_feasible) if max_feasible is not None else self._ws.get(key, (1 << 21) * min(shard_count, 4))
        for _ in range(8):
            nbytes = self.lib.td_pool_shards_workspace_bytes(n, n_stands, pool_size, shard_count, mf)
            ws = self._workspace("pool", nbytes)
            st = (PoolStats * shard_count)()
            rc = self.lib.td_pool_find_shards(_ptr(demand), n, _ptr(dist), n_stands, pool_size, shard_begin, shard_count,
                                              n_shards, _ptr(out), int(out.shape[1]), _ptr(cnt),
                                              st if (want_stats and not defer_stats) else None, _ptr(ws), ws.numel(), mf,
                                              _stream())
            if rc == _lib.TD_ERR_CAPACITY and want_stats:
                need = sum(int(s.feasible) for s in st)
                if need > mf:
                    mf = need + 1024                      # grow the materialised list and retry
                    self._ws[key] = mf
                    continue
            check(rc, "td_pool_find_shards")
            if want_stats and not defer_stats and max_feasible is None and st[0].passes > 1:
                # the feasible set did not fit the record list in one pass: remember a capacity that does (bounded
                # by ~4 GiB per list) so that later calls -- in particular asynchronous ones, which cannot fall back
                # to cost windows -- run single-pass
                need = sum(int(s.feasible) for s in st) + 1024
                self._ws[key] = max(mf, min(need, 1 << 28))
            if defer_stats:
                return out, cnt, (ws, shard_count)
            return out, cnt, (list(st) if want_stats else None)
        raise TaxiDispatchError(_lib.TD_ERR_CAPACITY, "td_pool_find_shards")

    def pool_find_shards_headed(self, demand: torch.Tensor, dist: torch.Tensor, pool_size: int, shard_begin: int,
                                shard_count: int, n_shards: int, out: torch.Tensor, max_feasible: Optional[int] = None):
        """Asynchronous single pass into headed blocks: out is [shard_count, cap + 1, 9] int32 (device), row 0 of every
        block = {count, evaluated lo / hi, feasible lo / hi, ...} (td_pool_find_shards_headed).  Needs a record capacity
        that holds every feasible plan -- remembered by an earlier synchronous pool_find_shards call of the same shape."""
        n = int(demand.shape[0])
        n_stands = int(dist.shape[0])
        cap = int(out.shape[1]) - 1
        key = ("pool_mf", n, pool_size, shard_count)
        mf = int(max_feasible) if max_feasible is not None else self._ws.get(key, (1 << 21) * min(shard_count, 4))
        nbytes = self.lib.td_pool_shards_workspace_bytes(n, n_stands, pool_size, shard_count, mf)
        ws = self._workspace("pool", nbytes)
        rc = self.lib.td_pool_find_shards_headed(_ptr(demand), n, _ptr(dist), n_stands, pool_size, shard_begin, shard_count,
                                                 n_shards, _ptr(out), cap, _ptr(ws), ws.numel(), mf, _stream())
        check(rc, "td_pool_find_shards_headed")
        return out

    @staticmethod
    def _merged_count(m: int, where: str) -> int:
        """The merge's count, or TaxiDispatchError when it is -1 (a row names a customer outside [0, n))."""
        if m < 0:
            raise TaxiDispatchError(_lib.TD_ERR_INVALID, where, "a plan names a customer outside [0, n)")
        return m

    def pool_merge_headed(self, blocks: torch.Tensor, slot_shard: Optional[torch.Tensor], n: int, pool_size: int):
        """blocks [n_slots, cap + 1, 9] headed blocks (device).  Returns (plans, count) device tensors without a host round
        trip; the count is -1 when a row names a customer outside [0, n)."""
        n_slots, cap = int(blocks.shape[0]), int(blocks.shape[1]) - 1
        total = n_slots * cap
        out = torch.empty((max(total, 1), POOL_REC_W), dtype=torch.int32, device=self.device)
        cnt = torch.zeros(1, dtype=torch.int32, device=self.device)
        ws = self._workspace("merge", self.lib.td_pool_merge_workspace_bytes(total, n))
        rc = self.lib.td_pool_merge_headed(_ptr(blocks), _ptr(slot_shard), n_slots, cap, n, pool_size, _ptr(out), _ptr(cnt),
                                           _ptr(ws), ws.numel(), _stream())
        check(rc, "td_pool_merge_headed")
        return out, cnt

    def pool_merge_headed_packed(self, blocks: torch.Tensor, slot_shard: Optional[torch.Tensor], n: int, pool_size: int):
        """Merge of headed blocks with everything the host wants in ONE buffer: row 0 = {merged count}, rows 1..n//pool_size
        = the merged plans, then one header row per block.  One device->host copy completes a whole `findpool` job."""
        n_slots, cap = int(blocks.shape[0]), int(blocks.shape[1]) - 1
        total = n_slots * cap
        keep = n // pool_size + 1                                     # merged plans are customer-disjoint
        pack = torch.empty((1 + max(total, keep) + n_slots, POOL_REC_W), dtype=torch.int32, device=self.device)
        ws = self._workspace("merge", self.lib.td_pool_merge_workspace_bytes(total, n))
        rc = self.lib.td_pool_merge_headed(_ptr(blocks), _ptr(slot_shard), n_slots, cap, n, pool_size,
                                           ctypes.c_void_p(pack.data_ptr() + 4 * POOL_REC_W), _ptr(pack), _ptr(ws), ws.numel(),
                                           _stream())
        check(rc, "td_pool_merge_headed")
        pack[1 + keep: 1 + keep + n_slots] = blocks[:, 0, :]          # the headers ride along (a few hundred bytes)
        host = _d2h(pack[: 1 + keep + n_slots])
        m = self._merged_count(int(host[0, 0]), "td_pool_merge_headed")
        counts, ev, fe = self.headers_host_view(host[1 + keep:])
        return host[1: 1 + m].copy(), counts, ev, fe

    @staticmethod
    def headers_host_view(headers: np.ndarray):
        """headers: [n_slots, 9] int32 header rows -> (counts, evaluated, feasible) int64 arrays"""
        h = np.asarray(headers).astype(np.int64) & 0xFFFFFFFF
        counts = np.asarray(headers)[:, 0].astype(np.int64)
        return counts, h[:, 1] | (h[:, 2] << 32), h[:, 3] | (h[:, 4] << 32)

    def pool_read_stats(self, token):
        """Completes a defer_stats=True call: waits for the stream, returns (stats list, overflowed)."""
        ws, shard_count = token
        st = (PoolStats * shard_count)()
        ov = ctypes.c_int(0)
        check(self.lib.td_pool_read_stats(_ptr(ws), shard_count, st, ctypes.byref(ov), _stream()), "td_pool_read_stats")
        COPIED["d2h"] += int(self.lib.td_pool_read_stats_bytes())
        return list(st), bool(ov.value)

    def pool_pairs(self, frm: torch.Tensor, to: torch.Tensor, dist: torch.Tensor, accept_all: bool = True,
                   max_loss: float = 1.01):
        """Simulator.findPool: returns (pairs [cap,4] = custA, custB, plan, cost; count) device tensors."""
        n = int(frm.numel())
        cap = n // 2 + 1
        out = torch.empty((cap, 4), dtype=torch.int32, device=self.device)
        cnt = torch.zeros(1, dtype=torch.int32, device=self.device)
        nbytes = self.lib.td_pool_pairs_workspace_bytes(n)
        ws = self._workspace("pairs", nbytes)
        rc = self.lib.td_pool_pairs(_ptr(frm), _ptr(to), n, _ptr(dist), int(dist.shape[0]), 1 if accept_all else 0,
                                    float(max_loss), _ptr(out), cap, _ptr(cnt), _ptr(ws), ws.numel(), _stream())
        check(rc, "td_pool_pairs")
        return out, cnt

    def pool_pairs_exact_batch(self, frm: torch.Tensor, to: torch.Tensor, sizes: torch.Tensor, offsets: torch.Tensor,
                               n_max: int, dist: torch.Tensor, accept_all: bool = True, max_loss: float = 1.01,
                               out: Optional[dict] = None):
        """Minimum-cost maximum-cardinality pair matching of every instance (customers sizes[b] at frm / to[offsets[b]:]),
        one launch.  Returns device tensors (rows [B, n_max // 2, 4] int32 = custA, custB, plan, cost in (cost, A*n+B)
        order, n_pairs [B] int32, cost [B] int64); a withdrawn instance has n_pairs -1.  `out` may supply any of them by
        name ("rows", "n_pairs", "cost")."""
        B = int(sizes.numel())
        rows = self._batch_out(out, "rows", (B, n_max // 2, 4), torch.int32)
        npairs = self._batch_out(out, "n_pairs", (B,), torch.int32)
        cost = self._batch_out(out, "cost", (B,), torch.int64)
        ws = self._workspace("pairs_exact", self.lib.td_pool_pairs_exact_workspace_bytes(B, int(n_max)))
        rc = self.lib.td_pool_pairs_exact_batch(_ptr(frm), _ptr(to), _ptr(sizes), _ptr(offsets), B, int(n_max), _ptr(dist),
                                                int(dist.shape[0]), 1 if accept_all else 0, float(max_loss), _ptr(rows),
                                                _ptr(npairs), _ptr(cost), _ptr(ws), ws.numel(), _stream())
        check(rc, "td_pool_pairs_exact_batch")
        return rows, npairs, cost

    def pool_pairs_batch(self, frm: torch.Tensor, to: torch.Tensor, sizes: torch.Tensor, offsets: torch.Tensor, n_max: int,
                         dist: torch.Tensor, accept_all: bool = True, max_loss: float = 1.01, out: Optional[dict] = None):
        """Simulator.findPool's greedy of every instance (the batch layout of pool_pairs_exact_batch), one launch.  Returns
        device tensors (rows [B, n_max // 2, 4] int32 = exactly the rows pool_pairs returns, n_pairs [B] int32, cost [B]
        int64); a withdrawn instance has n_pairs -1.  `out` may supply any of them by name ("rows", "n_pairs", "cost")."""
        B = int(sizes.numel())
        rows = self._batch_out(out, "rows", (B, n_max // 2, 4), torch.int32)
        npairs = self._batch_out(out, "n_pairs", (B,), torch.int32)
        cost = self._batch_out(out, "cost", (B,), torch.int64)
        rc = self.lib.td_pool_pairs_batch(_ptr(frm), _ptr(to), _ptr(sizes), _ptr(offsets), B, int(n_max), _ptr(dist),
                                          int(dist.shape[0]), 1 if accept_all else 0, float(max_loss), _ptr(rows),
                                          _ptr(npairs), _ptr(cost), _stream())
        check(rc, "td_pool_pairs_batch")
        return rows, npairs, cost

    def pool_find_all_batch(self, demand: torch.Tensor, sizes: torch.Tensor, offsets: torch.Tensor, n_max: int,
                            dist: torch.Tensor, pool_size: int, n_shards: int = 8, records_per_shard: int = 4096,
                            out: Optional[dict] = None):
        """The findpool job (every logical shard + the merge) of every instance (sizes[b] demand rows of 5 int32 at row
        offsets[b] of `demand`), one launch.  Returns device tensors (plans [B, n_max // pool_size + 1, 9] int32, n_plans
        [B] int32 (-1 withdrawn, -2 records_per_shard too small), evaluated / feasible [B, n_shards] int64, kept
        [B, n_shards] int32, needed [B] int64).  `out` may supply any of them by name."""
        B = int(sizes.numel())
        plans = self._batch_out(out, "plans", (B, n_max // pool_size + 1, POOL_REC_W), torch.int32)
        n_plans = self._batch_out(out, "n_plans", (B,), torch.int32)
        evaluated = self._batch_out(out, "evaluated", (B, n_shards), torch.int64)
        feasible = self._batch_out(out, "feasible", (B, n_shards), torch.int64)
        kept = self._batch_out(out, "kept", (B, n_shards), torch.int32)
        needed = self._batch_out(out, "needed", (B,), torch.int64)
        ws = self._workspace("pool_batch", self.lib.td_pool_batch_workspace_bytes(B, int(n_shards), int(records_per_shard)))
        rc = self.lib.td_pool_find_all_batch(_ptr(demand), _ptr(sizes), _ptr(offsets), B, int(n_max), _ptr(dist),
                                             int(dist.shape[0]), int(pool_size), int(n_shards), _ptr(plans), _ptr(n_plans),
                                             _ptr(evaluated), _ptr(feasible), _ptr(kept), _ptr(needed), _ptr(ws), ws.numel(),
                                             int(records_per_shard), _stream())
        check(rc, "td_pool_find_all_batch")
        return plans, n_plans, evaluated, feasible, kept, needed

    def pool_merge(self, shard_plans: torch.Tensor, total: int, n: int, pool_size: int):
        out = torch.empty((max(total, 1), POOL_REC_W), dtype=torch.int32, device=self.device)
        cnt = torch.zeros(1, dtype=torch.int32, device=self.device)
        nbytes = self.lib.td_pool_merge_workspace_bytes(total, n)
        ws = self._workspace("merge", nbytes)
        rc = self.lib.td_pool_merge(_ptr(shard_plans), total, n, pool_size, _ptr(out), _ptr(cnt), _ptr(ws), ws.numel(),
                                    _stream())
        check(rc, "td_pool_merge")
        self._merged_count(_d2h_int(cnt), "td_pool_merge")
        return out, cnt


    def pool_merge_padded(self, slot_plans: torch.Tensor, slot_counts: torch.Tensor, slot_shard: Optional[torch.Tensor],
                          n: int, pool_size: int):
        """slot_plans [n_slots, cap, 9], slot_counts [n_slots] (device).  Returns (plans, count) device tensors; waits for
        the count and raises TaxiDispatchError when a row names a customer outside [0, n)."""
        n_slots, cap = int(slot_plans.shape[0]), int(slot_plans.shape[1])
        total = n_slots * cap
        out = torch.empty((max(total, 1), POOL_REC_W), dtype=torch.int32, device=self.device)
        cnt = torch.zeros(1, dtype=torch.int32, device=self.device)
        nbytes = self.lib.td_pool_merge_workspace_bytes(total, n)
        ws = self._workspace("merge", nbytes)
        rc = self.lib.td_pool_merge_padded(_ptr(slot_plans), _ptr(slot_counts), _ptr(slot_shard), n_slots, cap, n, pool_size,
                                           _ptr(out), _ptr(cnt), _ptr(ws), ws.numel(), _stream())
        check(rc, "td_pool_merge_padded")
        self._merged_count(_d2h_int(cnt), "td_pool_merge_padded")
        return out, cnt


_engine: Optional[Engine] = None


def engine() -> Engine:
    global _engine
    if _engine is None:
        _engine = Engine()
    return _engine


# ================================================================================================
# reference-shaped host API
# ================================================================================================
def _cost_device(distances, demand: Sequence, cabs: Sequence, fill: int, cutoff: Optional[int]):
    """Device-resident cost matrix of calculate_cost (None when n == 0)."""
    n_cabs, n_cust = len(cabs), len(demand)
    n = max(n_cabs, n_cust)
    if n == 0:
        return 0, None
    eng = engine()
    dist = _h2d_i32(distances)
    cab_to = _h2d_i32([c[2] for c in cabs]) if n_cabs else torch.empty(0, dtype=torch.int32, device=eng.device)
    cust_from = _h2d_i32([d[1] for d in demand]) if n_cust else torch.empty(0, dtype=torch.int32, device=eng.device)
    if n_cabs and n_cust:
        s = int(dist.shape[0])
        if int(cab_to.max()) >= s or int(cab_to.min()) < 0 or int(cust_from.max()) >= s or int(cust_from.min()) < 0:
            raise IndexError("stand index out of range of the distance table")  # the reference raises IndexError too
    return n, eng.cost_matrix(dist, cab_to, cust_from, fill, cutoff)


def calculate_cost(distances, demand: Sequence, cabs: Sequence, fill: int = BIG_COST, cutoff: Optional[int] = None,
                   as_list: bool = False):
    """split.py:123-136: (n, cost) with cost[c_idx][d_idx] = distances[cab.to][customer.from],
    square-padded with `fill` (big_cost).  cutoff=DROP_TIME gives simulate.py:27 / Simulator.java:509.
    demand / cabs are lists of (id, from, to); indexing is positional.  n == 0 -> (0, 0)
    (simulate.py:21).  cost is an int32 ndarray (list of rows with as_list=True)."""
    n, cost_d = _cost_device(distances, demand, cabs, fill, cutoff)
    if n == 0:
        return 0, 0
    cost = cost_d.cpu().numpy()
    return n, (cost.tolist() if as_list else cost)


def solve_full(n: int, cost):
    """Exact optimum; returns (x, col_of_row, objective, stats).  x is the reference vector."""
    if n == 0:
        return np.zeros(0, np.uint8), np.zeros(0, np.int32), 0, None
    eng = engine()
    c = _h2d_i32(np.asarray(cost).reshape(n, n))
    col, obj, x, st = eng.assign(c, want_x=True, want_stats=True)
    return x.cpu().numpy(), col.cpu().numpy(), int(obj.item()), st


def solve(n: int, cost):
    """solver.py:11-27: `x` with x[n*cab + cust] == 1 for the chosen cells.  n == 0 -> (0, [])
    exactly like solver.py:12."""
    if n == 0:
        return 0, []
    return solve_full(n, cost)[0]


def solve_dispatch(distances, demand, cabs, fill: int = BIG_COST, cutoff: Optional[int] = None):
    """split.py:139-155 / simulate.py:36-53: (n, x, cost).  n == 0 -> (0, [], 0) (simulate.py:38).
    The cost matrix goes from K1 to K2 on the device; the host copy is only the returned value."""
    n, cost_d = _cost_device(distances, demand, cabs, fill, cutoff)
    if n == 0:
        return 0, [], 0
    # every real call is unbalanced (dummy rows / columns of `fill`): only the real block is searched
    _, obj, x, _ = engine().assign(cost_d, want_x=True, n_real_rows=max(len(cabs), 1) if len(cabs) < n else n,
                                   n_real_cols=max(len(demand), 1) if len(demand) < n else n)
    if int(obj.item()) == -(1 << 63):              # the kernel withdraws its result when it gave up (td_assign.cu)
        raise TaxiDispatchError(_lib.TD_ERR_NOT_CONVERGED, "td_assign_exact_rect")
    return n, x.cpu().numpy(), cost_d.cpu().numpy()


def solve_assignment(dist_d: torch.Tensor, cab_to, cust_from, fill: int = BIG_COST, cutoff: Optional[int] = None):
    """K1 + K2 for callers that only need the matching (split.py's range solves, the Simulator): stand indices in,
    (n, col_of_row[n], cost_of_row[n]) out as small host arrays -- the n x n matrix and the n^2 solution vector never
    leave the device.  dist_d is the stand table already on the device (it is shared by every range of a split).
    cost_of_row[i] = cost[i][col_of_row[i]] (== fill for a dummy pairing, split.py:89)."""
    n_cabs, n_cust = len(cab_to), len(cust_from)
    n = max(n_cabs, n_cust)
    if n == 0:
        return 0, np.zeros(0, np.int32), np.zeros(0, np.int32)
    eng = engine()
    cab_d = _h2d_i32(cab_to) if n_cabs else torch.empty(0, dtype=torch.int32, device=eng.device)
    cust_d = _h2d_i32(cust_from) if n_cust else torch.empty(0, dtype=torch.int32, device=eng.device)
    cost_d = eng.cost_matrix(dist_d, cab_d, cust_d, fill, cutoff)
    col, _, _, _ = eng.assign(cost_d, n_real_rows=max(n_cabs, 1) if n_cabs < n else n,
                              n_real_cols=max(n_cust, 1) if n_cust < n else n)
    col_h = _d2h(col)
    if n and int(col_h.min()) < 0:                 # the kernel withdraws the matching when it gave up (td_assign.cu)
        raise TaxiDispatchError(_lib.TD_ERR_NOT_CONVERGED, "td_assign_exact_rect")
    picked = cost_d.gather(1, col.to(torch.int64).unsqueeze(1)).squeeze(1)      # n cells: plumbing, not compute
    return n, col_h, _d2h(picked)


def LCM(n: int, c, mask_value: int = BIG_COST, stop_above: int = INT32_MAX, stop_at_value: int = INT32_MAX,
        sum_below: int = INT32_MAX, residual_size: int = 0, max_iters: int = -1):
    """Generic LCM; c is an n x n matrix (or flat n*n) whose row-major flattening is cost[cab][cust].
    Returns dict(total, n_pairs, rows, cols, last_min)."""
    if n == 0:
        return {"total": 0, "n_pairs": 0, "rows": np.zeros(0, np.int32), "cols": np.zeros(0, np.int32),
                "last_min": INT32_MAX}
    eng = engine()
    cost = _h2d_i32(np.asarray(c).reshape(n, n))
    return Engine.lcm_host_view(*eng.lcm(cost, mask_value, stop_above, stop_at_value, sum_below, residual_size, max_iters))


def _lcm_params(mask_value, stop_above, stop_at_value, sum_below, residual_size, max_iters):
    return dict(mask_value=mask_value, stop_above=stop_above, stop_at_value=stop_at_value, sum_below=sum_below,
                residual_size=residual_size, max_iters=max_iters)


def run_packed(packed: torch.Tensor, sizes: torch.Tensor, offsets: torch.Tensor, n_max: int, ns: Sequence[int],
               assign: bool = True, want_duals: bool = False, lcm: Optional[dict] = None):
    """The launch and read-back half of run_batch for a packed buffer already on the device (pack_batch,
    pack_cost_matrices): one launch per kernel, both reading the same buffer, and one device->host copy.  ns are the
    instance sizes on the host (n_max <= BATCH_LARGE_MAX_N).  Returns (assign results, LCM results) as run_batch."""
    eng = engine()
    B = len(ns)
    parts = []
    if assign:
        parts += [(B * n_max, torch.int32), (B, torch.int64)] + ([(B * n_max, torch.int64)] * 2 if want_duals else [])
    if lcm is not None:
        parts += [(B * n_max, torch.int32), (B * n_max, torch.int32), (B, torch.int32), (B, torch.int64), (B, torch.int32)]
    arena = _Arena(eng.device, parts)
    views = list(arena.views)
    if assign:
        names = ["col", "objective"] + (["u", "v"] if want_duals else [])
        out = {k: views.pop(0) for k in names}
        for k in ("col", "u", "v"):
            if k in out:
                out[k] = out[k].view(B, n_max)
        eng.assign_batch(packed, sizes, offsets, n_max, want_duals=want_duals, out=out)
    if lcm is not None:
        out = {k: views.pop(0) for k in ("rows", "cols", "n_pairs", "total", "last_min")}
        out["rows"], out["cols"] = out["rows"].view(B, n_max), out["cols"].view(B, n_max)
        eng.lcm_batch(packed, sizes, offsets, n_max, out=out, **lcm)
    host = arena.host()                                            # the one read-back of the batch
    res_a = res_l = None
    if assign:
        col, obj = host.pop(0).reshape(B, n_max), host.pop(0)
        u = host.pop(0).reshape(B, n_max) if want_duals else None
        v = host.pop(0).reshape(B, n_max) if want_duals else None
        res_a = []
        for k, n in enumerate(ns):
            r = (col[k, :n].copy(), int(obj[k]))
            res_a.append(r + (u[k, :n].copy(), v[k, :n].copy()) if want_duals else r)
    if lcm is not None:
        rows, cols = host.pop(0).reshape(B, n_max), host.pop(0).reshape(B, n_max)
        npairs, total, last = host.pop(0), host.pop(0), host.pop(0)
        res_l = []
        for k in range(B):
            m = int(npairs[k])
            res_l.append({"total": int(total[k]), "n_pairs": m, "rows": rows[k, :m].copy(), "cols": cols[k, :m].copy(),
                          "last_min": int(last[k])})
    return res_a, res_l


def size_groups(ns: Sequence[int]):
    """Positions of the instances per batched kernel: ([n <= BATCH_MAX_N], [BATCH_MAX_N < n <= BATCH_CLUSTER_MAX_N],
    [BATCH_CLUSTER_MAX_N < n <= BATCH_LARGE_MAX_N], [larger])."""
    small = [b for b, n in enumerate(ns) if n <= BATCH_MAX_N]
    mid = [b for b, n in enumerate(ns) if BATCH_MAX_N < n <= BATCH_CLUSTER_MAX_N]
    large = [b for b, n in enumerate(ns) if BATCH_CLUSTER_MAX_N < n <= BATCH_LARGE_MAX_N]
    huge = [b for b, n in enumerate(ns) if n > BATCH_LARGE_MAX_N]
    return small, mid, large, huge


def batch_routes(ns: Sequence[int], assign: bool = True, lcm: bool = True):
    """How run_batch serves instances of sizes ns: ([(positions, assignment batched, LCM batched)] for every batched
    group that launches, positions whose assignment takes a single call, positions whose LCM takes a single call).  A
    group goes to its batch kernel when it holds at least the kernel's minimum batch (LCM_CLUSTER_MIN_BATCH,
    ASSIGN_LARGE_MIN_BATCH, LCM_LARGE_MIN_BATCH); instances above BATCH_LARGE_MAX_N always take single calls."""
    small, mid, large, huge = size_groups(ns)
    groups, single_a, single_l = [], list(huge) if assign else [], list(huge) if lcm else []
    for group, a_min, l_min in ((small, 1, 1), (mid, 1, LCM_CLUSTER_MIN_BATCH),
                                (large, ASSIGN_LARGE_MIN_BATCH, LCM_LARGE_MIN_BATCH)):
        ga, gl = assign and len(group) >= a_min, lcm and len(group) >= l_min
        if assign and not ga:
            single_a += group
        if lcm and not gl:
            single_l += group
        if group and (ga or gl):
            groups.append((group, ga, gl))
    return groups, sorted(single_a), sorted(single_l)


def _stand_indices(dist_d: torch.Tensor, instances: Sequence):
    """(cab_to, cust_from) pairs of stand index arrays -> (cabs, custs, idx, pos): the int32 host arrays, their
    concatenation (all cab arrays, then all customer arrays, then one pad word) and the start of every array in it.
    Raises IndexError for a stand outside the table, as calculate_cost does."""
    cabs = [np.asarray(c, dtype=np.int32).reshape(-1) for c, _ in instances]
    custs = [np.asarray(d, dtype=np.int32).reshape(-1) for _, d in instances]
    s = int(dist_d.shape[0]) if dist_d.numel() else 0
    for c, d in zip(cabs, custs):
        if len(c) and len(d) and (int(c.max()) >= s or int(c.min()) < 0 or int(d.max()) >= s or int(d.min()) < 0):
            raise IndexError("stand index out of range of the distance table")   # as calculate_cost
    idx = np.concatenate(cabs + custs + [np.zeros(1, np.int32)])
    pos = [0]
    for a in cabs + custs:
        pos.append(pos[-1] + len(a))
    return cabs, custs, idx, pos


def pack_cost_matrices(dist_d: torch.Tensor, instances: Sequence, fill: int = BIG_COST, cutoff: Optional[int] = None,
                       transpose: bool = False):
    """calculate_cost (positional, square-padded with `fill`, optional cutoff) of every (cab_to, cust_from) pair of stand
    index arrays, built by K1 straight into one packed device buffer in the layout of pack_batch: the n x n matrices
    never cross PCIe.  transpose=True builds every matrix transposed (customer rows, cab columns; dist_d must then be the
    transposed stand table).  The index arrays and the sizes / offsets travel in ONE host->device copy.  Returns
    (packed, sizes, offsets, n_max, ns)."""
    eng = engine()
    cabs, custs, idx, pos = _stand_indices(dist_d, instances)
    ns = [max(len(c), len(d)) for c, d in zip(cabs, custs)]
    B = len(ns)
    offsets = np.zeros(B, dtype=np.int64)
    total = 0
    for b, n in enumerate(ns):
        offsets[b] = total
        total += (n * n + 3) & ~3
    off_at = (B + 1) & ~1                                 # offsets at an even int32 index (int64 view)
    meta = np.zeros(off_at + 2 * B + 1, dtype=np.int32)
    meta[:B] = ns
    meta[off_at: off_at + 2 * B] = offsets.view(np.int32)
    idx_d, meta_d = _h2d_i32_many([idx, meta])
    packed = torch.empty(max(total, 4), dtype=torch.int32, device=eng.device)
    for b, n in enumerate(ns):
        if n == 0:
            continue
        cab_d = idx_d[pos[b]: pos[b + 1]]
        cust_d = idx_d[pos[B + b]: pos[B + b + 1]]
        rows, cols = (cust_d, cab_d) if transpose else (cab_d, cust_d)
        eng.cost_matrix(dist_d, rows, cols, fill, cutoff, out=packed[int(offsets[b]): int(offsets[b]) + n * n].view(n, n))
    return packed, meta_d[:B], meta_d[off_at: off_at + 2 * B].view(torch.int64), (max(ns) if B else 0), ns


def pack_stands_batch(instances: Sequence, dist=None):
    """(cab_to, cust_from) stand index arrays of every instance -> the device arguments of Engine.assign_stands_batch,
    in ONE pinned host->device copy: a dict with cab_to, cab_off, n_c, cust_from, cust_off, n_d (device tensors; both
    index arguments view the same concatenated buffer), n_max and ns (host).  With `dist` (host stand table) the table
    travels in the same copy and comes back as "dist"; without it the stand check is left to the kernel (an instance
    with a stand outside the table is withdrawn)."""
    dist_np = None if dist is None else np.ascontiguousarray(np.asarray(dist, dtype=np.int32))
    probe = torch.empty((0, 0)) if dist_np is None else torch.from_numpy(dist_np)
    if dist_np is None:
        cabs = [np.asarray(c, dtype=np.int32).reshape(-1) for c, _ in instances]
        custs = [np.asarray(d, dtype=np.int32).reshape(-1) for _, d in instances]
        idx = np.concatenate(cabs + custs + [np.zeros(1, np.int32)])
    else:
        cabs, custs, idx, _ = _stand_indices(probe, instances)
    B = len(cabs)
    nc = np.array([len(c) for c in cabs], dtype=np.int32)
    nd = np.array([len(d) for d in custs], dtype=np.int32)
    cab_off = np.zeros(B, dtype=np.int64)
    cust_off = np.zeros(B, dtype=np.int64)
    if B:
        cab_off[1:] = np.cumsum(nc[:-1])
        cust_off[:] = int(nc.sum()) + np.concatenate([[0], np.cumsum(nd[:-1])])
    off_at = (2 * B + 1) & ~1
    meta = np.zeros(off_at + 4 * B + 1, dtype=np.int32)
    meta[:B], meta[B: 2 * B] = nc, nd
    meta[off_at: off_at + 2 * B] = cab_off.view(np.int32)
    meta[off_at + 2 * B: off_at + 4 * B] = cust_off.view(np.int32)
    parts = [idx, meta] + ([] if dist_np is None else [dist_np])
    up = _h2d_i32_many(parts)
    idx_d, meta_d = up[0], up[1]
    ns = [int(max(a, b)) for a, b in zip(nc, nd)]
    out = {"cab_to": idx_d, "cust_from": idx_d, "n_c": meta_d[:B], "n_d": meta_d[B: 2 * B],
           "cab_off": meta_d[off_at: off_at + 2 * B].view(torch.int64),
           "cust_off": meta_d[off_at + 2 * B: off_at + 4 * B].view(torch.int64), "n_max": max(ns) if B else 0, "ns": ns}
    if dist_np is not None:
        out["dist"] = up[2]
    return out


def solve_stands_batch(distances, instances: Sequence, fill: int = BIG_COST, cutoff: Optional[int] = None,
                       want_duals: bool = False):
    """Exact optimum of calculate_cost(distances, ...) for every (cab_to, cust_from) pair of stand index arrays, solved
    as S x S transportation problems (td_assign_stands_batch, S <= STANDS_MAX_S): one upload, one call and one read-back,
    no n x n matrix anywhere.  Returns a list of (col_of_row, objective), or (col_of_row, objective, u, v) with the
    stand potentials (u per cab stand, v per customer stand) when want_duals.  Raises IndexError for a stand outside the
    table, as calculate_cost does."""
    eng = engine()
    dist = np.asarray(distances)
    pk = pack_stands_batch(instances, dist)
    B, n_max, S = len(pk["ns"]), pk["n_max"], int(dist.shape[0])
    parts = [(B * n_max, torch.int32), (B, torch.int64)] + ([(B * S, torch.int64)] * 2 if want_duals else [])
    arena = _Arena(eng.device, parts)
    views = list(arena.views)
    out = {"col": views[0].view(B, n_max), "objective": views[1]}
    if want_duals:
        out["u"], out["v"] = views[2].view(B, S), views[3].view(B, S)
    eng.assign_stands_batch(pk["dist"], pk["cab_to"], pk["cab_off"], pk["n_c"], pk["cust_from"], pk["cust_off"], pk["n_d"],
                            n_max, fill, cutoff, want_duals=want_duals, out=out)
    host = arena.host()
    col, obj = host[0].reshape(B, n_max), host[1]
    res = []
    for b, n in enumerate(pk["ns"]):
        r = (col[b, :n].copy(), int(obj[b]))
        res.append(r + (host[2].reshape(B, S)[b].copy(), host[3].reshape(B, S)[b].copy()) if want_duals else r)
    return res


def solve_assignment_stands(dist_d: torch.Tensor, cab_to, cust_from, fill: int = BIG_COST, cutoff: Optional[int] = None):
    """solve_assignment through the stand transportation solver: the same (n, col_of_row[n], cost_of_row[n]) triple
    with the same optimum (possibly another of the tied optima), no n x n matrix built.  dist_d is the stand table on
    the device (n_stands <= STANDS_MAX_S).  IndexError for a stand outside the table (as calculate_cost);
    TaxiDispatchError when the kernel withdraws the instance."""
    n = max(len(cab_to), len(cust_from))
    if n == 0:
        return 0, np.zeros(0, np.int32), np.zeros(0, np.int32)
    eng = engine()
    _stand_indices(dist_d, [(cab_to, cust_from)])
    pk = pack_stands_batch([(cab_to, cust_from)])
    arena = _Arena(eng.device, [(n, torch.int32), (n, torch.int32), (1, torch.int64)])
    col, cost, obj = arena.views
    eng.assign_stands_batch(dist_d, pk["cab_to"], pk["cab_off"], pk["n_c"], pk["cust_from"], pk["cust_off"], pk["n_d"], n,
                            fill, cutoff, out={"col": col.view(1, n), "cost": cost.view(1, n), "objective": obj},
                            want_cost=True)
    col_h, cost_h, obj_h = arena.host()
    if int(obj_h[0]) == -(1 << 63):
        raise TaxiDispatchError(_lib.TD_ERR_INVALID, "td_assign_stands_batch", "instance withdrawn")
    return n, col_h.copy(), cost_h.copy()


def run_batch(costs: Sequence, assign: bool = True, want_duals: bool = False, lcm: Optional[dict] = None):
    """Exact assignment and / or LCM (`lcm` = its keyword parameters) of every square matrix in `costs`.  The instances
    are grouped by size: up to BATCH_MAX_N (one CTA each), up to BATCH_CLUSTER_MAX_N and up to BATCH_LARGE_MAX_N (one
    thread-block cluster each), every group uploaded once and served by one launch per kernel, both kernels reading the
    same packed buffer, and read back in one device->host copy; larger ones, and groups smaller than a kernel's minimum
    batch (batch_routes), take the single-instance path.  Returns (assign results, LCM
    results): lists of (col_of_row, objective[, u, v]) and of LCM() dicts, None for the side not asked for."""
    mats = [np.asarray(c) for c in costs]
    for a in mats:
        if a.ndim != 2 or a.shape[0] != a.shape[1]:
            raise ValueError("run_batch takes square matrices, got shape %s" % (a.shape,))
    groups, single_a, single_l = batch_routes([a.shape[0] for a in mats], assign, lcm is not None)
    res_a = [None] * len(mats) if assign else None
    res_l = [None] * len(mats) if lcm is not None else None
    for group, group_assign, group_lcm in groups:
        packed, sizes, offsets, n_max = pack_batch([mats[b] for b in group])
        ra, rl = run_packed(packed, sizes, offsets, n_max, [mats[b].shape[0] for b in group], group_assign, want_duals,
                            lcm if group_lcm else None)
        for k, b in enumerate(group):
            if group_assign:
                res_a[b] = ra[k]
            if group_lcm:
                res_l[b] = rl[k]
    for b in sorted(set(single_a) | set(single_l)):                # one call each
        a = mats[b]
        eng = engine()
        n = a.shape[0]
        c = _h2d_i32(a)
        if b in single_a:
            col, obj, _, _ = eng.assign(c)
            r = (_d2h(col), _d2h_int(obj))
            if want_duals:
                u, v = eng.assign_duals(n)
                r = r + (_d2h(u), _d2h(v))
            res_a[b] = r
        if b in single_l:
            res_l[b] = Engine.lcm_host_view(*eng.lcm(c, **lcm))
    return res_a, res_l


def solve_batch(costs: Sequence, want_duals: bool = False):
    """Exact optimum of every square matrix in `costs` (python.py:6-25, heuristic.py:37 run over many instances): a list
    of (col_of_row, objective), or (col_of_row, objective, u, v) with the dual potentials when want_duals."""
    return run_batch(costs, assign=True, want_duals=want_duals)[0]


def LCM_batch(costs: Sequence, mask_value: int = BIG_COST, stop_above: int = INT32_MAX, stop_at_value: int = INT32_MAX,
              sum_below: int = INT32_MAX, residual_size: int = 0, max_iters: int = -1):
    """LCM() of every square matrix in `costs` with the same parameters (heuristic.py:24-33 run over many instances):
    a list of the dicts LCM() returns."""
    prm = _lcm_params(mask_value, stop_above, stop_at_value, sum_below, residual_size, max_iters)
    return run_batch(costs, assign=False, lcm=prm)[1]


def LCM_heuristic(n, c, mask: int = 100):
    """heuristic.py:24-33 -> total_cost (mask 100, every value summed)."""
    return LCM(n, c, mask_value=mask)["total"]


def LCM_split(n, c, big_cost: int = BIG_COST):
    """split.py:161-175 -> total_cost (mask big_cost, dummy costs not summed)."""
    return LCM(n, c, mask_value=big_cost, sum_below=big_cost)["total"]


def LCM_greedy_opt(n, c, threshold: int = 10, big_cost: int = BIG_COST):
    """greedy_opt.py:61-82 -> (total_cost, allocated_supply, allocated_demand)."""
    r = LCM(n, c, mask_value=big_cost, stop_above=threshold, sum_below=big_cost)
    return r["total"], r["rows"].tolist(), r["cols"].tolist()


def LCM_simulate(n, c, threshold: int = 20, big_cost: int = BIG_COST):
    """simulate.py:76-97 -> (total_cost, allocated_supply, allocated_demand, allocated)."""
    tot, sup, dem = LCM_greedy_opt(n, c, threshold, big_cost)
    return tot, sup, dem, list(zip(sup, dem))


def LCM_java(cost, big_cost: int = BIG_COST, max_non_lcm: int = 600):
    """Simulator.java:523-549 -> (pairs, LCM_min_val)."""
    cost = np.asarray(cost)
    n = cost.shape[0]
    if n == 0:
        return [], big_cost
    r = LCM(n, cost, mask_value=big_cost, stop_at_value=big_cost, residual_size=max_non_lcm)
    mn = r["last_min"]
    return list(zip(r["rows"].tolist(), r["cols"].tolist())), (big_cost if mn >= big_cost else mn)


def find_pool(demand, dist, pool_size: int, shard: int = 0, n_shards: int = 8):
    """One pool_n process (pool_n.c:209-238): returns (plans [m,9] int32 in the record layout of
    pool_n.c:123-134, stats dict evaluated/feasible/kept)."""
    eng = engine()
    dem = _h2d_i32(np.asarray(demand, dtype=np.int32).reshape(-1, 5))
    d = _h2d_i32(dist)
    out, cnt, st = eng.pool_find(dem, d, pool_size, shard, n_shards)
    m = int(cnt.item())
    return out[:m].cpu().numpy(), {"evaluated": st.evaluated, "feasible": st.feasible, "kept": st.kept,
                                   "rounds": st.rounds, "passes": st.passes}


def find_pool_block(demand, dist, pool_size: int, shard_begin: int, shard_count: int, n_shards: int = 8):
    """Consecutive logical shards in one device call.  Returns [(plans, stats dict)] per shard."""
    if shard_count <= 0:
        return []
    eng = engine()
    dem = _h2d_i32(np.asarray(demand, dtype=np.int32).reshape(-1, 5))
    d = _h2d_i32(dist)
    out, cnt, st = eng.pool_find_shards(dem, d, pool_size, shard_begin, shard_count, n_shards)
    counts = cnt.cpu().numpy()
    plans = out.cpu().numpy()
    return [(plans[s, : int(counts[s])].copy(),
             {"evaluated": st[s].evaluated, "feasible": st[s].feasible, "kept": st[s].kept, "rounds": st[s].rounds,
              "passes": st[s].passes}) for s in range(shard_count)]


def find_pool_pairs(frm, to, dist, accept_all: bool = True, max_loss: float = 1.01):
    """Simulator.findPool (Simulator.java:681-758): list of (custA, custB, plan, cost) in scan order;
    custA / custB are positions in the given arrays; from < 0 marks a removed row."""
    n = len(frm)
    if n < 2:
        return np.zeros((0, 4), np.int32)
    eng = engine()
    out, cnt = eng.pool_pairs(_h2d_i32(frm), _h2d_i32(to), _h2d_i32(dist), accept_all, max_loss)
    return out[: int(cnt.item())].cpu().numpy()


def pack_pairs_batch(instances: Sequence, dist):
    """[(frm, to)] host arrays + the stand table -> (frm, to, sizes, offsets, n_max, dist) on the device for
    Engine.pool_pairs_exact_batch.  Every part travels in ONE pinned buffer and ONE host->device copy."""
    fr = [np.asarray(f, dtype=np.int32).reshape(-1) for f, _ in instances]
    tt = [np.asarray(t, dtype=np.int32).reshape(-1) for _, t in instances]
    for f, t in zip(fr, tt):
        if f.shape != t.shape:
            raise ValueError("frm and to of an instance differ in length")
    d = np.ascontiguousarray(np.asarray(dist, dtype=np.int32))
    B = len(fr)
    sizes = np.array([len(f) for f in fr], dtype=np.int32)
    offsets = np.zeros(B, dtype=np.int64)
    total = 0
    for b, f in enumerate(fr):
        offsets[b] = total
        total += (len(f) + 3) & ~3
    to_at = total
    meta = 2 * total
    off_at = (meta + B + 1) & ~1                          # int64 view: even int32 index
    dist_at = (off_at + 2 * B + 3) & ~3
    words = max(dist_at + d.size, 4)
    COPIED["h2d"] += words * 4
    bucket = 1 << max(8, int(words - 1).bit_length())
    key = ("pairs", bucket)
    slot = _PINNED.get(key) if bucket <= (1 << 24) else None
    if slot is None:
        slot = {"buf": torch.empty(bucket, dtype=torch.int32).pin_memory(), "ev": None}
        if bucket <= (1 << 24):
            _PINNED[key] = slot
    if slot["ev"] is not None:
        slot["ev"].synchronize()
    host = slot["buf"].numpy()
    for f, t, o in zip(fr, tt, offsets):
        host[o: o + len(f)] = f
        host[to_at + o: to_at + o + len(t)] = t
    host[meta: meta + B] = sizes
    host[off_at: off_at + 2 * B] = offsets.view(np.int32)
    host[dist_at: dist_at + d.size] = d.reshape(-1)
    dev = slot["buf"][:words].to("cuda", non_blocking=True)
    ev = torch.cuda.Event()
    ev.record()
    slot["ev"] = ev
    n_max = int(sizes.max()) if B else 0
    return (dev[:max(total, 1)], dev[to_at: to_at + max(total, 1)], dev[meta: meta + B],
            dev[off_at: off_at + 2 * B].view(torch.int64), n_max, dev[dist_at: dist_at + d.size].reshape(d.shape))


def _find_pairs_batches(instances: Sequence, dist, accept_all: bool, max_loss: float, kinds: Sequence[str]):
    """Every (frm, to) instance through each of the pair kernels named in `kinds` ("greedy": td_pool_pairs_batch,
    "exact": td_pool_pairs_exact_batch): one pinned upload, one launch per kind and one read-back for all of them.
    Returns per kind the per-instance rows, or None for an instance the library withdrew."""
    B = len(instances)
    if B == 0:
        return [[] for _ in kinds]
    eng = engine()
    frm, to, sizes, offsets, n_max, d = pack_pairs_batch(instances, dist)
    if n_max > PAIRS_EXACT_MAX_N:
        raise ValueError("an instance has %d customers; the batched 2-passenger pools take at most %d" % (n_max, PAIRS_EXACT_MAX_N))
    cap = n_max // 2
    arena = _Arena(eng.device, [(B * cap * 4, torch.int32), (B, torch.int32), (B, torch.int64)] * len(kinds))
    for k, kind in enumerate(kinds):
        rows_v, np_v, cost_v = arena.views[3 * k: 3 * k + 3]
        launch = {"greedy": eng.pool_pairs_batch, "exact": eng.pool_pairs_exact_batch}[kind]
        launch(frm, to, sizes, offsets, n_max, d, accept_all, max_loss,
               out={"rows": rows_v.view(B, cap, 4), "n_pairs": np_v, "cost": cost_v})
    host = arena.host()                                            # the one read-back of the batch
    out = []
    for k in range(len(kinds)):
        rows, npairs = host[3 * k].reshape(B, cap, 4), host[3 * k + 1]
        out.append([None if npairs[b] < 0 else rows[b, : int(npairs[b])].copy() for b in range(B)])
    return out


def find_pool_pairs_batch(instances: Sequence, dist, accept_all: bool = True, max_loss: float = 1.01):
    """Simulator.findPool for every (frm, to) instance over one stand table: one pinned upload, one launch and one
    read-back.  Returns per instance exactly the array find_pool_pairs returns, or None for an instance the library
    withdrew (a live row whose stand lies outside the table).  Instances hold at most PAIRS_BATCH_MAX_N customers and
    every table entry must lie in [0, 2^22]."""
    return _find_pairs_batches(instances, dist, accept_all, max_loss, ("greedy",))[0]


def find_pool_pairs_exact_batch(instances: Sequence, dist, accept_all: bool = True, max_loss: float = 1.01):
    """The exact 2-passenger pool of every (frm, to) instance over one stand table: one pinned upload, one launch and one
    read-back.  Returns per instance the rows (custA, custB, plan, cost) of a minimum-cost maximum-cardinality pairing
    in (cost, A*n+B) order -- the layout find_pool_pairs returns -- or None for an instance the library withdrew (a
    live row whose stand lies outside the table)."""
    return _find_pairs_batches(instances, dist, accept_all, max_loss, ("exact",))[0]


def find_pool_pairs_exact(frm, to, dist, accept_all: bool = True, max_loss: float = 1.01):
    """The exact counterpart of find_pool_pairs: rows (custA, custB, plan, cost) of a maximum-cardinality pairing of
    minimum total cost, in (cost, A*n+B) order; custA / custB are positions in the given arrays (from < 0: removed)."""
    r = find_pool_pairs_exact_batch([(frm, to)], dist, accept_all, max_loss)[0]
    if r is None:
        raise TaxiDispatchError(_lib.TD_ERR_INVALID, "find_pool_pairs_exact", "a live customer's stand lies outside the table")
    return r


def pool_merge(shard_plans, n: int, pool_size: int):
    """findpool.c:83-108 on shard outputs given in shard order."""
    eng = engine()
    parts = [np.asarray(p, dtype=np.int32).reshape(-1, POOL_REC_W) for p in shard_plans]
    allp = np.concatenate(parts, axis=0) if parts else np.zeros((0, POOL_REC_W), np.int32)
    if len(allp) == 0:
        return allp
    out, cnt = eng.pool_merge(_h2d_i32(allp), len(allp), n, pool_size)
    return out[: int(cnt.item())].cpu().numpy()


class PoolJobGraph:
    """The steady-state `findpool` job of one shape as ONE CUDA graph: host->device copy of the demand and the stand table
    out of a pinned buffer, enumeration + selection of this rank's shards into headed blocks, the merge, and the
    device->host copy of the packed result into a pinned buffer.  A call is then: fill the pinned input, one graph launch,
    one stream synchronisation -- the ~10 launches and copies of the job cost one submission (at 8 GPUs the job takes
    0.45 ms on the devices: queuing it piece by piece from Python takes longer than running it).  When the job is spread
    over ranks the all_gather of the blocks is issued between two graphs (front: copy-in + shards, back: merge + copy-out).  Built by find_pool_all / parallel.find_pool_sharded once the asynchronous path has
    succeeded for the shape (the record capacity is known then); an overflow (count -1) makes the caller drop the graph
    and take the cost-window path."""

    def __init__(self, eng: "Engine", n: int, n_stands: int, pool_size: int, n_shards: int, shard_begin: int,
                 shard_count: int, gather=None, slots: Optional[int] = None, slot_shard: Optional[torch.Tensor] = None):
        self.eng, self.n, self.S, self.k = eng, n, n_stands, pool_size
        dev = eng.device
        cap = n // 2 + 1
        self.cap = cap
        self.dem_words = n * 5
        self.dist_off = (self.dem_words + 3) & ~3                      # 16-byte boundary
        total_in = self.dist_off + n_stands * n_stands
        self.h_in = torch.empty(total_in, dtype=torch.int32).pin_memory()
        self.d_in = torch.empty(total_in, dtype=torch.int32, device=dev)
        slots = shard_count if slots is None else slots
        world_slots = slots if gather is None else gather[1] * slots
        self.blocks = torch.zeros((slots, cap + 1, POOL_REC_W), dtype=torch.int32, device=dev)
        self.all_blocks = self.blocks if gather is None else torch.zeros((world_slots, cap + 1, POOL_REC_W), dtype=torch.int32, device=dev)
        self.keep = n // pool_size + 1
        self.n_slots = world_slots
        total = world_slots * cap
        self.rows = 1 + self.keep + world_slots
        self.pack = torch.zeros((1 + max(total, self.keep) + world_slots, POOL_REC_W), dtype=torch.int32, device=dev)
        self.h_out = torch.empty((self.rows, POOL_REC_W), dtype=torch.int32).pin_memory()
        self.in_bytes = (self.dem_words + n_stands * n_stands) * 4
        self.out_bytes = self.rows * POOL_REC_W * 4
        dem_d = self.d_in[: self.dem_words].reshape(n, 5)
        dist_d = self.d_in[self.dist_off:].reshape(n_stands, n_stands)
        ws_m = eng._workspace("merge", eng.lib.td_pool_merge_workspace_bytes(total, n))
        torch.cuda.synchronize()
        self.gather = gather
        self.graph = torch.cuda.CUDAGraph()
        self.graph_post = None

        def front():
            self.d_in.copy_(self.h_in, non_blocking=True)
            if shard_count > 0:
                eng.pool_find_shards_headed(dem_d, dist_d, pool_size, shard_begin, shard_count, n_shards,
                                            out=self.blocks[:shard_count])

        def back():
            rc = eng.lib.td_pool_merge_headed(_ptr(self.all_blocks), _ptr(slot_shard), world_slots, cap, n, pool_size,
                                              ctypes.c_void_p(self.pack.data_ptr() + 4 * POOL_REC_W), _ptr(self.pack),
                                              _ptr(ws_m), ws_m.numel(), _stream())
            check(rc, "td_pool_merge_headed")
            self.pack[1 + self.keep: 1 + self.keep + world_slots] = self.all_blocks[:, 0, :]
            self.h_out.copy_(self.pack[: self.rows], non_blocking=True)

        if gather is None:
            with torch.cuda.graph(self.graph):
                front()
                back()
        else:
            # the collective stays OUTSIDE the graphs (a captured NCCL kernel keeps the communicator busy at teardown):
            # graph - all_gather - graph, three submissions per job
            with torch.cuda.graph(self.graph):
                front()
            self.graph_post = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph_post):
                back()
        self._slot_shard = slot_shard                                    # keep alive: the graph holds its address
        self._ws_ptrs = (eng._ws["pool"].data_ptr() if shard_count > 0 else 0, ws_m.data_ptr())

    def valid(self) -> bool:
        """The graph holds raw pointers into the engine's grow-only workspaces: a call of another shape may have
        reallocated them, after which the graph must not run again."""
        ws_p, ws_m = self.eng._ws.get("pool"), self.eng._ws.get("merge")
        return (self._ws_ptrs[0] == 0 or (ws_p is not None and ws_p.data_ptr() == self._ws_ptrs[0])) and \
               ws_m is not None and ws_m.data_ptr() == self._ws_ptrs[1]

    def run(self, dem_np: np.ndarray, dist_np: np.ndarray):
        """(merged plans, counts per slot, evaluated per slot, feasible per slot) -- like Engine.pool_merge_headed_packed"""
        host = self.h_in.numpy()
        host[: self.dem_words] = dem_np.reshape(-1)
        host[self.dist_off:] = dist_np.reshape(-1)
        COPIED["h2d"] += self.in_bytes
        self.graph.replay()
        if self.graph_post is not None:
            self.gather[0](self.all_blocks, self.blocks)
            self.graph_post.replay()
        torch.cuda.current_stream().synchronize()
        COPIED["d2h"] += self.out_bytes
        out = self.h_out.numpy()
        m = int(out[0, 0])
        counts, ev, fe = Engine.headers_host_view(out[1 + self.keep:])
        return out[1: 1 + m].copy(), counts, ev, fe


_POOL_GRAPHS = {}          # shape key -> PoolJobGraph, or a success counter before the graph is built


def release_pool_graphs():
    """Drops every captured job graph (they hold raw pointers into the engine's workspaces)."""
    if _POOL_GRAPHS:
        _POOL_GRAPHS.clear()
        if torch.cuda.is_available():
            torch.cuda.synchronize()


def _capture_pool_job(*args, **kwargs):
    """PoolJobGraph, or a counter value that never reaches the capture threshold again when the capture fails (the
    piecewise path keeps serving the shape; the result of the current call has been computed already)."""
    try:
        return PoolJobGraph(*args, **kwargs)
    except Exception:                                     # noqa: BLE001 -- any capture failure means "no graph", never "no result"
        return -(1 << 30)


def _pool_graphs_enabled() -> bool:
    return os.environ.get("TD_POOL_GRAPH", "1") != "0"


def find_pool_all(demand, dist, pool_size: int, n_shards: int = 8):
    """What `findpool` produces (findpool.c:122-176): all logical shards, merged in shard order."""
    eng = engine()
    dem_np = np.asarray(demand, dtype=np.int32).reshape(-1, 5)
    n = dem_np.shape[0]
    stats = {"evaluated": 0, "feasible": 0, "kept_per_shard": [], "rounds": 0}
    fast_key = ("pool_single_pass_ok", n, pool_size, n_shards)
    dist_np = np.ascontiguousarray(np.asarray(dist, dtype=np.int32))
    gkey = ("all", n, dist_np.shape[0], pool_size, n_shards, eng.device.index)
    job = _POOL_GRAPHS.get(gkey)
    if isinstance(job, PoolJobGraph) and not job.valid():
        _POOL_GRAPHS.pop(gkey, None)
        job = None
    if isinstance(job, PoolJobGraph):
        # steady state of a repeated shape: the whole job is one graph launch (PoolJobGraph)
        plans, counts, ev, fe = job.run(dem_np, dist_np)
        if int(counts.min()) >= 0:
            stats.update(evaluated=int(ev.sum()), feasible=int(fe.sum()), kept_per_shard=[int(c) for c in counts], kept=len(plans))
            return plans, stats
        _POOL_GRAPHS.pop(gkey, None)                      # the input outgrew the record list
        eng._ws[fast_key] = False
    dem, d = _h2d_i32_many([dem_np, dist_np])             # one pinned staging buffer, one copy
    if n_shards <= 64 and eng._ws.get(fast_key):
        # steady state: enumeration, selection and merge are queued back to back into headed blocks; ONE device->host copy
        # (merged plans + count + the per-shard counters) and one synchronisation complete the job
        cap = n // 2 + 1
        bkey = ("pool_blocks", n, n_shards)
        blocks = eng._ws.get(bkey)
        if blocks is None:
            blocks = eng._ws[bkey] = torch.zeros((n_shards, cap + 1, POOL_REC_W), dtype=torch.int32, device=eng.device)
        eng.pool_find_shards_headed(dem, d, pool_size, 0, n_shards, n_shards, out=blocks)
        plans, counts, ev, fe = eng.pool_merge_headed_packed(blocks, None, n, pool_size)
        if int(counts.min()) >= 0:
            stats.update(evaluated=int(ev.sum()), feasible=int(fe.sum()), kept_per_shard=[int(c) for c in counts],
                         kept=len(plans))
            if _pool_graphs_enabled() and n > 0 and dist_np.ndim == 2:
                seen = _POOL_GRAPHS.get(gkey, 0) + 1      # second success of the shape: capture the job
                _POOL_GRAPHS[gkey] = seen if seen < 2 else _capture_pool_job(eng, n, dist_np.shape[0], pool_size, n_shards, 0, n_shards)
            return plans, stats
        eng._ws[fast_key] = False                         # input outgrew the record list: cost windows below
        _POOL_GRAPHS.pop(gkey, None)
    parts, counts = [], []
    single = True
    for b in range(0, n_shards, 64):                       # one call serves up to 64 consecutive shards
        cnt_sh = min(64, n_shards - b)
        out, cnt, st = eng.pool_find_shards(dem, d, pool_size, b, cnt_sh, n_shards)
        parts.append(out)
        counts.append(cnt)
        single = single and st[0].passes == 1
        stats["evaluated"] += sum(int(s.evaluated) for s in st)
        stats["feasible"] += sum(int(s.feasible) for s in st)
        stats["rounds"] += int(st[0].rounds)
        stats["kept_per_shard"] += [int(s.kept) for s in st]
    # next time: asynchronous single pass, provided the remembered record capacity can hold every feasible plan
    eng._ws[fast_key] = n_shards <= 64 and (single or eng._ws.get(("pool_mf", n, pool_size, n_shards), 0) > stats["feasible"])
    slot_plans = parts[0] if len(parts) == 1 else torch.cat(parts, dim=0)
    slot_counts = counts[0] if len(counts) == 1 else torch.cat(counts, dim=0)
    merged, cnt = eng.pool_merge_padded(slot_plans, slot_counts, None, n, pool_size)
    m = _d2h_int(cnt)
    stats["kept"] = m
    return _d2h(merged[:m]), stats


POOL_BATCH_MAX_N = _lib.POOL_BATCH_MAX_N
# find_pool_all_batch sends K = 4 instances above this size through find_pool_all.  One CTA per (instance, shard) runs a
# shard's whole enumeration, while find_pool_all spreads one instance over the GPU.  Measured on one NVIDIA B200 at 1000 W
# (profiles/pool_batch_b200.json): 8 x 512 customers take 65.7 ms in the batch kernel against 4.5 ms for the loop of
# find_pool_all; 148 x 300 customers take 30.9 ms against 38.8 ms.  Sizes in between were not measured.
POOL_BATCH_K4_LOOP_N = 300
# Record slices one find_pool_all_batch call may allocate (bytes).  A batch whose rerun would need more goes through
# find_pool_all instance by instance instead.
POOL_BATCH_RECORD_BUDGET = 4 << 30
POOL_BATCH_FIRST_RECORDS = 4096      # records per shard of the first call of a shape (1000 x 100 customers, K = 4: 1778)
_POOL_BATCH_RPS = {}                 # (pool_size, n_shards, n_max rounded up to a power of two) -> largest slice needed so far


def pack_pool_batch(instances: Sequence, dist):
    """[demand n x 5] host arrays + the stand table -> (demand, sizes, offsets, n_max, dist) on the device for
    Engine.pool_find_all_batch: instance b is sizes[b] rows at row offsets[b] of `demand`.  Every part travels in ONE
    pinned buffer and ONE host->device copy."""
    dems = [np.asarray(d, dtype=np.int32).reshape(-1, 5) for d in instances]
    d = np.ascontiguousarray(np.asarray(dist, dtype=np.int32))
    B = len(dems)
    sizes = np.array([len(x) for x in dems], dtype=np.int32)
    offsets = np.zeros(B, dtype=np.int64)
    rows = 0
    for b, x in enumerate(dems):
        offsets[b] = rows
        rows += len(x)
    meta = (rows * 5 + 1) & ~1                            # sizes start here; offsets at an even int32 index (int64 view)
    off_at = (meta + B + 1) & ~1
    dist_at = (off_at + 2 * B + 3) & ~3
    words = max(dist_at + d.size, 4)
    COPIED["h2d"] += words * 4
    bucket = 1 << max(8, int(words - 1).bit_length())
    key = ("pool_batch", bucket)
    slot = _PINNED.get(key) if bucket <= (1 << 24) else None
    if slot is None:
        slot = {"buf": torch.empty(bucket, dtype=torch.int32).pin_memory(), "ev": None}
        if bucket <= (1 << 24):
            _PINNED[key] = slot
    if slot["ev"] is not None:
        slot["ev"].synchronize()
    host = slot["buf"].numpy()
    for x, o in zip(dems, offsets):
        host[5 * o: 5 * o + x.size] = x.reshape(-1)
    host[meta: meta + B] = sizes
    host[off_at: off_at + 2 * B] = offsets.view(np.int32)
    host[dist_at: dist_at + d.size] = d.reshape(-1)
    dev = slot["buf"][:words].to("cuda", non_blocking=True)
    ev = torch.cuda.Event()
    ev.record()
    slot["ev"] = ev
    n_max = int(sizes.max()) if B else 0
    return (dev[: max(rows, 1) * 5].view(-1, 5), dev[meta: meta + B], dev[off_at: off_at + 2 * B].view(torch.int64), n_max,
            dev[dist_at: dist_at + d.size].reshape(d.shape))


def pool_batch_routes(sizes: Sequence[int], pool_size: int):
    """Indices of the instances find_pool_all_batch runs in the batched kernel and of those it sends through
    find_pool_all: above POOL_BATCH_MAX_N customers, or above POOL_BATCH_K4_LOOP_N at K = 4."""
    limit = POOL_BATCH_K4_LOOP_N if pool_size == 4 else POOL_BATCH_MAX_N
    small = [i for i, n in enumerate(sizes) if n <= limit]
    large = [i for i, n in enumerate(sizes) if n > limit]
    return small, large


def pool_batch_records(batch: int, n_shards: int, needed: int, budget: int = POOL_BATCH_RECORD_BUDGET):
    """Records per shard for a batch call whose largest shard materialises `needed` records, or None when the record
    slices of `batch` instances would exceed `budget` bytes."""
    rps = max(int(needed), 1)
    return rps if batch * n_shards * rps * 8 <= budget else None


def _pool_batch_call(dems: Sequence, dist_np: np.ndarray, pool_size: int, n_shards: int, rps: int):
    """One upload, one launch, one read-back.  Per instance (n_plans, plans, stats, needed)."""
    eng = engine()
    B = len(dems)
    demand, sizes, offsets, n_max, d = pack_pool_batch(dems, dist_np)
    rows = n_max // pool_size + 1
    arena = _Arena(eng.device, [(B * rows * POOL_REC_W, torch.int32), (B, torch.int32), (B * n_shards, torch.int64),
                                (B * n_shards, torch.int64), (B * n_shards, torch.int32), (B, torch.int64)])
    v = arena.views
    eng.pool_find_all_batch(demand, sizes, offsets, n_max, d, pool_size, n_shards, rps,
                            out={"plans": v[0].view(B, rows, POOL_REC_W), "n_plans": v[1], "evaluated": v[2].view(B, n_shards),
                                 "feasible": v[3].view(B, n_shards), "kept": v[4].view(B, n_shards), "needed": v[5]})
    plans, n_plans, ev, fe, kept, needed = arena.host()
    plans, ev, fe, kept = plans.reshape(B, rows, POOL_REC_W), ev.reshape(B, n_shards), fe.reshape(B, n_shards), \
        kept.reshape(B, n_shards)
    out = []
    for b in range(B):
        m = int(n_plans[b])
        stats = {"evaluated": int(ev[b].sum()), "feasible": int(fe[b].sum()), "kept_per_shard": [int(c) for c in kept[b]],
                 "kept": m}
        out.append((m, plans[b, : max(m, 0)].copy(), stats, int(needed[b])))
    return out


def _find_pool_all_or_none(dem, dist_np, pool_size: int, n_shards: int):
    try:
        plans, stats = find_pool_all(dem, dist_np, pool_size, n_shards)
    except TaxiDispatchError as e:
        if e.code != _lib.TD_ERR_INVALID:
            raise
        return None
    stats.pop("rounds", None)
    return plans, stats


def find_pool_all_batch(instances: Sequence, dist, pool_size: int, n_shards: int = 8):
    """find_pool_all for every demand set (n x 5 rows) over one stand table.  Returns per instance exactly the plans and
    the evaluated / feasible / kept_per_shard / kept counters find_pool_all gives (its internal `rounds` is not
    reported), or None for an instance the library withdrew (a stand outside the table, or a table entry outside
    [0, 2^22]).  Instances of up to POOL_BATCH_MAX_N customers (POOL_BATCH_K4_LOOP_N at K = 4) run in one batched launch;
    larger ones, and a rerun that would exceed POOL_BATCH_RECORD_BUDGET, go through find_pool_all.  The result does not
    depend on the route."""
    if not 1 <= n_shards <= 64:
        raise ValueError("find_pool_all_batch takes 1 to 64 shards, got %d" % n_shards)
    dist_np = np.ascontiguousarray(np.asarray(dist, dtype=np.int32))
    dems = [np.asarray(d, dtype=np.int32).reshape(-1, 5) for d in instances]
    results = [None] * len(dems)
    small, large = pool_batch_routes([len(x) for x in dems], pool_size)
    for i in large:
        results[i] = _find_pool_all_or_none(dems[i], dist_np, pool_size, n_shards)
    if not small:
        return results
    n_max = max(len(dems[i]) for i in small)
    key = (pool_size, n_shards, 1 << max(n_max - 1, 0).bit_length())
    rps = _POOL_BATCH_RPS.get(key, POOL_BATCH_FIRST_RECORDS)
    rps = max(1, min(rps, POOL_BATCH_RECORD_BUDGET // (8 * n_shards * len(small))))
    redo = []
    for i, (m, plans, stats, needed) in zip(small, _pool_batch_call([dems[i] for i in small], dist_np, pool_size, n_shards, rps)):
        if m == -2:
            redo.append((i, needed))
        elif m >= 0:
            results[i] = (plans, stats)
    if redo:
        need = max(nd for _, nd in redo)
        _POOL_BATCH_RPS[key] = max(_POOL_BATCH_RPS.get(key, 0), need)
        rps = pool_batch_records(len(redo), n_shards, need)
        if rps is None:
            for i, _ in redo:
                results[i] = _find_pool_all_or_none(dems[i], dist_np, pool_size, n_shards)
        else:
            idx = [i for i, _ in redo]
            for i, (m, plans, stats, _) in zip(idx, _pool_batch_call([dems[i] for i in idx], dist_np, pool_size, n_shards, rps)):
                results[i] = (plans, stats) if m >= 0 else None
    return results
