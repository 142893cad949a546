"""The reference LCM bodies, lifted out of their scripts.  TEST INFRASTRUCTURE ONLY.

The reference functions are pure numpy but live in scripts whose first line imports cvxopt
(absent here), so they cannot be imported; each function below follows its source line by line
in behaviour (same argmin, same masking, float64 like `matrix(..., tc='d')`).
Parity status: PINNED (these ARE the reference algorithm, executed by numpy).
"""
from __future__ import annotations

import ctypes

import numpy as np

from . import _clib

BIG_COST = 250000
INT32_MAX = 2**31 - 1


def lcm_heuristic(n, c, mask=100.0):
    """heuristic.py:24-33.  c: flat n*n costs (row-major n*row+col).  Returns (total, rows, cols)."""
    d = np.array(c, dtype=np.float64).reshape(-1).copy()
    total_cost = 0.0
    rows, cols = [], []
    for _ in range(n):
        elem = int(d.argmin(0))                # heuristic.py:27
        total_cost += d[elem]                  # :28
        row = int(elem / n)                    # :29
        col = elem - row * n                   # :30
        rows.append(row)
        cols.append(col)
        d[n * row: n * row + n] = mask         # :32
        d[col::n] = mask                       # :33
    return total_cost, rows, cols


def lcm_split(n, c, big_cost=BIG_COST):
    """split.py:161-175: mask big_cost, dummy costs not summed (:167).  Returns (total, rows, cols)."""
    d = np.array(c, dtype=np.float64).flatten()
    total_cost = 0.0
    rows, cols = [], []
    for _ in range(n):
        elem = int(d.argmin(0))
        if d[elem] < big_cost:
            total_cost += d[elem]
        row = int(elem / n)
        col = elem - row * n
        rows.append(row)
        cols.append(col)
        d[n * row: n * row + n] = big_cost
        d[col::n] = big_cost
    return total_cost, rows, cols


def lcm_greedy_opt(n, c, threshold=10, big_cost=BIG_COST):
    """greedy_opt.py:61-82 (THRESHOLD 10) / simulate.py:76-97 (THRESHOLD 20).

    Returns (total, allocated_supply, allocated_demand); simulate.py's 4th value is zip of the two.
    """
    d = np.array(c, dtype=np.float64).flatten()
    total_cost = 0.0
    sup, dem = [], []
    for _ in range(n):
        elem = int(d.argmin(0))
        if d[elem] > threshold:                # greedy_opt.py:69
            break
        row = int(elem / n)
        col = elem - row * n
        sup.append(row)
        dem.append(col)
        if d[elem] < big_cost:
            total_cost += d[elem]
        d[n * row: n * row + n] = big_cost
        d[col::n] = big_cost
    return total_cost, sup, dem


def lcm_java(cost, big_cost=BIG_COST, max_non_lcm=600):
    """Simulator.java:523-549.  Returns (pairs, LCM_min_val)."""
    c = np.array(cost, dtype=np.int64)
    n = c.shape[0]
    pairs = []
    size = n
    lcm_min_val = big_cost
    for _ in range(n):
        lcm_min_val = big_cost
        flat = c.reshape(-1)
        e = int(flat.argmin()) if n else 0
        if n == 0 or flat[e] >= big_cost:      # strict '<' scan from big_cost (:531-538)
            break
        lcm_min_val = int(flat[e])
        s_min, d_min = divmod(e, n)
        pairs.append((s_min, d_min))
        c[:, d_min] = big_cost
        c[s_min, :] = big_cost
        size -= 1
        if size == max_non_lcm:                # :545
            break
    return pairs, lcm_min_val


class _Params(ctypes.Structure):
    _fields_ = [("mask_value", ctypes.c_int32), ("stop_above", ctypes.c_int32), ("stop_at_value", ctypes.c_int32),
                ("sum_below", ctypes.c_int32), ("residual_size", ctypes.c_int32), ("max_iters", ctypes.c_int32)]


def lcm_c(cost, mask_value, stop_above=INT32_MAX, stop_at_value=INT32_MAX, sum_below=INT32_MAX,
          residual_size=0, max_iters=-1):
    """C twin (oracle/lcm_oracle.c) of the literal array algorithm; returns dict."""
    c = np.ascontiguousarray(np.asarray(cost, dtype=np.int32))
    n = int(round(c.size ** 0.5)) if c.ndim == 1 else c.shape[0]
    assert c.size == n * n
    rows = np.zeros(max(n, 1), dtype=np.int32)
    cols = np.zeros(max(n, 1), dtype=np.int32)
    npairs = ctypes.c_int32(0)
    total = ctypes.c_int64(0)
    last = ctypes.c_int32(0)
    p = _Params(mask_value, stop_above, stop_at_value, sum_below, residual_size, max_iters)
    rc = _clib.lib().lcm_oracle(c.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(n), ctypes.byref(p),
                                rows.ctypes.data_as(ctypes.c_void_p), cols.ctypes.data_as(ctypes.c_void_p),
                                ctypes.byref(npairs), ctypes.byref(total), ctypes.byref(last))
    if rc != 0:
        raise RuntimeError("lcm_oracle rc=%d" % rc)
    k = npairs.value
    return {"total": total.value, "rows": rows[:k].copy(), "cols": cols[:k].copy(), "n_pairs": k,
            "last_min": last.value}


def lcm_sort_keys(cost) -> np.ndarray:
    """Every cell's 64-bit key ((uint32(cost) ^ 0x80000000) << 32 | flat index), sorted: the first-index argmin order
    of the whole matrix.  One sort serves every parameter set of lcm_walk.  n <= 65535 (the index fits 32 bits)."""
    c = np.asarray(cost, dtype=np.int32)
    n = int(round(c.size ** 0.5)) if c.ndim == 1 else c.shape[0]
    assert c.size == n * n and n <= 65535
    flat = c.reshape(-1)
    keys = np.empty(n * n, dtype=np.uint64)
    step = 1 << 24                                    # bounded temporaries at n = 20000 (400 M cells)
    for lo in range(0, n * n, step):
        hi = min(lo + step, n * n)
        k = (flat[lo:hi].view(np.uint32) ^ np.uint32(0x80000000)).astype(np.uint64) << np.uint64(32)
        k |= np.arange(lo, hi, dtype=np.uint64)
        keys[lo:hi] = k
    keys.sort()
    return keys


def lcm_walk(keys, n, mask_value, stop_above=INT32_MAX, stop_at_value=INT32_MAX, sum_below=INT32_MAX,
             residual_size=0, max_iters=-1):
    """The literal algorithm walked over lcm_sort_keys(cost) (oracle/lcm_oracle.c: lcm_sorted_walk); the dict of
    lcm_c, equal to it for every input."""
    keys = np.ascontiguousarray(keys, dtype=np.uint64)
    assert keys.size == n * n
    rows = np.zeros(max(n, 1), dtype=np.int32)
    cols = np.zeros(max(n, 1), dtype=np.int32)
    npairs = ctypes.c_int32(0)
    total = ctypes.c_int64(0)
    last = ctypes.c_int32(0)
    p = _Params(mask_value, stop_above, stop_at_value, sum_below, residual_size, max_iters)
    rc = _clib.lib().lcm_sorted_walk(keys.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(n), ctypes.byref(p),
                                     rows.ctypes.data_as(ctypes.c_void_p), cols.ctypes.data_as(ctypes.c_void_p),
                                     ctypes.byref(npairs), ctypes.byref(total), ctypes.byref(last))
    if rc != 0:
        raise RuntimeError("lcm_sorted_walk rc=%d" % rc)
    k = npairs.value
    return {"total": total.value, "rows": rows[:k].copy(), "cols": cols[:k].copy(), "n_pairs": k,
            "last_min": last.value}


def lcm_sorted(cost, mask_value, **kw):
    """lcm_c's result through the sorted walk: one sort and one walk."""
    c = np.asarray(cost, dtype=np.int32)
    n = int(round(c.size ** 0.5)) if c.ndim == 1 else c.shape[0]
    return lcm_walk(lcm_sort_keys(c), n, mask_value, **kw)
