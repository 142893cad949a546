"""Exact 2-passenger pool oracle.  TEST INFRASTRUCTURE ONLY.

  pairs_exact       ctypes front end of oracle/pairs_oracle.c: minimum-cost maximum-cardinality pair matching
                    over the candidates Simulator.findPool accepts (the optimum pool_optimum.py /
                    pool_opt_min.py ask for), built into its own oracle/_build/libpairs_oracle.so
  OracleBackend     oracle.sim_backend.OracleBackend whose 2-passenger pool is, with exact_pool=True, the exact
                    matching instead of the greedy scan
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import time

import numpy as np

from . import pool_ref, sim_backend

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "_build", "libpairs_oracle.so")
_SRC = os.path.join(_HERE, "pairs_oracle.c")
_lib = None


def build(force: bool = False) -> str:
    if force or not os.path.exists(_SO) or os.path.getmtime(_SRC) > os.path.getmtime(_SO):
        os.makedirs(os.path.dirname(_SO), exist_ok=True)
        cc = os.environ.get("CC", "gcc")
        subprocess.check_call([cc, "-O3", "-Wall", "-fPIC", "-shared", "-o", _SO, _SRC])
    return _SO


def lib() -> ctypes.CDLL:
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(build())
    return _lib


def pairs_exact(frm, to, dist, accept_all=True, max_loss=1.01):
    """(rows [m, 4] int32 = custA, custB, plan, cost in (cost, A*n+B) order, m, total) of a minimum-cost
    maximum-cardinality matching; None when a live row names a stand outside the table (withdrawn)."""
    f = np.ascontiguousarray(np.asarray(frm, dtype=np.int32))
    t = np.ascontiguousarray(np.asarray(to, dtype=np.int32))
    d = np.ascontiguousarray(np.asarray(dist, dtype=np.int32))
    n = len(f)
    out = np.zeros((n // 2 + 1, 4), dtype=np.int32)
    cnt = ctypes.c_int32(0)
    total = ctypes.c_int64(0)
    rc = lib().pairs_exact_oracle(f.ctypes.data_as(ctypes.c_void_p), t.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(n),
                                  d.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(d.shape[0] if d.ndim == 2 else 0),
                                  ctypes.c_int(1 if accept_all else 0), ctypes.c_double(max_loss),
                                  out.ctypes.data_as(ctypes.c_void_p), ctypes.byref(cnt), ctypes.byref(total))
    if rc == -2:
        return None
    if rc != 0:
        raise RuntimeError("pairs_exact_oracle rc=%d" % rc)
    m = int(cnt.value)
    return out[:m].copy(), m, int(total.value)


class OracleBackend(sim_backend.OracleBackend):
    """The Simulator's CPU backend; exact_pool=True pools customers by the exact matching."""

    def __init__(self, exact_pool: bool = False):
        super().__init__()
        self.exact_pool = exact_pool

    def pool_pairs(self, frm, to, dist):
        if not self.exact_pool:
            return super().pool_pairs(frm, to, dist)
        t0 = time.perf_counter()
        r = pairs_exact(frm, to, dist, accept_all=True)[0]
        self.times["pool"] += time.perf_counter() - t0
        return r


def greedy(frm, to, dist, accept_all=True, max_loss=1.01):
    """The greedy scan (pool_ref.pairs) as (rows, count, total)."""
    r = pool_ref.pairs(frm, to, dist, accept_all=accept_all, max_loss=max_loss)
    return r, len(r), int(r[:, 3].astype(np.int64).sum()) if len(r) else 0
