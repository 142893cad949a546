"""Pool finder oracles.  TEST INFRASTRUCTURE ONLY.

  find / merge        ctypes front end of oracle/pool_oracle.c (our C restatement of
                      pool_n.c:101-207,226-229 and findpool.c:83-108)
  run_reference       runs the compiled reference binary oracle/_ref/pool_n_big (built from
                      $TD_REFERENCE_DIR/pool_n.c by oracle/Makefile) on a temp CSV and parses its
                      CSV output and the three counters it prints
"""
from __future__ import annotations

import ctypes
import os
import re
import subprocess
import tempfile

import numpy as np

from . import _clib
from .gen_inputs import demand_csv

REC_W = 9


class Stats(ctypes.Structure):
    _fields_ = [("evaluated", ctypes.c_int64), ("feasible", ctypes.c_int64), ("kept", ctypes.c_int64)]


def find(demand, dist, pool_size, shard=0, n_shards=8, dedup=True, cap=None):
    dem = np.ascontiguousarray(np.asarray(demand, dtype=np.int32).reshape(-1, 5))
    d = np.ascontiguousarray(np.asarray(dist, dtype=np.int32))
    n = dem.shape[0]
    if cap is None:
        cap = max(n, 16) if dedup else 1 << 22
    while True:
        out = np.zeros((cap, REC_W), dtype=np.int32)
        cnt = ctypes.c_int64(0)
        st = Stats()
        rc = _clib.lib().pool_oracle_find(dem.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(n),
                                          d.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(d.shape[0]),
                                          ctypes.c_int(pool_size), ctypes.c_int(shard), ctypes.c_int(n_shards),
                                          ctypes.c_int(1 if dedup else 0), out.ctypes.data_as(ctypes.c_void_p),
                                          ctypes.c_int64(cap), ctypes.byref(cnt), ctypes.byref(st))
        if rc == -3:
            cap = int(cnt.value)
            continue
        if rc != 0:
            raise RuntimeError("pool_oracle_find rc=%d" % rc)
        return out[: cnt.value].copy(), {"evaluated": st.evaluated, "feasible": st.feasible, "kept": st.kept}


def merge(shard_plans, n_cust, pool_size):
    """shard_plans: list of [m_i, 9] arrays in shard order."""
    parts = [np.asarray(p, dtype=np.int32).reshape(-1, REC_W) for p in shard_plans]
    allp = np.ascontiguousarray(np.concatenate(parts, axis=0)) if parts else np.zeros((0, REC_W), np.int32)
    out = np.zeros((max(len(allp), 1), REC_W), dtype=np.int32)
    cnt = ctypes.c_int64(0)
    rc = _clib.lib().pool_oracle_merge(allp.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(len(allp)),
                                       ctypes.c_int(n_cust), ctypes.c_int(pool_size),
                                       out.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(len(out)),
                                       ctypes.byref(cnt))
    if rc != 0:
        raise RuntimeError("pool_oracle_merge rc=%d" % rc)
    return out[: cnt.value].copy()


def reference_binary():
    return _clib.build_ref()


def run_reference(demand, pool_size, shard, workdir=None):
    """Run the compiled reference on one shard.  Returns (plans [m,9] int32 in pool_n layout, stats)."""
    dem = np.asarray(demand, dtype=np.int32).reshape(-1, 5)
    return run_reference_csv(demand_csv(dem), len(dem), pool_size, shard, workdir)


def run_reference_csv(text, rec_number, pool_size, shard, workdir=None):
    """`pool_n pool_size shard demand.csv rec_number out.csv` on a demand file of the given text."""
    exe = reference_binary()
    if exe is None or not os.path.exists(exe):
        raise FileNotFoundError("oracle/_ref/pool_n_big is not built (make -C oracle ref)")
    with tempfile.TemporaryDirectory(dir=workdir) as td:
        with open(os.path.join(td, "demand.csv"), "w") as f:
            f.write(text)
        res = subprocess.run([exe, str(pool_size), str(shard), "demand.csv", str(rec_number), "out.csv"],
                             cwd=td, capture_output=True, text=True, check=True)
        plans = parse_result_csv(open(os.path.join(td, "out.csv")).read(), pool_size)
    # count_all is a 32-bit `int` in the reference (pool_n.c:28) and wraps beyond 2^31 leaf plans per shard
    m = {k: int(v) for k, v in re.findall(r"(Count ALL|Count|Not duplicated count): (-?\d+)", res.stdout)}
    stats = {"evaluated": m.get("Count ALL"), "feasible": m.get("Count"), "kept": m.get("Not duplicated count")}
    return plans, stats


def parse_result_csv(text, pool_size):
    """pool_n.c:72-78 lines 'p0,..,d0,..,cost,' -> rows in the in-memory layout (cost at column 8)."""
    rows = []
    for line in text.splitlines():
        f = [int(v) for v in line.strip().strip(",").split(",") if v != ""]
        if not f:
            continue
        r = [0] * REC_W
        r[: 2 * pool_size] = f[: 2 * pool_size]
        r[8] = f[2 * pool_size]
        rows.append(r)
    return np.asarray(rows, dtype=np.int32).reshape(-1, REC_W)


def format_result_csv(plans, pool_size):
    out = []
    for r in np.asarray(plans).reshape(-1, REC_W):
        out.append("".join("%d," % int(v) for v in r[: 2 * pool_size]) + "%d,\n" % int(r[8]))
    return "".join(out)


def pairs(frm, to, dist, accept_all=True, max_loss=1.01):
    """Simulator.findPool restated (oracle/pool_oracle.c: pool_pairs_oracle)."""
    f = np.ascontiguousarray(np.asarray(frm, dtype=np.int32))
    t = np.ascontiguousarray(np.asarray(to, dtype=np.int32))
    d = np.ascontiguousarray(np.asarray(dist, dtype=np.int32))
    n = len(f)
    out = np.zeros((n // 2 + 1, 4), dtype=np.int32)
    cnt = ctypes.c_int64(0)
    rc = _clib.lib().pool_pairs_oracle(f.ctypes.data_as(ctypes.c_void_p), t.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(n),
                                       d.ctypes.data_as(ctypes.c_void_p), ctypes.c_int(d.shape[0]),
                                       ctypes.c_int(1 if accept_all else 0), ctypes.c_double(max_loss),
                                       out.ctypes.data_as(ctypes.c_void_p), ctypes.c_int64(len(out)), ctypes.byref(cnt))
    if rc != 0:
        raise RuntimeError("pool_pairs_oracle rc=%d" % rc)
    return out[: cnt.value].copy()
