"""Deterministic synthetic inputs for every BASELINE.json config (SURVEY.md section 8(d)).

TEST INFRASTRUCTURE (part of oracle/): importable from tests/, bench.py and
__graft_entry__.smoke() only.  Nothing here reads the reference's sources.

All generators use numpy.random.default_rng(seed) (PCG64); costs are int32.
"""
from __future__ import annotations

import hashlib

import numpy as np

BIG_COST = 250000  # split.py:5, greedy_opt.py:5, simulate.py:13, Simulator.java:114


def stand_distances(n_stands: int) -> np.ndarray:
    """dist[i][j] = |i-j| -- split.py:179-184, pool_n.c:179-185, Simulator.java:553-560."""
    idx = np.arange(n_stands, dtype=np.int32)
    return np.abs(idx[:, None] - idx[None, :]).astype(np.int32)


# ---- config 1: 200 x 200 assignment ------------------------------------------------------------
def config1a(n: int = 200, seed: int = 20201007) -> np.ndarray:
    """heuristic.py:21 distribution: randint(1,40)."""
    return np.random.default_rng(seed).integers(1, 40, (n, n)).astype(np.int32)


def config1b(n_cabs: int = 190, n_cust: int = 200, n_stands: int = 50, seed: int = 50):
    """Stand-derived, python.py-style dummy padding (10 dummy rows of big_cost)."""
    rng = np.random.default_rng(seed)
    cab_to = rng.integers(0, n_stands, 200).astype(np.int32)[:n_cabs]
    cust_from = rng.integers(0, n_stands, 200).astype(np.int32)[:n_cust]
    return stand_distances(n_stands), cab_to, cust_from


# ---- config 2: 2000 x 2000 LCM vs optimum ------------------------------------------------------
def config2(n: int = 2000, seed: int = 2000) -> np.ndarray:
    return np.random.default_rng(seed).integers(1, 40, (n, n)).astype(np.int32)


def config2_stand(n: int = 2000, n_stands: int = 4000, seed: int = 2001):
    """greedy_opt.py:7 uses 4000 stands; mask = big_cost variant."""
    rng = np.random.default_rng(seed)
    cab_to = rng.integers(0, n_stands, n).astype(np.int32)
    cust_from = rng.integers(0, n_stands, n).astype(np.int32)
    return np.abs(cab_to[:, None] - cust_from[None, :]).astype(np.int32)


# ---- config 3: pool_n, 4 passengers, 722 customers ---------------------------------------------
def pool_demand(n: int = 722, n_stands: int = 50, seed: int = 1, wait: int = 3, loss: int = 1) -> np.ndarray:
    """SURVEY.md appendix A.2: one scalar integers() call per draw, in exactly this order.

    Returns int32 [n,5] rows (id, from, to, maxWait, maxLoss) -- pool_n.c:20.
    wait 3 = Pool.java:20, loss 1 % = Pool.java:21.
    """
    rng = np.random.default_rng(seed)
    rows = np.empty((n, 5), dtype=np.int32)
    for i in range(n):
        fr = int(rng.integers(0, n_stands))
        while True:
            to = int(rng.integers(0, n_stands))
            if to != fr:
                break
        rows[i] = (i, fr, to, wait, loss)
    return rows


def demand_csv(rows: np.ndarray) -> str:
    """The pool_n demand file format (pool_n.c:42-52): 'id,from,to,maxWait,maxLoss' per line."""
    return "".join("%d,%d,%d,%d,%d\n" % tuple(int(v) for v in r) for r in rows)


def demand_md5(rows: np.ndarray) -> str:
    return hashlib.md5(demand_csv(rows).encode()).hexdigest()


POOL722_MD5 = "6bfbc99dc994e1e15f988363e197ccc6"
# Known answers of the compiled reference (SURVEY.md section 8(d) config 3, KAT P2)
POOL722_EVALUATED = [382592136, 383212296, 384193104, 391107600, 367492056, 378532392, 381004824, 374816856]
POOL722_FEASIBLE = [2268957, 2201027, 1922139, 1909089, 2339340, 1986344, 1958445, 2069043]
POOL722_KEPT = [86, 87, 85, 82, 89, 86, 85, 78]


def pool_crosscheck_cases():
    """Inputs of the pool cross-check against the compiled pool_n.c: [(pool size, demand, shard)], 9 cases x 2 shards --
    ragged waits and losses, from == to trips, every pool size, over MAX_STAND = 51 stands (pool_n.c:179-185)."""
    rng = np.random.default_rng(424242)
    out = []
    for case in range(9):
        k = 2 + case % 3
        n = int(rng.integers(12, 64 if k == 4 else 120))
        fr = rng.integers(0, 51, n)
        to = np.where(rng.random(n) < 0.15, fr, rng.integers(0, 51, n))
        dem = np.stack([np.arange(n), fr, to, rng.integers(0, 9, n), rng.integers(0, 60, n)], axis=1).astype(np.int32)
        for shard in (0, int(rng.integers(1, 8))):
            out.append((k, dem, shard))
    return out


# readDemand quirks (pool_n.c:30-54): a blank line, a short record and FEWER lines than rec-number
DEMAND_QUIRKS_REC_NUMBER = 40
DEMAND_QUIRKS_RUNS = ((2, 0), (3, 1), (4, 0))      # (pool size, shard)


def demand_quirks_csv() -> str:
    lines = demand_csv(pool_demand(40, seed=9)).splitlines()
    lines[7] = ""                       # blank line -> a record of zeros
    lines[11] = "11,3"                  # to / wait / loss stay 0
    return "\n".join(lines[:33]) + "\n"  # seven fewer records than DEMAND_QUIRKS_REC_NUMBER


# ---- config 5: 20k x 20k ----------------------------------------------------------------------
def config5a(n: int = 20000, seed: int = 20000) -> np.ndarray:
    return np.random.default_rng(seed).integers(1, 40, (n, n), dtype=np.int32)


def config5b(n: int = 20000, n_stands: int = 4000, seed: int = 20001):
    rng = np.random.default_rng(seed)
    cab_to = rng.integers(0, n_stands, n).astype(np.int32)
    cust_from = rng.integers(0, n_stands, n).astype(np.int32)
    return cab_to, cust_from


def config5b_cost(n: int = 20000, n_stands: int = 4000, seed: int = 20001) -> np.ndarray:
    cab_to, cust_from = config5b(n, n_stands, seed)
    return np.abs(cab_to[:, None] - cust_from[None, :]).astype(np.int32)


def rand_list(rng: np.random.Generator, numb: int, size: int):
    """split.py:41-52 / greedy_opt.py:40-52 with a seeded generator: drop rows with from == to."""
    out = []
    for _ in range(numb):
        frm = int(rng.integers(0, size))
        to = int(rng.integers(0, size))
        if frm != to:
            out.append((len(out), frm, to))
    return out
