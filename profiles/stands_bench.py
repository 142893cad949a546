"""Stand-derived assignment as S x S transportation problems (td_assign_stands_batch) against the dense exact routes:
prints ONE JSON line (kept in profiles/stands_b200.json), with the card name and power limit read in the same run.

Workloads:
  sim1000   1000 Simulator-shaped instances: 600 cabs against 218-368 customers over 50 stands, cutoff 10.
            solve_stands_batch end to end and the td_assign_stands_batch call alone (device-resident inputs), against
            the loop of solve_assignment and against pack_cost_matrices + run_packed.  Objectives asserted equal.
  sim1      one such instance: solve_assignment_stands against solve_assignment (end to end, host arrays in).
  n20000    20 000 x 20 000 over 50 and 128 stands: the stands call against K1 + td_assign_exact_rect (1.6 GB matrix).
  huge      10^6 and 10^7 per side over 128 stands: only this route runs them.  Bytes per element of the counting
            and expansion passes (index reads, col_of_row / cost_of_row and slot writes) over the call time, against
            the 7.7 TB/s of HBM3e, and the oracle's time on one host core (bincount + the S x S solve) beside it.

Times are medians of --reps CUDA-event windows after a warm-up (end-to-end host functions: host clock around a call
that ends in a read-back).

    python profiles/stands_bench.py [--reps 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BIG_COST = 250000
HBM_TBS = 7.7


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    parts = [p.strip() for p in line.split(",")] if line else ["unknown", "unknown", "unknown"]
    return {"name": parts[0], "power_limit": parts[1], "max_sm_clock": parts[2]}


def events_ms(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return float(np.median(times))


def host_ms(fn, reps):
    fn()
    times = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        times.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(times))


def stands_call(d, pk, n_max, cutoff, want_cost=False):
    return lambda: d.engine().assign_stands_batch(pk["dist"], pk["cab_to"], pk["cab_off"], pk["n_c"], pk["cust_from"],
                                                  pk["cust_off"], pk["n_d"], n_max, BIG_COST, cutoff, want_cost=want_cost)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from taxidispatcher_b200 import dispatch as d
    from oracle import transport_ref as T
    out = {"card": card(), "workloads": {}}
    rng = np.random.default_rng(2026)
    W = out["workloads"]

    # 1. 1000 Simulator-shaped instances
    S = 50
    dist = np.abs(np.subtract.outer(np.arange(S), np.arange(S))).astype(np.int32)
    insts = [(rng.integers(0, S, 600).astype(np.int32), rng.integers(0, S, int(rng.integers(218, 369))).astype(np.int32))
             for _ in range(1000)]
    dist_d = d._h2d_i32(dist)
    st_res = d.solve_stands_batch(dist, insts, cutoff=10)
    packed, sizes, offsets, n_max, ns = d.pack_cost_matrices(dist_d, insts, BIG_COST, 10)
    dense_res, _ = d.run_packed(packed, sizes, offsets, n_max, ns)
    loop_obj = [int(c.astype(np.int64).sum()) for _, _, c in (d.solve_assignment(dist_d, a, b, BIG_COST, 10)
                                                              for a, b in insts[:50])]
    assert [o for _, o in st_res] == [o for _, o in dense_res], "stands and packed dense objectives differ"
    assert loop_obj == [o for _, o in st_res[:50]], "stands and solve_assignment objectives differ"
    pk = d.pack_stands_batch(insts, dist)
    loop50 = host_ms(lambda: [d.solve_assignment(dist_d, a, b, BIG_COST, 10) for a, b in insts[:50]], max(1, args.reps // 2))
    W["sim1000"] = {
        "instances": 1000, "stands": S, "cabs": 600, "customers": "218-368", "cutoff": 10,
        "stands_e2e_ms": host_ms(lambda: d.solve_stands_batch(dist, insts, cutoff=10), args.reps),
        "stands_call_ms": events_ms(stands_call(d, pk, pk["n_max"], 10), args.reps),
        "dense_packed_e2e_ms": host_ms(lambda: d.run_packed(*d.pack_cost_matrices(dist_d, insts, BIG_COST, 10)), args.reps),
        "dense_solve_assignment_loop_ms": loop50 * 20, "dense_loop_measured_on": "first 50 instances, scaled x20",
        "objectives_equal": True}

    # 2. one Simulator-shaped instance
    a, b = insts[0]
    W["sim1"] = {"cabs": 600, "customers": len(b),
                 "solve_assignment_stands_ms": host_ms(lambda: d.solve_assignment_stands(dist_d, a, b, BIG_COST, 10), 20),
                 "solve_assignment_ms": host_ms(lambda: d.solve_assignment(dist_d, a, b, BIG_COST, 10), 20)}

    # 3. 20 000 x 20 000
    eng = d.engine()
    for S in (50, 128):
        dist = rng.integers(0, 60, (S, S)).astype(np.int32)
        a, b = rng.integers(0, S, 20000).astype(np.int32), rng.integers(0, S, 20000).astype(np.int32)
        pk = d.pack_stands_batch([(a, b)], dist)
        _, _, obj, _, _, _ = stands_call(d, pk, 20000, None)()
        dd, ad, bd = d._h2d_i32(dist), d._h2d_i32(a), d._h2d_i32(b)

        def dense():
            return eng.assign(eng.cost_matrix(dd, ad, bd, BIG_COST, None))[1]
        dobj = int(dense().item())
        assert dobj == int(obj.item()), "20000: stands and dense objectives differ"
        W["n20000_S%d" % S] = {"stands_call_ms": events_ms(stands_call(d, pk, 20000, None), args.reps),
                               "dense_k1_plus_exact_ms": events_ms(dense, max(1, args.reps // 2)),
                               "objectives_equal": True}

    # 4. 10^6 and 10^7 per side over 128 stands
    S = 128
    dist = rng.integers(0, 60, (S, S)).astype(np.int32)
    for n in (10**6, 10**7):
        a, b = rng.integers(0, S, n).astype(np.int32), rng.integers(0, S, n - n // 7).astype(np.int32)
        pk = d.pack_stands_batch([(a, b)], dist)
        t0 = time.perf_counter()
        ref = T.solve(dist, a, b, BIG_COST, 30)
        oracle_ms = (time.perf_counter() - t0) * 1e3
        _, _, obj, _, _, _ = stands_call(d, pk, n, 30, True)()
        assert int(obj.item()) == ref["objective"], "huge: stands objective differs from the oracle"
        ms = events_ms(stands_call(d, pk, n, 30, True), args.reps)
        nd = len(b)
        # count: read both index arrays; customer expansion: read customers twice (histogram + ranks), write slot
        # (or padding row + cost); cab expansion: read cabs twice, read slot, read cust_from[j], write col + cost
        bytes_moved = 4 * (n + nd) + 4 * (2 * nd + nd) + 4 * (2 * n + n + n + 2 * n)
        W["huge_%d" % n] = {"stands": S, "cabs": n, "customers": nd, "cutoff": 30, "call_ms": ms,
                            "bytes": bytes_moved, "bytes_per_element": bytes_moved / (n + nd),
                            "achieved_TBps": bytes_moved / (ms * 1e-3) / 1e12, "hbm_TBps": HBM_TBS,
                            "oracle_one_core_ms": oracle_ms, "objective_equal_oracle": True}
        del pk
        torch.cuda.empty_cache()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
