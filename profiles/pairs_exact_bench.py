"""Exact 2-passenger pool (td_pool_pairs_exact_batch) on the GPU against the C oracle and networkx on one host core.

  batch    1000 instances x 100 customers over 50 stands (dist |i - j|), accept_all 1 and 0, one launch per call
  single   one instance at n = 142, 722 and 1445 (the Simulator's first, a middle and its largest pool step size)
  gap      pool_greedy_vs_optimum on the 1000-case batch: (greedy total / optimal total - 1), pool_opt_min.py's figure

Times are CUDA events around the launch (inputs already on the device), median of repeated runs.  The batch's working
set (inputs, 27 MB of workspace, outputs) fits the 126 MB L2 and is L2-resident after the warm-up.  Prints one JSON line,
with the card's name and power limit read in the same run, and also writes it to the file --out names
(profiles/pairs_exact_b200.json holds the committed line)."""
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in q.split(",")]
        return name, power
    except Exception as e:  # noqa: BLE001
        import torch
        return torch.cuda.get_device_name(0), "unknown (%s)" % type(e).__name__


def timed(fn, reps):
    import torch
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--networkx-max-n", type=int, default=142)
    args = ap.parse_args()
    import torch
    from oracle import pairs_ref
    from taxidispatcher_b200 import dispatch, experiments
    D = np.abs(np.subtract.outer(np.arange(50), np.arange(50))).astype(np.int32)
    rng = np.random.default_rng(2025)
    eng = dispatch.engine()
    res = {"card": None, "power_limit": None, "l2": "batch working set L2-resident (warmed, < 126 MB)"}
    res["card"], res["power_limit"] = card()

    inst = [(rng.integers(0, 50, 100).astype(np.int32), rng.integers(0, 50, 100).astype(np.int32)) for _ in range(1000)]
    for acc in (1, 0):
        frm, to, sizes, offs, n_max, d = dispatch.pack_pairs_batch(inst, D)
        run = lambda: eng.pool_pairs_exact_batch(frm, to, sizes, offs, n_max, d, bool(acc), 1.01)  # noqa: E731
        run()
        torch.cuda.synchronize()
        res["batch1000x100_acc%d_ms" % acc] = round(timed(run, args.reps), 3)
        t0 = time.perf_counter()
        for f, t in inst[:50]:
            pairs_ref.pairs_exact(f, t, D, bool(acc), 1.01)
        res["batch1000x100_acc%d_oracle_1core_ms_est" % acc] = round((time.perf_counter() - t0) * 1000 * 20, 1)
        # outputs against the oracle on the whole batch
        got = dispatch.find_pool_pairs_exact_batch(inst, D, bool(acc), 1.01)
        ok = all((len(g), int(g[:, 3].sum())) == pairs_ref.pairs_exact(f, t, D, bool(acc), 1.01)[1:] for (f, t), g in zip(inst, got))
        res["batch1000x100_acc%d_equal_oracle" % acc] = ok

    for n in (142, 722, 1445):
        f, t = rng.integers(0, 50, n).astype(np.int32), rng.integers(0, 50, n).astype(np.int32)
        frm, to, sizes, offs, n_max, d = dispatch.pack_pairs_batch([(f, t)], D)
        run = lambda: eng.pool_pairs_exact_batch(frm, to, sizes, offs, n_max, d, True, 1.01)  # noqa: E731
        rows, npairs, cost = run()
        torch.cuda.synchronize()
        res["single_n%d_ms" % n] = round(timed(run, max(3, args.reps // 2)), 3)
        t0 = time.perf_counter()
        _, m, total = pairs_ref.pairs_exact(f, t, D, True)
        res["single_n%d_oracle_1core_ms" % n] = round((time.perf_counter() - t0) * 1000, 1)
        res["single_n%d_equal_oracle" % n] = (int(npairs[0]), int(cost[0])) == (m, total)
        if n <= args.networkx_max_n:
            import networkx as nx
            G = nx.Graph()
            for i in range(n):
                for j in range(i + 1, n):
                    c = min(int(D[f[i], f[j]] + D[f[j], t[i]] + D[t[i], t[j]]), int(D[f[i], f[j]] + D[f[j], t[j]] + D[t[j], t[i]]),
                            int(D[f[j], f[i]] + D[f[i], t[j]] + D[t[j], t[i]]), int(D[f[j], f[i]] + D[f[i], t[i]] + D[t[i], t[j]]))
                    G.add_edge(i, j, neg=-c)
            t0 = time.perf_counter()
            nx.max_weight_matching(G, maxcardinality=True, weight="neg")
            res["single_n%d_networkx_1core_ms" % n] = round((time.perf_counter() - t0) * 1000, 1)
        else:
            res["single_n%d_networkx_1core_ms" % n] = "not run (minutes on one core)"

    r = experiments.pool_greedy_vs_optimum(inst, D, True, 1.01)
    g, o = sum(x[1] for x in r), sum(x[3] for x in r)
    gaps = [x[1] / x[3] - 1 for x in r if x[3] > 0]
    res["gap_1000x100_acc1"] = {"total": round(g / o - 1, 4), "mean": round(float(np.mean(gaps)), 4),
                                "max": round(float(np.max(gaps)), 4), "counts_equal": all(x[0] == x[2] for x in r)}
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
