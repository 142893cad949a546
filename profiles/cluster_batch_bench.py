"""Batches of mid-size instances on thread-block clusters against per-instance calls and one host core: prints ONE JSON
line (kept in profiles/cluster_batch_b200.json).

Workloads (B instances of n x n):
  uniform_400     1000 x 400^2, U[1,39] costs
  stand_400       1000 x 400^2, 400 cabs x 400 customers over 4000 stands (the paper's split / hybrid experiment)
  sim_600         200 x 600^2, 560 cabs x 600 customers over 4000 stands, big_cost padding rows (Simulator.java's
                  MAX_NON_LCM = 600 solver shape)
  sim_600_b1..b8  1, 2, 3, 4 and 8 instances of the sim_600 shape, and 2 to 4 instances of 240 x 240 (the smallest
                  cluster size): where the loop of single-instance calls may win (run_batch's LCM crossover)

For each: td_assign_exact_batch_cluster / td_lcm_batch_cluster (CUDA events, median of --reps launches after a warm-up),
the loop of single-instance calls (Engine.assign / Engine.lcm) over the same device-resident matrices (CUDA events around
the whole loop, median of --loop-reps loops), and one host core running scipy's linear_sum_assignment and the C
restatement of the literal LCM (oracle/lcm_oracle.c) over the same instances.  Batch and loop are asserted to return the
same objectives and the same LCM traces in the same run.  Then split_hybrid_vs_optimum end to end on 1000 paper cases
(host clock, median of 3 runs after one warm-up run).

The 1000 x 400^2 working sets are 640 MB and the 200 x 600^2 one 288 MB: larger than the 126 MB L2, so those batches
read their matrices from HBM.  The 1- to 8-instance workloads (at most 11.5 MB) are L2-resident.

    python profiles/cluster_batch_bench.py [--reps 10] [--loop-reps 2] [--out FILE]
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
LCM_SPLIT = dict(mask_value=BIG_COST, sum_below=BIG_COST)
WORKLOADS = [("uniform_400", 1000, 400, None, dict(mask_value=100)),
             ("stand_400", 1000, 400, 400, LCM_SPLIT),
             ("sim_600", 200, 600, 560, LCM_SPLIT),
             ("sim_600_b1", 1, 600, 560, LCM_SPLIT),
             ("sim_600_b2", 2, 600, 560, LCM_SPLIT),
             ("sim_600_b3", 3, 600, 560, LCM_SPLIT),
             ("sim_600_b4", 4, 600, 560, LCM_SPLIT),
             ("sim_600_b8", 8, 600, 560, LCM_SPLIT),
             ("stand_240_b2", 2, 240, 240, LCM_SPLIT),
             ("stand_240_b3", 3, 240, 240, LCM_SPLIT),
             ("stand_240_b4", 4, 240, 240, LCM_SPLIT)]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    line = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else ""
    parts = [p.strip() for p in line.split(",")] if line else ["unknown", "unknown", "unknown"]
    return {"name": parts[0], "power_limit": parts[1], "max_sm_clock": parts[2]}


def events_ms(fn, reps):
    import torch
    times = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        times.append(a.elapsed_time(b))
    return {"median": float(np.median(times)), "min": float(np.min(times)), "max": float(np.max(times)), "reps": reps}


def build_cases(B, n, n_cabs, seed):
    from oracle import cost_ref, gen_inputs as g
    rng = np.random.default_rng(seed)
    if n_cabs is None:
        return [rng.integers(1, 40, (n, n)).astype(np.int32) for _ in range(B)]
    dist = g.stand_distances(4000)
    return [cost_ref.calculate_cost_np(dist, rng.integers(0, 4000, n_cabs), rng.integers(0, 4000, n))[1] for _ in range(B)]


def run_workload(name, B, n, n_cabs, lcm_kw, reps, loop_reps, seed):
    import torch
    from scipy.optimize import linear_sum_assignment
    from oracle import lcm_ref
    from taxidispatcher_b200 import dispatch

    eng = dispatch.engine()
    cases = build_cases(B, n, n_cabs, seed)
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    mats = [packed[int(o): int(o) + n * n].view(n, n) for o in offs.cpu().numpy()]
    a_out = {"col": torch.empty((B, n_max), dtype=torch.int32, device="cuda"),
             "objective": torch.empty(B, dtype=torch.int64, device="cuda")}
    l_out = {"rows": torch.empty((B, n_max), dtype=torch.int32, device="cuda"),
             "cols": torch.empty((B, n_max), dtype=torch.int32, device="cuda"),
             "n_pairs": torch.empty(B, dtype=torch.int32, device="cuda"),
             "total": torch.empty(B, dtype=torch.int64, device="cuda"),
             "last_min": torch.empty(B, dtype=torch.int32, device="cuda")}
    do_assign = lambda: eng.assign_batch(packed, sizes, offs, n_max, out=a_out)          # noqa: E731
    do_lcm = lambda: eng.lcm_batch(packed, sizes, offs, n_max, out=l_out, **lcm_kw)      # noqa: E731
    for _ in range(2):
        do_assign()
        do_lcm()
    torch.cuda.synchronize()
    t_assign = events_ms(do_assign, reps)
    t_lcm = events_ms(do_lcm, reps)

    loop_out = {}

    def loop_assign():
        loop_out["assign"] = [eng.assign(m)[:2] for m in mats]

    def loop_lcm():
        loop_out["lcm"] = [eng.lcm(m, **lcm_kw) for m in mats]

    loop_assign()
    loop_lcm()
    torch.cuda.synchronize()
    t_loop_assign = events_ms(loop_assign, loop_reps)
    t_loop_lcm = events_ms(loop_lcm, loop_reps)

    # the same objectives and LCM traces, batch vs loop (same run); the tie choice of the matching may differ
    obj_b = a_out["objective"].cpu().numpy()
    col_b = a_out["col"].cpu().numpy()
    obj_l = torch.cat([o for _, o in loop_out["assign"]]).cpu().numpy()
    assert np.array_equal(obj_b, obj_l), "assign: batch objective != loop objective"
    assert all(sorted(col_b[k, :n].tolist()) == list(range(n)) for k in range(B))
    rows_b, cols_b = l_out["rows"].cpu().numpy(), l_out["cols"].cpu().numpy()
    np_b, tot_b, last_b = (l_out[k].cpu().numpy() for k in ("n_pairs", "total", "last_min"))
    for k, (r, c, s) in enumerate(loop_out["lcm"]):
        h = dispatch.Engine.lcm_host_view(r, c, s)
        m = h["n_pairs"]
        assert (np_b[k], tot_b[k], last_b[k]) == (m, h["total"], h["last_min"]), ("lcm: batch != loop", k)
        assert np.array_equal(rows_b[k, :m], h["rows"]) and np.array_equal(cols_b[k, :m], h["cols"]), ("lcm rows", k)

    # one host core
    t0 = time.perf_counter()
    cpu_obj = []
    for c in cases:
        r, cc = linear_sum_assignment(c)
        cpu_obj.append(int(c.astype(np.int64)[r, cc].sum()))
    t_cpu_lsa = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    cpu_lcm = [lcm_ref.lcm_c(c, lcm_kw["mask_value"], sum_below=lcm_kw.get("sum_below", 2**31 - 1))["total"] for c in cases]
    t_cpu_lcm = (time.perf_counter() - t0) * 1e3
    assert cpu_obj == obj_b.tolist() and cpu_lcm == tot_b.tolist(), "GPU != host reference"
    return {
        "workload": name, "B": B, "n": n, "n_cabs": n_cabs or n, "lcm_params": lcm_kw,
        "working_set_MB": round(B * n * n * 4 / 1e6, 1),
        "assign_batch_ms": t_assign, "lcm_batch_ms": t_lcm, "assign_loop_ms": t_loop_assign, "lcm_loop_ms": t_loop_lcm,
        "host_core_scipy_lsa_ms": t_cpu_lsa, "host_core_lcm_c_ms": t_cpu_lcm,
        "speedup_assign_vs_loop": t_loop_assign["median"] / t_assign["median"],
        "speedup_lcm_vs_loop": t_loop_lcm["median"] / t_lcm["median"],
        "batch_equals_loop": True,
    }


def run_paper(cases_n, seed):
    import torch
    from oracle import gen_inputs as g
    from taxidispatcher_b200 import experiments as ex
    dist = g.stand_distances(4000)
    rng = np.random.default_rng(seed)
    cases = [(g.rand_list(rng, 400, 4000), g.rand_list(rng, 400, 4000)) for _ in range(cases_n)]
    times, res = [], None
    for _ in range(4):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        res = ex.split_hybrid_vs_optimum(dist, cases, threshold=10)
        times.append((time.perf_counter() - t0) * 1e3)
    r = np.array([[a, b, c, d, e] for a, b, c, d, e in res], dtype=np.float64)
    return {"cases": cases_n, "e2e_ms": float(np.median(times[1:])), "runs_ms": times,
            "mean_split_over_opt": float(np.mean(r[:, 1] / r[:, 0])), "mean_lcm_over_opt": float(np.mean(r[:, 2] / r[:, 0])),
            "mean_best_over_opt": float(np.mean(np.minimum(r[:, 1], r[:, 2]) / r[:, 0])),
            "mean_hybrid_over_opt": float(np.mean(r[:, 3] / r[:, 0])), "mean_n2": float(np.mean(r[:, 4]))}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--loop-reps", type=int, default=2)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("cluster_batch_bench.py needs a CUDA device")
    res = {"bench": "batch_cluster_instances", "card": card(),
           "note": "1000 x 400^2 (640 MB) and 200 x 600^2 (288 MB) exceed the 126 MB L2: HBM figures; "
                   "the 1- to 8-instance workloads are L2-resident",
           "workloads": [run_workload(*w, args.reps, args.loop_reps, args.seed + i) for i, w in enumerate(WORKLOADS)],
           "split_hybrid_vs_optimum": run_paper(1000, 56)}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
