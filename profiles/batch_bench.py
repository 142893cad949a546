"""Batched small instances against per-instance calls and one host core: prints ONE JSON line.

Workloads (B instances of n x n, U[1,39] costs like heuristic.py:20-40):
  (1000, 100)   heuristic.py:20-40, the paper's p.4 experiment
  (592, 200)    config 1 shape (python.py), 4 waves of 148 CTAs at one CTA per SM
  (20000, 32)   many tiny instances

For each: the batched kernels (td_assign_exact_batch, td_lcm_batch; CUDA events, median of --reps launches after a
warm-up), the loop of existing single-instance calls (Engine.assign / Engine.lcm) over the same device-resident
matrices (CUDA events around the whole loop, median of --loop-reps loops), the end-to-end helper (dispatch.run_batch:
pack + one upload + both kernels + one read-back; host clock), and one host core running scipy's
linear_sum_assignment and the C restatement of the literal LCM (oracle/lcm_oracle.c) over the same instances.
The batch and the loop are asserted to give identical outputs in the same run.

The working sets are small (40 MB at (1000, 100), 95 MB at (592, 200), 82 MB at (20000, 32)) and are read from the
126 MB L2 after the first pass, so the kernel times are L2-resident figures, not HBM ones.

    python profiles/batch_bench.py [--reps 30] [--loop-reps 3] [--out FILE]
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

WORKLOADS = [(1000, 100), (592, 200), (20000, 32)]


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
    return float(np.median(times)), float(np.min(times)), float(np.max(times))


def run_workload(B, n, reps, loop_reps, seed):
    import torch
    from scipy.optimize import linear_sum_assignment
    from oracle import lcm_ref
    from taxidispatcher_b200 import dispatch

    eng = dispatch.engine()
    rng = np.random.default_rng(seed)
    cases = [rng.integers(1, 40, (n, n)).astype(np.int32) for _ in range(B)]
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    offs_h = offs.cpu().numpy()
    mats = [packed[int(o): int(o) + n * n].view(n, n) for o in offs_h]
    a_out = {"col": torch.empty((B, n_max), dtype=torch.int32, device="cuda"),
             "objective": torch.empty(B, dtype=torch.int64, device="cuda")}
    l_out = {"rows": torch.empty((B, n_max), dtype=torch.int32, device="cuda"),
             "cols": torch.empty((B, n_max), dtype=torch.int32, device="cuda"),
             "n_pairs": torch.empty(B, dtype=torch.int32, device="cuda"),
             "total": torch.empty(B, dtype=torch.int64, device="cuda"),
             "last_min": torch.empty(B, dtype=torch.int32, device="cuda")}
    do_assign = lambda: eng.assign_batch(packed, sizes, offs, n_max, out=a_out)          # noqa: E731
    do_lcm = lambda: eng.lcm_batch(packed, sizes, offs, n_max, mask_value=100, out=l_out)  # noqa: E731
    for _ in range(3):
        do_assign()
        do_lcm()
    torch.cuda.synchronize()
    t_assign = events_ms(do_assign, reps)
    t_lcm = events_ms(do_lcm, reps)

    loop_out = {}

    def loop_assign():
        loop_out["assign"] = [eng.assign(m)[:2] for m in mats]

    def loop_lcm():
        loop_out["lcm"] = [eng.lcm(m, 100) for m in mats]

    loop_assign()
    loop_lcm()
    torch.cuda.synchronize()
    t_loop_assign = events_ms(loop_assign, loop_reps)
    t_loop_lcm = events_ms(loop_lcm, loop_reps)

    # identical outputs, batch vs loop (same run)
    col_b, obj_b = a_out["col"].cpu().numpy(), a_out["objective"].cpu().numpy()
    col_l = torch.stack([c for c, _ in loop_out["assign"]]).cpu().numpy()
    obj_l = torch.cat([o for _, o in loop_out["assign"]]).cpu().numpy()
    assert np.array_equal(col_b[:, :n], col_l) and np.array_equal(obj_b, obj_l), "assign: batch != loop"
    rows_b, cols_b = l_out["rows"].cpu().numpy(), l_out["cols"].cpu().numpy()
    np_b, tot_b, last_b = (l_out[k].cpu().numpy() for k in ("n_pairs", "total", "last_min"))
    for k, (r, c, s) in enumerate(loop_out["lcm"]):
        h = dispatch.Engine.lcm_host_view(r, c, s)
        m = h["n_pairs"]
        assert (np_b[k], tot_b[k], last_b[k]) == (m, h["total"], h["last_min"]), ("lcm: batch != loop", k)
        assert np.array_equal(rows_b[k, :m], h["rows"]) and np.array_equal(cols_b[k, :m], h["cols"]), ("lcm rows", k)

    # end to end: pack + one upload + both kernels + one read-back
    e2e = []
    for _ in range(4):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        opt, lcm = dispatch.run_batch(cases, assign=True, lcm=dict(mask_value=100))
        e2e.append((time.perf_counter() - t0) * 1e3)
    e2e_ms = float(np.median(e2e[1:]))
    assert [o[1] for o in opt] == obj_b.tolist() and [d["total"] for d in lcm] == tot_b.tolist()

    # one host core: scipy LSA and the literal LCM in C
    t0 = time.perf_counter()
    cpu_obj = []
    for c in cases:
        r, cc = linear_sum_assignment(c)
        cpu_obj.append(int(c[r, cc].sum()))
    t_cpu_lsa = (time.perf_counter() - t0) * 1e3
    t0 = time.perf_counter()
    cpu_lcm = [lcm_ref.lcm_c(c, 100)["total"] for c in cases]
    t_cpu_lcm = (time.perf_counter() - t0) * 1e3
    assert cpu_obj == obj_b.tolist() and cpu_lcm == tot_b.tolist(), "GPU != host reference"

    ratio = float(np.mean(tot_b / obj_b))
    return {
        "B": B, "n": n, "working_set_MB": round(B * n * n * 4 / 1e6, 1),
        "assign_batch_ms": {"median": t_assign[0], "min": t_assign[1], "max": t_assign[2], "reps": reps},
        "lcm_batch_ms": {"median": t_lcm[0], "min": t_lcm[1], "max": t_lcm[2], "reps": reps},
        "assign_loop_ms": {"median": t_loop_assign[0], "min": t_loop_assign[1], "max": t_loop_assign[2], "reps": loop_reps},
        "lcm_loop_ms": {"median": t_loop_lcm[0], "min": t_loop_lcm[1], "max": t_loop_lcm[2], "reps": loop_reps},
        "run_batch_e2e_ms": e2e_ms,
        "host_core_scipy_lsa_ms": t_cpu_lsa, "host_core_lcm_c_ms": t_cpu_lcm,
        "speedup_assign_vs_loop": t_loop_assign[0] / t_assign[0], "speedup_lcm_vs_loop": t_loop_lcm[0] / t_lcm[0],
        "mean_lcm_over_opt": ratio,
        "batch_equals_loop": True,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=30)
    ap.add_argument("--loop-reps", type=int, default=3)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("batch_bench.py needs a CUDA device")
    res = {"bench": "batch_small_instances", "card": card(),
           "note": "working sets are L2-resident after the first pass (40 MB at (1000, 100)); kernel times are L2 figures",
           "workloads": [run_workload(B, n, args.reps, args.loop_reps, args.seed + i) for i, (B, n) in enumerate(WORKLOADS)]}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
