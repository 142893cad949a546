"""Batches of large instances (641 <= n <= 2048) on thread-block clusters that read the matrix from global memory, against
the loop of single-instance calls and one host core: prints ONE JSON line (kept in profiles/large_batch_b200.json).

Workloads (B instances of n x n):
  u2000      100 x 2000^2, U[1,39] costs (heuristic.py's config 2): assignment, and LCM with mask 100
  stand2000  100 x 2000^2, 2000 cabs x 2000 customers over 4000 stands (gen_inputs.config2_stand's distribution):
             assignment
  sim1300    100 x 1300^2, Simulator-shaped (50 stands, cutoff 10, big_cost fill, 1100-1300 cabs): the java LCM
             (stop at big_cost, residual 600)
  perf1000   200 x 1000^2, U[1,39] (perf.jl's size): assignment and LCM with mask 100
  crossover  1, 2, 4, 8 and 16 instances at 700, 1300 and 2000 rows, U[1,39] and stand-derived: where the batch starts
             to beat the loop (dispatch.ASSIGN_LARGE_MIN_BATCH / LCM_LARGE_MIN_BATCH)
  forms600   200 x 600^2, 560 cabs x 600 customers over 4000 stands: td_*_batch_cluster (matrix in DSMEM) against
             td_*_batch_large (matrix in global memory) on the same buffer, outputs asserted bit-identical

Batch times are CUDA-event medians of --reps launches after a warm-up; loop times are CUDA events around the whole loop
of Engine.assign / Engine.lcm over the same device-resident matrices, median of --loop-reps loops.  Batch and loop are
asserted to return the same objectives and the same LCM traces in the same run.  scipy's linear_sum_assignment runs on
one host core over the first --cpu-subset instances of a workload and is scaled to the whole batch (labelled as such).

The 100 x 2000^2 working sets are 1.6 GB, 100 x 1300^2 676 MB, 200 x 1000^2 800 MB and 200 x 600^2 288 MB: all larger
than the 126 MB L2, so these figures include HBM.  The crossover batches (at most 256 MB) are partly L2-resident.

    python profiles/large_batch_bench.py [--reps 5] [--loop-reps 2] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

BIG_COST = 250000
LCM_HEUR = dict(mask_value=100)
LCM_SPLIT = dict(mask_value=BIG_COST, sum_below=BIG_COST)
LCM_JAVA = dict(mask_value=BIG_COST, stop_at_value=BIG_COST, residual_size=600)


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


def uniform_cases(rng, B, n):
    return [rng.integers(1, 40, (n, n)).astype(np.int32) for _ in range(B)]


def stand_cases(rng, B, n, n_cabs=None, n_stands=4000):
    """calculate_cost over n_stands stands (|i - j| distances), n_cabs cabs x n customers, big_cost padding rows"""
    out = []
    for _ in range(B):
        cab_to = rng.integers(0, n_stands, n_cabs or n)
        cust = rng.integers(0, n_stands, n)
        m = np.full((n, n), BIG_COST, np.int32)
        m[: len(cab_to)] = np.abs(cab_to[:, None] - cust[None, :])
        out.append(m)
    return out


def device_batch(cases=None, packed_meta=None):
    from taxidispatcher_b200 import dispatch
    packed, sizes, offs, n_max = packed_meta if packed_meta is not None else dispatch.pack_batch(cases)
    ns = sizes.cpu().numpy()
    o = offs.cpu().numpy()
    mats = [packed[int(o[k]): int(o[k]) + int(n) * int(n)].view(int(n), int(n)) for k, n in enumerate(ns)]
    return packed, sizes, offs, n_max, mats


def outs(B, n_max):
    import torch
    a = {"col": torch.empty((B, n_max), dtype=torch.int32, device="cuda"),
         "objective": torch.empty(B, dtype=torch.int64, device="cuda"),
         "u": torch.empty((B, n_max), dtype=torch.int64, device="cuda"),
         "v": torch.empty((B, n_max), dtype=torch.int64, device="cuda")}
    l_ = {"rows": torch.empty((B, n_max), dtype=torch.int32, device="cuda"),
          "cols": torch.empty((B, n_max), dtype=torch.int32, device="cuda"),
          "n_pairs": torch.empty(B, dtype=torch.int32, device="cuda"),
          "total": torch.empty(B, dtype=torch.int64, device="cuda"),
          "last_min": torch.empty(B, dtype=torch.int32, device="cuda")}
    return a, l_


def raw_call(eng, kernel, packed, sizes, offs, n_max, a_out=None, l_out=None, lcm_kw=None):
    """td_<kernel> on the packed buffer at any n_max (Engine.assign_batch / lcm_batch pick the kernel from n_max)"""
    from taxidispatcher_b200 import _lib
    p = lambda t: ctypes.c_void_p(t.data_ptr()) if t is not None else None   # noqa: E731
    B = int(sizes.numel())
    if a_out is not None:
        rc = getattr(eng.lib, "td_assign_exact_batch_" + kernel)(p(packed), p(sizes), p(offs), B, int(n_max), p(a_out["col"]),
                                                                 p(a_out["objective"]), p(a_out["u"]), p(a_out["v"]), None)
    else:
        prm = _lib.LcmParams(lcm_kw["mask_value"], lcm_kw.get("stop_above", 2**31 - 1), lcm_kw.get("stop_at_value", 2**31 - 1),
                             lcm_kw.get("sum_below", 2**31 - 1), lcm_kw.get("residual_size", 0), lcm_kw.get("max_iters", -1))
        rc = getattr(eng.lib, "td_lcm_batch_" + kernel)(p(packed), p(sizes), p(offs), B, int(n_max), ctypes.byref(prm),
                                                        p(l_out["rows"]), p(l_out["cols"]), p(l_out["n_pairs"]),
                                                        p(l_out["total"]), p(l_out["last_min"]), None)
    assert rc == 0, (kernel, rc)


def time_side(eng, dev, which, lcm_kw, reps, loop_reps):
    """batch kernel and loop of single calls for one side ("assign" or "lcm"); asserts identical outputs"""
    import torch
    from taxidispatcher_b200 import dispatch
    packed, sizes, offs, n_max, mats = dev
    B = len(mats)
    a_out, l_out = outs(B, n_max)
    if which == "assign":
        batch = lambda: eng.assign_batch(packed, sizes, offs, n_max, want_duals=True, out=a_out)   # noqa: E731
    else:
        batch = lambda: eng.lcm_batch(packed, sizes, offs, n_max, out=l_out, **lcm_kw)             # noqa: E731
    loop_out = {}

    def loop():
        if which == "assign":
            loop_out["r"] = [eng.assign(m)[1] for m in mats]
        else:
            loop_out["r"] = [eng.lcm(m, **lcm_kw) for m in mats]
    batch()
    loop()
    torch.cuda.synchronize()
    t_batch = events_ms(batch, reps)
    t_loop = events_ms(loop, loop_reps)
    if which == "assign":
        obj_b = a_out["objective"].cpu().numpy()
        obj_l = torch.stack(loop_out["r"]).reshape(-1).cpu().numpy()
        assert np.array_equal(obj_b, obj_l), "assign: batch objective != loop objective"
        col = a_out["col"].cpu().numpy()
        assert all(sorted(col[k, : m.shape[0]].tolist()) == list(range(m.shape[0])) for k, m in enumerate(mats))
    else:
        rows_b, cols_b = l_out["rows"].cpu().numpy(), l_out["cols"].cpu().numpy()
        np_b, tot_b, last_b = (l_out[k].cpu().numpy() for k in ("n_pairs", "total", "last_min"))
        for k, r in enumerate(loop_out["r"]):
            h = dispatch.Engine.lcm_host_view(*r)
            m = h["n_pairs"]
            assert (np_b[k], tot_b[k], last_b[k]) == (m, h["total"], h["last_min"]), ("lcm: batch != loop", k)
            assert np.array_equal(rows_b[k, :m], h["rows"]) and np.array_equal(cols_b[k, :m], h["cols"]), ("lcm rows", k)
    return {"batch_ms": t_batch, "loop_ms": t_loop, "speedup_vs_loop": t_loop["median"] / t_batch["median"],
            "batch_equals_loop": True, "objective_sum" if which == "assign" else "lcm_total_sum":
            int(a_out["objective"].sum().item()) if which == "assign" else int(l_out["total"].sum().item())}


def host_lsa(cases, subset):
    from scipy.optimize import linear_sum_assignment
    t0 = time.perf_counter()
    for c in cases[:subset]:
        linear_sum_assignment(c)
    per = (time.perf_counter() - t0) * 1e3 / subset
    return {"instances_timed": subset, "ms_per_instance": per, "scaled_to_batch_ms": per * len(cases),
            "note": "one host core, scipy linear_sum_assignment; scaled from the timed subset"}


def workload(name, cases, sides, reps, loop_reps, cpu_subset):
    from taxidispatcher_b200 import dispatch
    eng = dispatch.engine()
    dev = device_batch(cases)
    n = cases[0].shape[0]
    res = {"workload": name, "B": len(cases), "n": n, "working_set_MB": round(sum(c.size for c in cases) * 4 / 1e6, 1)}
    for which, kw in sides:
        res[which] = time_side(eng, dev, which, kw, reps, loop_reps)
        if kw is not None:
            res[which]["lcm_params"] = kw
    if cpu_subset and any(w == "assign" for w, _ in sides):
        res["host_core_scipy_lsa"] = host_lsa(cases, cpu_subset)
    return res


def sim_cases(rng, B, n=1300):
    from oracle import gen_inputs as g
    from taxidispatcher_b200 import dispatch
    dist_d = dispatch._h2d_i32(g.stand_distances(50))
    insts = [(rng.integers(0, 50, int(rng.integers(1100, n + 1))), rng.integers(0, 50, n)) for _ in range(B)]
    packed, sizes, offs, n_max, _ = dispatch.pack_cost_matrices(dist_d, insts, fill=BIG_COST, cutoff=10)
    return device_batch(packed_meta=(packed, sizes, offs, n_max))


def forms600(rng, reps, B=200):
    """the same B x 600^2 buffer through the DSMEM (cluster) and global-memory (large) forms"""
    import torch
    from taxidispatcher_b200 import dispatch
    eng = dispatch.engine()
    packed, sizes, offs, n_max, mats = device_batch(stand_cases(rng, B, 600, 560))
    res = {"workload": "forms600", "B": B, "n": 600, "n_cabs": 560, "working_set_MB": round(B * 600 * 600 * 4 / 1e6, 1)}
    got = {}
    for form in ("cluster", "large"):
        a_out, l_out = outs(B, n_max)
        fa = lambda: raw_call(eng, form, packed, sizes, offs, n_max, a_out=a_out)                     # noqa: E731
        fl = lambda: raw_call(eng, form, packed, sizes, offs, n_max, l_out=l_out, lcm_kw=LCM_SPLIT)   # noqa: E731
        fa()
        fl()
        torch.cuda.synchronize()
        res[form] = {"assign_ms": events_ms(fa, reps), "lcm_ms": events_ms(fl, reps)}
        got[form] = [t.cpu().numpy() for t in list(a_out.values()) + list(l_out.values())]
    for a, b in zip(got["cluster"], got["large"]):
        assert np.array_equal(a, b), "forms600: DSMEM and global forms differ"
    res["outputs_bit_identical"] = True
    res["lcm_params"] = LCM_SPLIT
    return res


def crossover(rng, reps, loop_reps, kinds=("uniform", "stand"), sizes=(700, 1300, 2000), batches=(1, 2, 4, 8, 16),
              sides=("assign", "lcm")):
    from taxidispatcher_b200 import dispatch
    eng = dispatch.engine()
    out = []
    for kind in kinds:
        for n in sizes:
            pool = uniform_cases(rng, max(batches), n) if kind == "uniform" else stand_cases(rng, max(batches), n)
            for B in batches:
                dev = device_batch(pool[:B])
                kw = LCM_HEUR if kind == "uniform" else LCM_SPLIT
                row = {"kind": kind, "n": n, "B": B}
                if "assign" in sides:
                    a = time_side(eng, dev, "assign", None, reps, loop_reps)
                    row.update(assign_batch_ms=a["batch_ms"]["median"], assign_loop_ms=a["loop_ms"]["median"])
                if "lcm" in sides:
                    l_ = time_side(eng, dev, "lcm", kw, reps, loop_reps)
                    row.update(lcm_batch_ms=l_["batch_ms"]["median"], lcm_loop_ms=l_["loop_ms"]["median"], lcm_params=kw)
                out.append(row)
    return out


def min_batch(rows, side):
    """the smallest B from which the batch is at least as fast as the loop at every measured size and kind"""
    for B in sorted({r["B"] for r in rows}):
        if all(r[side + "_batch_ms"] <= r[side + "_loop_ms"] for r in rows if r["B"] >= B and side + "_batch_ms" in r):
            return B
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--loop-reps", type=int, default=2)
    ap.add_argument("--cpu-subset", type=int, default=2)
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--only", default=None, help="comma-separated subset of u2000,stand2000,sim1300,perf1000,crossover,forms600")
    ap.add_argument("--forms-b", default="200", help="batch sizes of the forms600 comparison")
    ap.add_argument("--cross-n", default="700,1300,2000")
    ap.add_argument("--cross-b", default="1,2,4,8,16")
    ap.add_argument("--cross-kinds", default="uniform,stand")
    ap.add_argument("--cross-sides", default="assign,lcm")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("large_batch_bench.py needs a CUDA device")
    from taxidispatcher_b200 import dispatch
    only = set(args.only.split(",")) if args.only else None
    want = lambda k: only is None or k in only   # noqa: E731
    rng = np.random.default_rng(args.seed)
    res = {"bench": "batch_large_instances", "card": card(),
           "note": "100 x 2000^2 (1.6 GB), 100 x 1300^2 (676 MB), 200 x 1000^2 (800 MB) and 200 x 600^2 (288 MB) exceed "
                   "the 126 MB L2: HBM figures; the crossover batches (<= 256 MB) are partly L2-resident",
           "workloads": []}
    eng = dispatch.engine()
    if want("u2000"):
        res["workloads"].append(workload("u2000", uniform_cases(rng, 100, 2000), [("assign", None), ("lcm", LCM_HEUR)],
                                         args.reps, args.loop_reps, args.cpu_subset))
    if want("stand2000"):
        res["workloads"].append(workload("stand2000", stand_cases(rng, 100, 2000), [("assign", None)],
                                         args.reps, args.loop_reps, args.cpu_subset))
    if want("sim1300"):
        dev = sim_cases(rng, 100)
        res["workloads"].append({"workload": "sim1300", "B": 100, "n": 1300, "stands": 50, "cutoff": 10,
                                 "working_set_MB": round(100 * 1300 * 1300 * 4 / 1e6, 1),
                                 "lcm": dict(time_side(eng, dev, "lcm", LCM_JAVA, args.reps, args.loop_reps),
                                             lcm_params=LCM_JAVA)})
    if want("perf1000"):
        res["workloads"].append(workload("perf1000", uniform_cases(rng, 200, 1000), [("assign", None), ("lcm", LCM_HEUR)],
                                         args.reps, args.loop_reps, args.cpu_subset))
    if want("forms600"):
        fb = [int(b) for b in args.forms_b.split(",")]
        res["forms600"] = forms600(rng, args.reps, fb[-1])
        res["forms600_small"] = [forms600(rng, args.reps, b) for b in fb[:-1]]
    if want("crossover"):
        rows = crossover(rng, max(3, args.reps // 2), args.loop_reps, args.cross_kinds.split(","),
                         [int(x) for x in args.cross_n.split(",")], [int(x) for x in args.cross_b.split(",")],
                         args.cross_sides.split(","))
        res["crossover"] = rows
        res["measured_min_batch"] = {s: min_batch(rows, s) for s in args.cross_sides.split(",")}
    res["routing"] = {"ASSIGN_LARGE_MIN_BATCH": dispatch.ASSIGN_LARGE_MIN_BATCH,
                      "LCM_LARGE_MIN_BATCH": dispatch.LCM_LARGE_MIN_BATCH}
    line = json.dumps(res)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
