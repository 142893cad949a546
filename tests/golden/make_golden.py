#!/usr/bin/env python
"""Regenerates tests/golden/*.json.  Run from the repo root with a checkout of the reference:

    TD_REFERENCE_DIR=<checkout of boguszjelinski/taxidispatcher> python tests/golden/make_golden.py [--skip-722]
        [--only-crosscheck]

Sources of truth (nothing here touches the CUDA path):
  pool_*      the compiled reference oracle/_ref/pool_n_big (pool_n.c from $TD_REFERENCE_DIR,
              built by `make -C oracle ref`), 8 logical shards, merged in shard order
              (findpool.c:83-108 restated in oracle/pool_oracle.c); pool_reference_crosscheck.json
              holds its single-shard answers for the cross-checks of tests/test_oracle.py
  lcm_*       the reference LCM bodies executed by numpy (oracle/lcm_ref.py)
  assign_*    scipy.optimize.linear_sum_assignment / linprog(HiGHS) on the reference layout and
              the literals of python.py:7, glpk.mod:27-31, procedure.py:32-51
The tests read the committed JSON; the cross-checks run the compiled reference instead where it is built.
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import hashlib
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import assign_ref, cost_ref, gen_inputs as g, lcm_ref, pool_ref  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
CROSSCHECK = "pool_reference_crosscheck.json"


def sha(arr) -> str:
    return hashlib.sha256(np.ascontiguousarray(np.asarray(arr, dtype=np.int32)).tobytes()).hexdigest()


def dump(name, obj):
    with open(os.path.join(OUT, name), "w") as f:
        json.dump(obj, f, separators=(",", ":"))
        f.write("\n")
    print("wrote", name)


def _ref_shard(args):
    dem, k, sh = args
    plans, st = pool_ref.run_reference(dem, k, sh)
    return sh, plans.tolist(), st


def pool_case(dem, k, label):
    with cf.ProcessPoolExecutor(8) as ex:
        res = sorted(ex.map(_ref_shard, [(dem, k, sh) for sh in range(8)]))
    shards = [{"shard": sh, "plans": p, "stats": st} for sh, p, st in res]
    merged = pool_ref.merge([np.asarray(s["plans"], dtype=np.int32).reshape(-1, 9) for s in shards], len(dem), k)
    return {"label": label, "pool_size": k, "n": int(len(dem)), "demand_sha256": sha(dem), "shards": shards,
            "merged": merged.tolist()}


def _huge_slice(args):
    """One `pool_n_huge512 4 t demand.csv n out.csv` run of the compiled reference (pool_n.c:209-238)."""
    import re
    import subprocess
    import tempfile
    exe, dem, t = args
    with tempfile.TemporaryDirectory() as td:
        with open(os.path.join(td, "demand.csv"), "w") as f:
            f.write(g.demand_csv(dem))
        res = subprocess.run([exe, "4", str(t), "demand.csv", str(len(dem)), "out.csv"], cwd=td, capture_output=True,
                             text=True, check=True)
        plans = pool_ref.parse_result_csv(open(os.path.join(td, "out.csv")).read(), 4)
    m = {k: int(v) for k, v in re.findall(r"(Count ALL|Count|Not duplicated count): (-?\d+)", res.stdout)}
    return {"slice": t, "plans": plans.tolist(),
            "stats": {"evaluated_mod_2_32": m["Count ALL"] % (1 << 32), "feasible": m["Count"], "kept": m["Not duplicated count"]}}


def large_slices(spec):
    """north star (>= 5k customers): slices of the reference's own shard rule with MAX_THREAD = 512 (pool_n.c:13,226-229)
    -- the rule is the same for any thread count, so `find_pool(dem, dist, 4, shard=t, n_shards=512)` must reproduce
    each slice bit for bit.  count_all is a 32-bit int in the reference (pool_n.c:28): compared modulo 2^32."""
    import subprocess
    n, ts = spec.split(":")
    n = int(n)
    ts = [int(t) for t in ts.split(",")]
    exe = os.path.join(ROOT, "oracle", "_ref", "pool_n_huge512")
    subprocess.check_call(["make", "-C", os.path.join(ROOT, "oracle"), "_ref/pool_n_huge512"])
    dem = g.pool_demand(n, seed=n)
    with cf.ProcessPoolExecutor(min(len(ts), 6)) as ex:
        slices = list(ex.map(_huge_slice, [(exe, dem, t) for t in ts]))
    dump("pool%d_slices.json" % n, {"label": "large_%d_512way" % n, "pool_size": 4, "n": n, "n_stands": 50, "seed": n,
                                    "n_shards": 512, "demand_sha256": sha(dem), "slices": slices})


def crosscheck():
    """What the two cross-checks of tests/test_oracle.py compare against, for checkouts without the compiled reference:
    its plans and counters on gen_inputs.pool_crosscheck_cases() and on gen_inputs.demand_quirks_csv()."""
    cases = [{"pool_size": k, "shard": sh, "demand_sha256": sha(dem), "plans": p.tolist(), "stats": st}
             for k, dem, sh in g.pool_crosscheck_cases() for p, st in [pool_ref.run_reference(dem, k, sh)]]
    text = g.demand_quirks_csv()
    quirks = [{"pool_size": k, "shard": sh,
               "plans": pool_ref.run_reference_csv(text, g.DEMAND_QUIRKS_REC_NUMBER, k, sh)[0].tolist()}
              for k, sh in g.DEMAND_QUIRKS_RUNS]
    dump(CROSSCHECK, {"source": "oracle/_ref/pool_n_big (pool_n.c compiled by `make -C oracle ref`)",
                      "cases": cases, "demand_quirks": quirks})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--skip-722", action="store_true")
    ap.add_argument("--only-crosscheck", action="store_true", help="only write " + CROSSCHECK)
    ap.add_argument("--only-large", type=int, default=0, help="only write pool<N>.json for N customers (minutes of CPU)")
    ap.add_argument("--large-slices", default="", help="N:t0,t1,...: slices t of the 512-way shard rule of pool_n.c for N "
                                                        "customers (north-star size; ~10 CPU-minutes per slice, run in parallel)")
    a = ap.parse_args()
    if a.large_slices:
        large_slices(a.large_slices)
        return
    if a.only_large:
        dem = g.pool_demand(a.only_large, seed=a.only_large)
        c = pool_case(dem, 4, "large_%d" % a.only_large)
        c["n_stands"] = 50
        c["seed"] = a.only_large
        dump("pool%d.json" % a.only_large, c)
        return
    assert pool_ref.reference_binary(), "build oracle/_ref first: make -C oracle ref"
    crosscheck()
    if a.only_crosscheck:
        return

    # ---- pool: small cases (KAT P1) with the inputs inlined ---------------------------------
    small = []
    rng = np.random.default_rng(3)
    for n, seed, vary in ((60, 7, False), (180, 11, False), (120, 12, True), (97, 13, True)):
        dem = g.pool_demand(n, seed=seed)
        if vary:
            dem[:, 3] = rng.integers(0, 8, n)
            dem[:, 4] = rng.integers(0, 60, n)
        for k in (2, 3, 4):
            c = pool_case(dem, k, "n%d_seed%d_k%d%s" % (n, seed, k, "_var" if vary else ""))
            c["demand"] = dem.tolist()
            c["n_stands"] = 51
            small.append(c)
    dump("pool_small.json", small)

    # ---- pool: config 3 (KAT P2), 722 customers, 4 passengers ------------------------------
    if not a.skip_722:
        dem = g.pool_demand()
        assert g.demand_md5(dem) == g.POOL722_MD5
        c = pool_case(dem, 4, "config3_722")
        c["n_stands"] = 50
        assert [s["stats"]["evaluated"] for s in c["shards"]] == g.POOL722_EVALUATED
        assert [s["stats"]["feasible"] for s in c["shards"]] == g.POOL722_FEASIBLE
        assert [s["stats"]["kept"] for s in c["shards"]] == g.POOL722_KEPT
        m = np.asarray(c["merged"])
        assert len(m) == 110 and int(m[:, 8].sum()) == 1840, (len(m), m[:, 8].sum())
        dump("pool722.json", c)

    # ---- LCM --------------------------------------------------------------------------------
    lcm = {}
    C = g.config2()
    tot, rows, cols = lcm_ref.lcm_heuristic(2000, C.reshape(-1))
    lcm["config2_heuristic"] = {"n": 2000, "seed": 2000, "mask": 100, "total": int(tot), "rows_sha256": sha(rows),
                                "cols_sha256": sha(cols), "first": [rows[:8], cols[:8]], "last": [rows[-8:], cols[-8:]]}
    Cs = g.config2_stand()
    tot, rows, cols = lcm_ref.lcm_split(2000, Cs)
    lcm["config2_stand_split"] = {"n": 2000, "seed": 2001, "mask": g.BIG_COST, "total": int(tot),
                                  "rows_sha256": sha(rows), "cols_sha256": sha(cols)}
    tot, rows, cols = lcm_ref.lcm_greedy_opt(2000, Cs, threshold=10)
    lcm["config2_stand_greedy_opt_thr10"] = {"n": 2000, "total": int(tot), "n_pairs": len(rows),
                                             "rows_sha256": sha(rows), "cols_sha256": sha(cols)}
    # dummy rows (10 of big_cost) -> exercises the "mask is a value" tail (SURVEY section 4 trap 4)
    dist, cab_to, cust_from = g.config1b()
    n, cost = cost_ref.calculate_cost_np(dist, cab_to, cust_from)
    tot, rows, cols = lcm_ref.lcm_split(n, cost)
    lcm["config1b_split"] = {"n": n, "total": int(tot), "rows": [int(v) for v in rows], "cols": [int(v) for v in cols]}
    pairs, mn = lcm_ref.lcm_java(cost, max_non_lcm=150)
    lcm["config1b_java_res150"] = {"n": n, "pairs": [[int(a_), int(b_)] for a_, b_ in pairs], "lcm_min_val": int(mn)}
    dump("lcm.json", lcm)

    # ---- assignment -------------------------------------------------------------------------
    asg = {}
    A1 = np.array([5, 5, 0, 5, 1, 1, 3, 8, 9, 9, 5, 0, 100, 100, 100, 100]).reshape(4, 4)   # python.py:7
    asg["A1_python_py"] = {"cost": A1.tolist(), "objective": 101, "optimal_perms": [[2, 0, 3, 1], [2, 1, 3, 0]],
                           "lp": assign_ref.lp_relaxation(A1)[0]}
    A2 = np.array([[5, 1, 9, 100], [5, 1, 9, 100], [0, 3, 5, 100], [5, 8, 0, 100]])          # glpk.mod:27-31
    asg["A2_glpk_mod"] = {"cost": A2.tolist(), "objective": 101, "lp": assign_ref.lp_relaxation(A2)[0]}
    d10 = g.stand_distances(10)
    n, c = cost_ref.calculate_cost_by_id(d10, [(0, 0, 2), (1, 0, 5), (2, 3, 1), (3, 5, 1)],
                                         [(0, 3, 3), (1, 3, 1), (2, 0, 5)])                  # procedure.py:32-51
    asg["A3_procedure_py"] = {"cost": c, "objective": 17}
    assert assign_ref.solve_scipy(np.array(c))[0] == 17 and assign_ref.solve_scipy(A1)[0] == 101
    C1 = g.config1a()
    asg["config1a"] = {"n": 200, "objective": assign_ref.solve_scipy(C1)[0], "lp": assign_ref.lp_relaxation(C1)[0]}
    dist, cab_to, cust_from = g.config1b()
    n, cost = cost_ref.calculate_cost_np(dist, cab_to, cust_from)
    asg["config1b"] = {"n": n, "objective": assign_ref.solve_scipy(cost)[0], "lp": assign_ref.lp_relaxation(cost)[0],
                       "cost_sha256": sha(cost)}
    asg["config2"] = {"n": 2000, "objective": assign_ref.solve_scipy(g.config2())[0]}
    asg["config2_stand"] = {"n": 2000, "objective": assign_ref.solve_scipy(g.config2_stand())[0]}
    for nn in (5000,):
        asg["config5a_n%d" % nn] = {"n": nn, "objective": assign_ref.solve_scipy(g.config5a(nn))[0]}
        asg["config5b_n%d" % nn] = {"n": nn, "objective": assign_ref.solve_scipy(g.config5b_cost(nn))[0]}
    dump("assign.json", asg)


if __name__ == "__main__":
    main()
