"""The findpool job batched (td_pool_find_all_batch), against the per-instance find_pool_all it replaces.

Workloads (gen_inputs.pool_demand: 50 stands, dist |i - j|, wait 3, loss 1 -- the Pool.java defaults):
  1000 x 100 customers at K = 2, 3 and 4; 148 x 300 customers at K = 4; 8 x 512 customers at K = 4 (few large
  instances: the side where the loop of single jobs may win).
Per workload:
  - kernel: td_pool_find_all_batch alone, inputs on the device, record slices sized from a first call (CUDA events);
  - batch end to end: find_pool_all_batch (pack + upload, one launch, one read-back; host clock, ends in a synchronise;
    K = 4 instances above POOL_BATCH_K4_LOOP_N customers take the find_pool_all route, reported as batch_route);
  - loop: find_pool_all over the same instances, end to end.  Its steady state replays a captured CUDA graph per shape
    (TD_POOL_GRAPH); whether that graph path was active is reported;
  - oracle: the C oracle (pool_ref.find per shard + pool_ref.merge) on one host core, on a subset, scaled to the batch.
Batch, kernel and loop outputs (plans and the four counters) are asserted identical for every instance, and batch
against the oracle on the subset.  Medians after a warm-up.  Prints one JSON line with the card's name and power limit read in the
same run, and also writes it to the file --out names (profiles/pool_batch_b200.json holds the committed line)."""
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

WORKLOADS = [("1000x100_k2", 1000, 100, 2), ("1000x100_k3", 1000, 100, 3), ("1000x100_k4", 1000, 100, 4),
             ("148x300_k4", 148, 300, 4), ("8x512_k4", 8, 512, 4)]


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
    """Median CUDA-event time of fn() in ms."""
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


def wall(fn, reps):
    """Median host time of fn() in ms; fn ends in a read-back, i.e. a synchronise."""
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return float(np.median(ts))


def oracle_all(dem, dist, k):
    from oracle import pool_ref
    parts, ev, fe, kept = [], 0, 0, []
    for s in range(8):
        p, st = pool_ref.find(dem, dist, k, s, 8)
        parts.append(p)
        ev += st["evaluated"]
        fe += st["feasible"]
        kept.append(st["kept"])
    merged = pool_ref.merge(parts, len(dem), k)
    return merged, {"evaluated": ev, "feasible": fe, "kept_per_shard": kept, "kept": len(merged)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--oracle-instances", type=int, default=4)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    assert torch.cuda.is_available(), "this benchmark measures the GPU; there is no CPU fallback"
    from oracle import gen_inputs as g
    from taxidispatcher_b200 import dispatch
    name, power = card()
    res = {"card": name, "power_limit": power}
    eng = dispatch.engine()
    dist = g.stand_distances(50)
    for label, B, n, k in WORKLOADS:
        inst = [g.pool_demand(n, seed=s) for s in range(B)]
        batch = dispatch.find_pool_all_batch(inst, dist, k)                    # warm-up; sizes the record slices
        demand, sizes, offsets, n_max, d = dispatch.pack_pool_batch(inst, dist)
        out = eng.pool_find_all_batch(demand, sizes, offsets, n_max, d, k, 8, dispatch.POOL_BATCH_FIRST_RECORDS)
        rps = max(1, int(out[5].max()))                                       # the kernel alone, slices sized exactly
        out = eng.pool_find_all_batch(demand, sizes, offsets, n_max, d, k, 8, rps)
        kplans, kcount, kev, kfe, kkept = [t.cpu().numpy() for t in out[:5]]
        assert int(kcount.min()) >= 0
        res["%s_kernel_ms" % label] = round(timed(lambda: eng.pool_find_all_batch(demand, sizes, offsets, n_max, d, k, 8, rps,
                                                                                  out=dict(zip(("plans", "n_plans", "evaluated",
                                                                                                "feasible", "kept", "needed"),
                                                                                               out))), args.reps), 3)
        res["%s_records_per_shard" % label] = rps
        res["%s_batch_end_to_end_ms" % label] = round(wall(lambda: dispatch.find_pool_all_batch(inst, dist, k), args.reps), 3)
        res["%s_batch_route" % label] = "kernel" if dispatch.pool_batch_routes([n], k)[0] else "find_pool_all"
        loop = [dispatch.find_pool_all(x, dist, k) for x in inst]               # warm-up: the graph of the shape is captured
        graph = any(isinstance(v, dispatch.PoolJobGraph) for v in dispatch._POOL_GRAPHS.values())
        res["%s_loop_find_pool_all_ms" % label] = round(wall(lambda: [dispatch.find_pool_all(x, dist, k) for x in inst],
                                                             max(1, args.reps // 2)), 3)
        res["%s_loop_graph_path" % label] = graph
        same = True
        for b, ((bp, bs), (lp, ls)) in enumerate(zip(batch, loop)):
            same &= bp.dtype == lp.dtype and bp.shape == lp.shape and bp.tobytes() == lp.tobytes()
            same &= all(bs[q] == ls[q] for q in ("evaluated", "feasible", "kept_per_shard", "kept"))
            m = int(kcount[b])                                                # and the kernel's own output
            same &= kplans[b, :m].tobytes() == lp.tobytes() and m == ls["kept"] and kkept[b].tolist() == ls["kept_per_shard"]
            same &= int(kev[b].sum()) == ls["evaluated"] and int(kfe[b].sum()) == ls["feasible"]
        assert same, label
        res["%s_equal_batch_and_loop" % label] = same
        m = min(B, args.oracle_instances)
        t0 = time.perf_counter()
        orc = [oracle_all(x, dist, k) for x in inst[:m]]
        res["%s_oracle_1core_ms" % label] = round((time.perf_counter() - t0) * 1e3 * B / m, 1)
        res["%s_oracle_instances_timed" % label] = m
        ok = all(np.array_equal(bp, op) and bs == os_ for (bp, bs), (op, os_) in zip(batch[:m], orc))
        assert ok, label
        res["%s_equal_oracle" % label] = ok
        dispatch.release_pool_graphs()
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
