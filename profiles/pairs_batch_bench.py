"""Greedy 2-passenger pool, batched (td_pool_pairs_batch), against the per-instance path it replaces.

  batch    1000 instances x 100 customers over 50 stands (dist |i - j|), accept_all 1 and 0:
           - the batch: kernel alone (CUDA events, inputs on the device) and find_pool_pairs_batch end to end
             (pack + upload, one launch, one read-back; host clock around work that ends in a synchronise);
           - the loop of find_pool_pairs over the same instances, end to end, which is what the pool experiment ran;
           - the C oracle (oracle/pool_ref.pairs) on one host core.
           Batch and loop rows are asserted byte-identical.
  gap      the whole pool_greedy_vs_optimum on those 1000 cases: the default path (one upload, the greedy and the exact
           batch launch, one read-back) against the old per-instance greedy (greedy=find_pool_pairs injected), wall clock;
           the outputs are asserted equal.
  single   one instance at n = 722 and 1445, random and all on one stand (the greedy's worst case: about n/2 rounds
           in which nearly every customer rescans): batch of one against td_pool_pairs, both with inputs on the device,
           CUDA events.  Informational: whether the single-instance path should use the batch kernel.

Medians of repeated runs after a warm-up.  The batch's working set (0.8 MB of inputs, 1.6 MB of outputs) is L2-resident
after the warm-up.  Prints one JSON line with the card's name and power limit read in the same run, and also writes it
to the file --out names (profiles/pairs_batch_b200.json holds the committed line)."""
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
    import torch
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1000)
    return float(np.median(ts))


def same(a, b):
    return all(x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes() for x, y in zip(a, b)) and len(a) == len(b)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    from oracle import pool_ref
    from taxidispatcher_b200 import dispatch, experiments
    D = np.abs(np.subtract.outer(np.arange(50), np.arange(50))).astype(np.int32)
    rng = np.random.default_rng(2026)
    eng = dispatch.engine()
    res = {"card": None, "power_limit": None, "l2": "batch working set L2-resident (warmed, < 126 MB)"}
    res["card"], res["power_limit"] = card()

    inst = [(rng.integers(0, 50, 100).astype(np.int32), rng.integers(0, 50, 100).astype(np.int32)) for _ in range(1000)]
    loop_reps = max(3, args.reps // 3)
    for acc in (1, 0):
        frm, to, sizes, offs, n_max, d = dispatch.pack_pairs_batch(inst, D)
        run = lambda: eng.pool_pairs_batch(frm, to, sizes, offs, n_max, d, bool(acc), 1.01)  # noqa: E731
        run()
        torch.cuda.synchronize()
        res["batch1000x100_acc%d_kernel_ms" % acc] = round(timed(run, args.reps), 3)
        batch = dispatch.find_pool_pairs_batch(inst, D, bool(acc), 1.01)
        res["batch1000x100_acc%d_end_to_end_ms" % acc] = round(
            wall(lambda: dispatch.find_pool_pairs_batch(inst, D, bool(acc), 1.01), args.reps), 3)
        loop = [dispatch.find_pool_pairs(f, t, D, bool(acc), 1.01) for f, t in inst]
        assert same(batch, loop), "batch rows differ from the find_pool_pairs loop"
        res["loop1000x100_acc%d_find_pool_pairs_ms" % acc] = round(
            wall(lambda: [dispatch.find_pool_pairs(f, t, D, bool(acc), 1.01) for f, t in inst], loop_reps), 1)
        t0 = time.perf_counter()
        ref = [pool_ref.pairs(f, t, D, bool(acc), 1.01) for f, t in inst]
        res["batch1000x100_acc%d_oracle_1core_ms" % acc] = round((time.perf_counter() - t0) * 1000, 1)
        res["batch1000x100_acc%d_equal_loop_and_oracle" % acc] = same(batch, loop) and all(
            np.array_equal(a, b) for a, b in zip(batch, ref))

    new = experiments.pool_greedy_vs_optimum(inst, D, True, 1.01)
    old = experiments.pool_greedy_vs_optimum(inst, D, True, 1.01, greedy=dispatch.find_pool_pairs)
    assert new == old, "pool_greedy_vs_optimum: default path differs from the per-instance greedy"
    res["experiment1000x100_default_ms"] = round(
        wall(lambda: experiments.pool_greedy_vs_optimum(inst, D, True, 1.01), args.reps), 1)
    res["experiment1000x100_per_instance_greedy_ms"] = round(
        wall(lambda: experiments.pool_greedy_vs_optimum(inst, D, True, 1.01, greedy=dispatch.find_pool_pairs), loop_reps), 1)
    res["experiment1000x100_equal"] = new == old

    for n in (722, 1445):
        for kind in ("random", "one_stand"):
            if kind == "random":
                f, t = rng.integers(0, 50, n).astype(np.int32), rng.integers(0, 50, n).astype(np.int32)
            else:
                f, t = np.full(n, 7, np.int32), np.full(n, 7, np.int32)
            frm, to, sizes, offs, n_max, d = dispatch.pack_pairs_batch([(f, t)], D)
            run_b = lambda: eng.pool_pairs_batch(frm, to, sizes, offs, n_max, d, True, 1.01)  # noqa: E731
            fd, td_, dd = dispatch._h2d_i32(f), dispatch._h2d_i32(t), dispatch._h2d_i32(D)
            run_s = lambda: eng.pool_pairs(fd, td_, dd, True, 1.01)  # noqa: E731
            rows, npairs, _ = run_b()
            out, cnt = run_s()
            k = int(cnt.item())
            equal = int(npairs[0]) == k and torch.equal(rows[0, :k], out[:k])
            assert equal, "batch of one differs from td_pool_pairs at n = %d (%s)" % (n, kind)
            key = "single_n%d_%s" % (n, kind)
            res[key + "_batch_of_one_ms"] = round(timed(run_b, max(3, args.reps // 2)), 3)
            res[key + "_td_pool_pairs_ms"] = round(timed(run_s, max(3, args.reps // 2)), 3)
            res[key + "_equal"] = equal

    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(args.out) or ".", exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
