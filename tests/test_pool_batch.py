"""The findpool job batched: td_pool_find_all_batch (every logical shard of pool_n.c + the findpool.c merge, one CTA per
(instance, shard), one launch), Engine.pool_find_all_batch, pack_pool_batch and find_pool_all_batch.

CPU: argument validation and the no-device return of the C ABI (no launches), the workspace query, the routing helpers.
GPU: plans byte for byte and every counter against both find_pool_all and the C oracle (pool_ref.find per shard, then
pool_ref.merge): the golden pool cases, sizes 0 to 512, 1 to 64 shards, the input families of the single-instance pool
tests, ragged / poisoned / withdrawn batches, independence from position, n_max and neighbours, repeatability, a forced
record-slice overflow, 1000 instances in one launch and a mix of sizes on both sides of the batch limit."""
import ctypes

import numpy as np
import pytest

from conftest import load_golden
from oracle import gen_inputs as g
from oracle import pool_ref

MAX_N = 512
D50 = g.stand_distances(50)


# ---- CPU: the C ABI refuses bad arguments before it looks for a device -----------------------------------------------
def _abi():
    from taxidispatcher_b200 import _lib
    return _lib, _lib.lib()


def _call(lib, demand=16, sizes=32, offsets=48, batch=2, n_max=100, dist=64, n_stands=50, pool_size=4, n_shards=8,
          plans=80, n_plans=96, evaluated=112, feasible=128, kept=144, needed=160, ws=176, ws_bytes=None, rps=1024):
    p = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    if ws_bytes is None:
        ws_bytes = lib.td_pool_batch_workspace_bytes(max(batch, 0), n_shards, rps) if 1 <= n_shards <= 64 else 1 << 40
    return lib.td_pool_find_all_batch(p(demand), p(sizes), p(offsets), batch, n_max, p(dist), n_stands, pool_size, n_shards,
                                      p(plans), p(n_plans), p(evaluated), p(feasible), p(kept), p(needed), p(ws), ws_bytes,
                                      rps, None)


def test_pool_batch_abi_argument_validation():
    _lib, lib = _abi()
    INV = _lib.TD_ERR_INVALID
    launches = lib.td_launch_count()
    assert _call(lib, batch=-1) == INV
    assert _call(lib, n_max=-1) == INV
    assert _call(lib, n_max=MAX_N + 1) == INV
    for k in (0, 1, 5):
        assert _call(lib, pool_size=k) == INV, k
    for s in (0, 65, -3):
        assert _call(lib, n_shards=s, ws_bytes=1 << 40) == INV, s
    assert _call(lib, n_stands=0) == INV
    assert _call(lib, n_stands=129) == INV
    assert _call(lib, rps=-1, ws_bytes=1 << 40) == INV
    for name in ("demand", "sizes", "offsets", "dist", "plans", "n_plans", "evaluated", "feasible", "kept", "needed"):
        assert _call(lib, **{name: None}) == INV, name
    # the size checks hold for an empty batch too
    assert _call(lib, batch=0, n_max=MAX_N + 1) == INV
    assert _call(lib, batch=0, pool_size=5) == INV
    assert _call(lib, batch=0, n_stands=0) == INV
    # a workspace smaller than the query (or none at all)
    need = lib.td_pool_batch_workspace_bytes(2, 8, 1024)
    assert _call(lib, ws_bytes=need - 1) == _lib.TD_ERR_WORKSPACE
    assert _call(lib, ws=None) == _lib.TD_ERR_WORKSPACE
    assert lib.td_launch_count() == launches


def test_pool_batch_workspace_query():
    _lib, lib = _abi()
    q = lib.td_pool_batch_workspace_bytes
    assert q(-1, 8, 10) == 0 and q(4, 0, 10) == 0 and q(4, 65, 10) == 0 and q(4, 8, -1) == 0 and q(4, 8, 1 << 31) == 0
    # one 8-byte key per record and (instance, shard)
    assert q(10, 8, 2000) - q(10, 8, 1000) == 10 * 8 * 1000 * 8
    assert q(20, 8, 1000) > q(10, 8, 1000) > 0


def test_pool_batch_abi_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    _lib, lib = _abi()
    launches = lib.td_launch_count()
    assert _call(lib) == _lib.TD_ERR_NO_DEVICE
    assert _call(lib, batch=0) == _lib.TD_ERR_NO_DEVICE
    assert _call(lib, n_max=MAX_N, pool_size=2, n_shards=64, n_stands=128) == _lib.TD_ERR_NO_DEVICE
    assert lib.td_launch_count() == launches


def test_pool_batch_routing():
    from taxidispatcher_b200 import dispatch
    assert dispatch.POOL_BATCH_MAX_N == MAX_N
    for k in (2, 3):
        small, large = dispatch.pool_batch_routes([0, 512, 513, 100, 5000, 1], k)
        assert small == [0, 1, 3, 5] and large == [2, 4]
    # K = 4: few large instances are faster through find_pool_all (measured crossover)
    small, large = dispatch.pool_batch_routes([0, 300, 301, 512, 100], 4)
    assert small == [0, 1, 4] and large == [2, 3]
    # a rerun is sized exactly from needed_out, unless the slices would exceed the budget
    assert dispatch.pool_batch_records(10, 8, 5000, budget=10 * 8 * 5000 * 8) == 5000
    assert dispatch.pool_batch_records(10, 8, 5001, budget=10 * 8 * 5000 * 8) is None
    assert dispatch.pool_batch_records(3, 1, 0) == 1


# ---- GPU ----------------------------------------------------------------------------------------------------------------
def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


def oracle_all(dem, dist, k, n_shards=8):
    parts, stats = [], {"evaluated": 0, "feasible": 0, "kept_per_shard": []}
    n = len(np.asarray(dem).reshape(-1, 5))
    for s in range(n_shards):
        plans, st = pool_ref.find(dem, dist, k, s, n_shards)
        parts.append(plans)
        stats["evaluated"] += st["evaluated"]
        stats["feasible"] += st["feasible"]
        stats["kept_per_shard"].append(st["kept"])
    merged = pool_ref.merge(parts, n, k)
    stats["kept"] = len(merged)
    return merged, stats


def check_batch(td, inst, dist, k, n_shards=8, loop=True, oracle=True):
    """find_pool_all_batch against the oracle and against find_pool_all, instance by instance"""
    res = td.find_pool_all_batch(inst, dist, k, n_shards)
    assert len(res) == len(inst)
    for i, (dem, r) in enumerate(zip(inst, res)):
        assert r is not None, i
        plans, stats = r
        if oracle:
            oplans, ost = oracle_all(dem, dist, k, n_shards)
            assert np.array_equal(plans, oplans), (i, len(dem), k, n_shards)
            assert stats == ost, (i, len(dem), k, n_shards)
        if loop:
            lplans, lst = td.find_pool_all(dem, dist, k, n_shards)
            assert _same(plans, lplans), (i, len(dem), k, n_shards)
            assert {q: lst[q] for q in ("evaluated", "feasible", "kept_per_shard", "kept")} == stats, (i, len(dem), k)
    return res


@pytest.mark.gpu
def test_golden_cases_in_one_batch(td):
    cases = load_golden("pool_small.json")
    for S in sorted({c["n_stands"] for c in cases}):
        group = [c for c in cases if c["n_stands"] == S]
        dist = g.stand_distances(S)
        inst = [np.array(c["demand"], dtype=np.int32) for c in group]
        for k in (2, 3, 4):
            res = check_batch(td, inst, dist, k)
            for c, (plans, _) in zip(group, res):
                if c["pool_size"] == k:
                    assert plans.tolist() == c["merged"], c["label"]


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3, 4])
def test_sizes_and_shard_counts(td, k):
    sizes = [0, 1, k - 1, k, 7, 8, 9, 60, 97, 200]
    inst = [g.pool_demand(n, seed=5 + n) for n in sizes]
    for n_shards in (1, 3, 8, 64):
        check_batch(td, inst, D50, k, n_shards)
    # the largest instances: the oracle takes seconds per instance at K = 4, so one pair of them, 8 shards
    big = [g.pool_demand(511, seed=3), g.pool_demand(512, seed=4)]
    res = check_batch(td, big + inst[:3], D50, k, 8)
    # the kernel itself at these sizes (find_pool_all_batch routes K = 4 above 300 customers through find_pool_all)
    from taxidispatcher_b200 import dispatch
    for (m, plans, stats, _), (rplans, rstats) in zip(dispatch._pool_batch_call(big, D50, k, 8, 1 << 20), res):
        assert m == len(rplans) and _same(plans, rplans) and stats == rstats


def _random_table_instances(k):
    rng = np.random.default_rng(40 + k)
    S = 23
    dist = rng.integers(0, 9, (S, S)).astype(np.int32)
    np.fill_diagonal(dist, 0)
    inst = []
    for n in (70, 33, 5, 120):
        inst.append(np.stack([np.arange(n), rng.integers(0, S, n), rng.integers(0, S, n), rng.integers(-1, 12, n),
                              rng.integers(-150, 120, n)], axis=1).astype(np.int32))
    return inst, dist


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3, 4])
def test_random_tables_negative_waits_and_losses(td, k):
    """asymmetric random tables, waits from -1 (pruned at the first pickup), losses from -150 % to 120 %"""
    inst, dist = _random_table_instances(k)
    for n_shards in (8, 3, 1):
        check_batch(td, inst, dist, k, n_shards)


@pytest.mark.gpu
def test_k4_non_metric_fuzz(td):
    """the table kinds of the K = 4 pruning-bound fuzz (one-way shortcuts, mostly zeros, wide asymmetric, constant rows,
    from == to trips), one batch per table"""
    rng = np.random.default_rng(20261018)
    for case in range(16):
        S = int(rng.integers(3, 30))
        kind = case % 4
        if kind == 0:
            dist = np.abs(np.arange(S)[:, None] - np.arange(S)[None, :]).astype(np.int32)
            for _ in range(S):
                dist[rng.integers(0, S), rng.integers(0, S)] = rng.integers(0, 3)
        elif kind == 1:
            dist = (rng.integers(0, 10, (S, S)) * (rng.random((S, S)) < 0.3)).astype(np.int32)
        elif kind == 2:
            dist = rng.integers(0, 200, (S, S)).astype(np.int32)
        else:
            dist = np.repeat(rng.integers(1, 12, (S, 1)), S, axis=1).astype(np.int32)
        np.fill_diagonal(dist, 0)
        scale = max(1, int(dist.max()))
        inst = []
        for _ in range(3):
            n = int(rng.integers(8, 56))
            fr = rng.integers(0, S, n)
            to = np.where(rng.random(n) < 0.1, fr, rng.integers(0, S, n))
            inst.append(np.stack([np.arange(n), fr, to, rng.integers(0, 3 * scale + 1, n), rng.integers(0, 150, n)],
                                 axis=1).astype(np.int32))
        check_batch(td, inst, dist, 4, int(rng.integers(1, 9)))


@pytest.mark.gpu
@pytest.mark.parametrize("k", [2, 3, 4])
def test_large_costs(td, k):
    """plan costs far above 255 and long waits"""
    rng = np.random.default_rng(90 + k)
    S = 17
    dist = rng.integers(40, 160, (S, S)).astype(np.int32)
    np.fill_diagonal(dist, 0)
    inst = [np.stack([np.arange(n), rng.integers(0, S, n), rng.integers(0, S, n), rng.integers(100, 400, n),
                      rng.integers(50, 400, n)], axis=1).astype(np.int32) for n in (60, 41)]
    for n_shards in (8, 2, 1):
        check_batch(td, inst, dist, k, n_shards)


@pytest.mark.gpu
def test_table_entries_at_the_limit_and_above(td):
    """entries of exactly 2^22 are exact in every pool size; one entry above it (or below 0) withdraws every instance"""
    rng = np.random.default_rng(7)
    S = 9
    dist = rng.integers(1, 1 << 22, (S, S)).astype(np.int32)
    dist[rng.integers(0, S, 6), rng.integers(0, S, 6)] = 1 << 22
    np.fill_diagonal(dist, 0)
    inst = [np.stack([np.arange(n), rng.integers(0, S, n), rng.integers(0, S, n), rng.integers(1 << 20, 1 << 24, n),
                      rng.integers(0, 300, n)], axis=1).astype(np.int32) for n in (26, 13)]
    for k in (2, 3, 4):
        check_batch(td, inst, dist, k, 1)
    for bad in ((1 << 22) + 1, -1):
        d = dist.copy()
        d[2, 5] = bad
        for k in (2, 4):
            assert td.find_pool_all_batch(inst + [g.pool_demand(5, n_stands=S)], d, k) == [None, None, None]


def _dev(a, dt=None):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).to(dtype=dt or torch.int32, device="cuda")


@pytest.mark.gpu
def test_ragged_poisoned_withdrawn_and_deterministic(td):
    import torch
    from taxidispatcher_b200 import dispatch
    k = 3
    inst = [g.pool_demand(n, seed=60 + n) for n in (37, 0, 120, 1, 64, 201, 2, 90)]
    res = check_batch(td, inst, D50, k, oracle=False)
    eng = dispatch.engine()
    # poisoned gaps: rows with stands far outside the table between the instances change nothing
    sizes = np.array([len(x) for x in inst], np.int32)
    offs = np.cumsum([0] + [s + 3 for s in sizes[:-1]]).astype(np.int64)
    rows = np.full((int(offs[-1] + sizes[-1] + 3), 5), 10 ** 6, np.int32)
    for x, o in zip(inst, offs):
        rows[o: o + len(x)] = x
    n_max = int(sizes.max())

    def run(dem, sz, of, rps=1 << 16):
        out = eng.pool_find_all_batch(_dev(dem), _dev(sz), _dev(of, torch.int64), n_max, _dev(D50), k, 8, rps)
        return [t.cpu().numpy() for t in out]

    plans, n_plans, ev, fe, kept, needed = run(rows, sizes, offs)
    for b, (p, st) in enumerate(res):
        assert n_plans[b] == len(p) and _same(plans[b, : len(p)], p) and (plans[b, len(p):] == -1).all()
        assert int(ev[b].sum()) == st["evaluated"] and int(fe[b].sum()) == st["feasible"]
        assert kept[b].tolist() == st["kept_per_shard"]
    # withdrawn instances next to valid ones: bad size, bad offset, a stand outside the table
    bad_sizes, bad_offs, bad_rows = sizes.copy(), offs.copy(), rows.copy()
    bad_sizes[1] = n_max + 1
    bad_sizes[6] = -1
    bad_offs[3] = -1
    bad_rows[offs[4] + 2, 2] = 50
    plans, n_plans, ev, fe, kept, needed = run(bad_rows, bad_sizes, bad_offs)
    for b, (p, st) in enumerate(res):
        if b in (1, 3, 4, 6):
            assert n_plans[b] == -1 and (plans[b] == -1).all() and (kept[b] == 0).all() and (ev[b] == 0).all()
        else:
            assert n_plans[b] == len(p) and _same(plans[b, : len(p)], p)
            assert int(ev[b].sum()) == st["evaluated"] and kept[b].tolist() == st["kept_per_shard"]
    assert td.find_pool_all_batch([inst[0], bad_rows[offs[4]: offs[4] + sizes[4]]], D50, k)[1] is None
    # the same instance at other positions, next to other neighbours and under a larger n_max: identical results
    x = inst[5]
    big = g.pool_demand(400, seed=9)
    for batch in ([x], [big, x], [inst[0], inst[2], x, big]):
        out = td.find_pool_all_batch(batch, D50, k)
        p, st = out[[i for i, y in enumerate(batch) if y is x][0]]
        assert _same(p, res[5][0]) and st == res[5][1]
    # repeated calls are byte-identical
    again = td.find_pool_all_batch(inst, D50, k)
    assert all(_same(a[0], b[0]) and a[1] == b[1] for a, b in zip(again, res))


@pytest.mark.gpu
def test_record_slice_overflow(td):
    import torch
    from taxidispatcher_b200 import dispatch
    eng = dispatch.engine()
    k = 4
    inst = [g.pool_demand(n, seed=70 + n) for n in (30, 150, 60)]
    res = check_batch(td, inst, D50, k, oracle=False)
    demand, sizes, offsets, n_max, d = dispatch.pack_pool_batch(inst, D50)
    # a slice that fits the two small instances but not the large one
    small_need = []
    for rps in (1 << 20, None):
        if rps is None:
            rps = max(small_need[0], small_need[2])
        plans, n_plans, ev, fe, kept, needed = [t.cpu().numpy() for t in
                                                eng.pool_find_all_batch(demand, sizes, offsets, n_max, d, k, 8, rps)]
        small_need = [int(v) for v in needed]
    assert small_need[1] > rps
    assert n_plans[1] == -2 and (plans[1] == -1).all() and (kept[1] == -1).any()
    for b in (0, 2):
        p, st = res[b]
        assert n_plans[b] == len(p) and _same(plans[b, : len(p)], p) and kept[b].tolist() == st["kept_per_shard"]
    # the counters of the overflowing instance are still exact, and a rerun sized from needed_out fits
    assert int(ev[1].sum()) == res[1][1]["evaluated"] and int(fe[1].sum()) == res[1][1]["feasible"]
    plans, n_plans = [t.cpu().numpy() for t in eng.pool_find_all_batch(demand, sizes, offsets, n_max, d, k, 8,
                                                                        int(needed[1]))[:2]]
    assert n_plans[1] == len(res[1][0]) and _same(plans[1, : n_plans[1]], res[1][0])
    # find_pool_all_batch reruns an overflowing instance and returns the right answer
    dispatch._POOL_BATCH_RPS.clear()
    old = dispatch.POOL_BATCH_FIRST_RECORDS
    dispatch.POOL_BATCH_FIRST_RECORDS = 8
    try:
        out = td.find_pool_all_batch(inst, D50, k)
    finally:
        dispatch.POOL_BATCH_FIRST_RECORDS = old
    assert all(_same(a[0], b[0]) and a[1] == b[1] for a, b in zip(out, res))


@pytest.mark.gpu
def test_batch_of_1000_in_one_launch(td):
    from taxidispatcher_b200 import _lib
    lib = _lib.lib()
    k = 4
    inst = [g.pool_demand(100, seed=s) for s in range(1000)]
    td.find_pool_all_batch(inst, D50, k)                               # sizes the record slices of this shape
    counts = []
    for batch in (inst[:1], inst):
        before = lib.td_launch_count()
        res = td.find_pool_all_batch(batch, D50, k)
        counts.append(lib.td_launch_count() - before)
    assert counts == [1, 1]
    for i in range(0, 1000, 97):
        oplans, ost = oracle_all(inst[i], D50, k)
        assert np.array_equal(res[i][0], oplans) and res[i][1] == ost, i


@pytest.mark.gpu
def test_sizes_on_both_sides_of_the_limit(td):
    inst = [g.pool_demand(n, seed=80 + n) for n in (100, 600, 513, 512, 30)]
    check_batch(td, inst, D50, 2)
    check_batch(td, [inst[4], inst[2], inst[0]], D50, 3, oracle=False)
