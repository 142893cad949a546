"""The two record formats of the pool finder (td_pool.cu): 8-byte keys when the input bounds every plan cost below
2^(64 - 4 cb - 5), 16-byte PoolRec otherwise.  Every case first restates from the inputs which format it takes (the rule of
key64_fits: max(W, 0) + max(thr, 0) against 2^(64 - 4 cb - 5), thr in IEEE fp64 as in oracle/pool_ref) and asserts it, then
compares plans and the evaluated / feasible counts with the C oracle, byte for byte.

Most inputs of tests/test_pool_select.py fit the bound, so they run on 8-byte keys; the cases below that raise one
customer's loss keep the 16-byte path (and its two-level keys) under the band knobs and cost windows."""
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

from oracle import gen_inputs as g
from oracle import pool_ref
from test_pool_select import (BAND0, GROWTH, KNOBS, assert_same, band_sizes, family_case, key_bits, materialised_costs,
                              set_knobs, single_key)

gpu = pytest.mark.gpu


# ---- the restated decision ---------------------------------------------------------------------------------------------
def detour_thr(dem, dist):
    """pool_detour_thr: floor(D(F, T) * (1 + L / 100.0)) in fp64, clamped to int32"""
    d = dist[dem[:, 1], dem[:, 2]].astype(np.float64)
    lim = np.floor(d * (1.0 + dem[:, 4].astype(np.float64) / 100.0))
    return np.clip(lim, -2147483648.0, 2147483647.0).astype(np.int64)


def cost_bound(dem, dist):
    return int(max(int(dem[:, 3].max()), 0)) + int(max(int(detour_thr(dem, dist).max()), 0))


def key64(dem, dist):
    cost_bits = 64 - 4 * key_bits(len(dem)) - 5
    return cost_bits >= 1 and cost_bound(dem, dist) < (1 << cost_bits)


def test_restated_rule():
    # n = 4097: 7 cost bits, n = 8193: 3, n = 722: 19
    assert [64 - 4 * key_bits(n) - 5 for n in (722, 4096, 4097, 8192, 8193, 16384)] == [19, 11, 7, 7, 3, 3]
    dem, dist = g.pool_demand(), g.stand_distances(50)
    assert cost_bound(dem, dist) <= 3 + 49 and key64(dem, dist)      # config 3: W = 3, thr <= floor(49 * 1.01)
    assert not key64(*raised_loss(dem, dist, 1_100_000))
    # the bound holds on the oracle's plans: no feasible plan costs more than max W + max thr
    for k in (2, 3, 4):
        d2, t2 = family_case(k, "table", True, 100 * k + 11)
        recs, _ = pool_ref.find(d2, t2, k, 0, 1, dedup=False)
        assert len(recs) and int(recs[:, 8].max()) <= cost_bound(d2, t2)


def raised_loss(dem, dist, loss):
    """The same input with the customer of the longest trip given `loss` percent."""
    dem = dem.copy()
    c = int(np.argmax(dist[dem[:, 1], dem[:, 2]]))
    dem[c, 4] = loss
    return dem, dist


def oracle_shards(dem, dist, k, n_shards, shards=None):
    """pool_ref.find per logical shard, the shards in threads (ctypes releases the GIL)"""
    shards = range(n_shards) if shards is None else shards
    with ThreadPoolExecutor(max_workers=8) as ex:
        return list(ex.map(lambda s: pool_ref.find(dem, dist, k, s, n_shards), shards))


# ---- config 3 on both formats ------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("fmt", ["key64", "rec16"])
def test_config3_both_formats(td, monkeypatch, fmt):
    """The golden 722-customer input (costs at most 52, 19 cost bits) takes the 8-byte records; one customer's loss at
    1.1 x 10^6 % puts its thr past 2^19 and the same plans through PoolRec.  find_pool_block (all 8 shards in one
    selection launch) and find_pool_all (cost windows, then the asynchronous headed path, then the captured graph)."""
    dem, dist = g.pool_demand(), g.stand_distances(50)
    if fmt == "rec16":
        dem, dist = raised_loss(dem, dist, 1_100_000)
    assert key64(dem, dist) == (fmt == "key64")
    want = oracle_shards(dem, dist, 4, 8)
    got = td.find_pool_block(dem, dist, 4, 0, 8, 8)
    for s in range(8):
        assert_same(got[s][0], got[s][1], want[s][0], want[s][1], s)
    merged = pool_ref.merge([w[0] for w in want], len(dem), 4)
    ev, fe = sum(w[1]["evaluated"] for w in want), sum(w[1]["feasible"] for w in want)
    monkeypatch.setenv("TD_POOL_GRAPH", "1")
    for rep in range(3):
        plans, st = td.find_pool_all(dem, dist, 4, 8)
        assert np.array_equal(plans, merged), rep
        assert (st["evaluated"], st["feasible"]) == (ev, fe), rep
        assert st["kept_per_shard"] == [len(w[0]) for w in want], rep


# ---- the bound's edge --------------------------------------------------------------------------------------------------
def bound_edge_case(n, k, over, seed):
    """Pickup groups of k + 1 .. k + 3 customers on their own stands (waits 0-1, other pickup stands 50 away); in every
    group some customers ride to stand X and the others to stand Z, D(s, X) = D(s, Z) = base, D(X, Z) = D(Z, X) = 1, so a
    plan costs base (one destination) or base + 1 (both).  The losses put every thr in [base + 1, limit - 2]: with the
    waits the bound is limit - 1, just inside the cost field.  over: one customer's thr becomes limit - 1, the bound
    limit, and the call takes PoolRec."""
    limit = 1 << (64 - 4 * key_bits(n) - 5)
    base = limit - 28 if limit > 64 else limit - 3            # 100 at n = 4097, 5 at n = 8193
    rng = np.random.default_rng(seed)
    sizes = []
    while sum(sizes) < n:
        sizes.append(int(rng.integers(k + 1, k + 4)))
    sizes[-1] -= sum(sizes) - n
    if sizes[-1] < 1:
        sizes.pop()
        sizes[-1] += n - sum(sizes)
    G = len(sizes)
    X, Z = G, G + 1
    dist = np.full((G + 2, G + 2), 50, np.int32)
    dist[:G, X] = dist[:G, Z] = base
    dist[X, Z] = dist[Z, X] = 1
    np.fill_diagonal(dist, 0)
    fr = np.repeat(np.arange(G), sizes)
    to = np.where(rng.random(n) < 0.5, X, Z)
    perm = rng.permutation(n)
    fr, to = fr[perm], to[perm]
    waits = rng.integers(0, 2, n)
    waits[0] = 1
    # thr = floor(base * (1 + L / 100)) in fp64, as pool_detour_thr computes it
    thr_of = {L: int(np.floor(base * (1.0 + L / 100.0))) for L in range(0, 1000)}
    inside = [L for L, t in thr_of.items() if base + 1 <= t <= limit - 2]
    losses = rng.choice(inside, n)
    losses[1] = max(inside, key=lambda L: thr_of[L])
    dem = np.stack([np.arange(n), fr, to, waits, losses], axis=1).astype(np.int32)
    if over:
        dem[1, 4] = min(L for L, t in thr_of.items() if t == limit - 1)
    return dem, dist


EDGE = [(n, k, over) for n in (4097, 8193) for k in (2, 3, 4) for over in (False, True)]


@gpu
@pytest.mark.parametrize("n,k,over", EDGE)
def test_bound_edge(td, n, k, over):
    dem, dist = bound_edge_case(n, k, over, seed=n + 10 * k + int(over))
    limit = 1 << (64 - 4 * key_bits(n) - 5)
    assert cost_bound(dem, dist) == limit - 1 + int(over)
    assert key64(dem, dist) == (not over)
    want, wst = pool_ref.find(dem, dist, k, 0, 1)
    costs = set(want[:, 8].tolist())
    assert len(want) > 100 and len(costs) == 2                # plans of one and of two destinations
    got, gst = td.find_pool(dem, dist, k, 0, 1)
    assert_same(got, gst, want, wst, (n, k, over))


# ---- bands and grid knobs on both formats ------------------------------------------------------------------------------
def family_input(k, kind, big, seed, fmt):
    dem, dist = family_case(k, kind, big, seed)
    if fmt == "rec16":                  # the largest loss: thr past 2^27 (n = 220) or clamped to 2^31 - 1 (n = 70, 100)
        dem, dist = raised_loss(dem, dist, 2**31 - 1)
    assert key64(dem, dist) == (fmt == "key64")
    return dem, dist


# (4, fuzz): 64 customers leave 35 cost bits, more than any int32 wait plus thr -- always 8-byte keys
FAMILIES = [(2, "table", False, f) for f in ("key64", "rec16")] + [(3, "table", True, f) for f in ("key64", "rec16")] + \
           [(4, "table", True, f) for f in ("key64", "rec16")] + [(4, "fuzz", False, "key64")]
FEW_KNOBS = [(1, 1, None), (16, 2, 1), (256, 1, 1)]


@gpu
@pytest.mark.parametrize("k,kind,big,fmt", FAMILIES)
def test_bands_one_shard(td, monkeypatch, k, kind, big, fmt):
    """find_pool with TD_SEL_BAND0 / TD_SEL_GROWTH / TD_SEL_PER_SM: at least 4 non-empty bands; rec16 with costs past 255
    runs two-level keys."""
    dem, dist = family_input(k, kind, big, 100 * k + 11, fmt)
    want, wst = pool_ref.find(dem, dist, k, 0, 1)
    costs = [materialised_costs(dem, dist, k, 0, 1)]
    if fmt == "rec16" and big:
        assert not single_key(len(dem), costs)
    for band0, growth, per_sm in KNOBS:
        assert np.count_nonzero(band_sizes(costs, band0, growth)) >= 4
        set_knobs(monkeypatch, band0, growth, per_sm)
        got, gst = td.find_pool(dem, dist, k, 0, 1)
        assert_same(got, gst, want, wst, (band0, growth, per_sm))


@gpu
@pytest.mark.parametrize("k,kind,big,fmt", FAMILIES)
def test_bands_64_ragged_slots(td, monkeypatch, k, kind, big, fmt):
    """find_pool_block with 64 logical shards in one selection launch and with a ragged block (37 shards, 30 of them)."""
    dem, dist = family_input(k, kind, big, 700 + 10 * k + int(big), fmt)
    for n_shards, begin, count in ((64, 0, 64), (37, 5, 30)):
        want = oracle_shards(dem, dist, k, n_shards, range(begin, begin + count))
        costs = [materialised_costs(dem, dist, k, s, n_shards) for s in range(begin, begin + count)]
        for band0, growth, per_sm in FEW_KNOBS:
            if band0 == 256:
                continue
            assert np.count_nonzero(band_sizes(costs, band0, growth)) >= 4
            set_knobs(monkeypatch, band0, growth, per_sm)
            got = td.find_pool_block(dem, dist, k, begin, count, n_shards)
            for s in range(count):
                assert_same(got[s][0], got[s][1], want[s][0], want[s][1], (n_shards, begin + s, band0, growth, per_sm))


# ---- cost windows ------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("fmt", ["key64", "rec16"])
def test_cost_windows(td, monkeypatch, fmt):
    """A record list far below the feasible count: several enumeration passes and selection launches (cost windows), on
    the 8-byte records and on PoolRec, with the default bands and with the band knobs."""
    import torch
    eng = td.engine()
    rng = np.random.default_rng(2601)
    n, k, S = 2600, 2, 80
    dist = (np.abs(np.arange(S)[:, None] - np.arange(S)[None, :]) * 3 + rng.integers(0, 3, (S, S))).astype(np.int32)
    np.fill_diagonal(dist, 0)
    dem = np.stack([np.arange(n), rng.integers(0, S, n), rng.integers(0, S, n), rng.integers(150, 300, n),
                    rng.integers(100, 300, n)], axis=1).astype(np.int32)
    if fmt == "rec16":
        dem, dist = raised_loss(dem, dist, 1_000_000)
    assert key64(dem, dist) == (fmt == "key64")
    want, wst = pool_ref.find(dem, dist, k, 0, 1)
    assert wst["feasible"] > 40 * 100_000
    dd, ds = torch.from_numpy(dem).cuda(), torch.from_numpy(dist).cuda()
    for band0, growth, per_sm in ((BAND0, GROWTH, None), (16, 2, 1)):
        set_knobs(monkeypatch, band0, growth, per_sm)
        out, cnt, st = eng.pool_find(dd, ds, k, 0, 1, max_feasible=100_000)
        assert st.passes >= 4, st.passes
        got = out[: int(cnt.item())].cpu().numpy()
        assert_same(got, {"evaluated": st.evaluated, "feasible": st.feasible, "kept": st.kept}, want, wst,
                    (band0, growth, per_sm))
