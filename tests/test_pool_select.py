"""Pool selection (pool_select_kernel) and merge (pool_merge_kernel) paths that the golden inputs never reach, against the
C oracle, byte for byte: later cost bands, empty middle bands and the open-ended last band; two-level keys together with
bands and cost windows; the single-key limit at every key width; the merge's general path; out-of-range customers in a
caller's merge rows.

Every test first restates, from the oracle, the path it claims to reach (number of non-empty bands, single or two-level
keys, rows beyond the merge's shared-memory capacity) and asserts it, so that a green run says what it covered.  The
selection reads TD_SEL_BAND0 / TD_SEL_GROWTH / TD_SEL_PER_SM at every call; small inputs reach many bands through them."""
import numpy as np
import pytest

from oracle import pool_ref

gpu = pytest.mark.gpu

# mirrors of td_pool.cu's constants
BUCKETS = 256          # kBuckets: cost histogram, last bucket open-ended
MAX_BANDS = 8          # kMaxBands
BAND0, GROWTH = 65536, 4
MERGE_FAST = 8192      # kMergeFast
REC_W = pool_ref.REC_W


# ---- restated decisions of the kernels ---------------------------------------------------------------------------------
def materialised_costs(dem, dist, k, shard, n_shards):
    """Costs of the records the enumeration materialises for one shard: every pickup tuple with a feasible drop-off
    order keeps its cheapest one (from the oracle's dedup=False output, which lists every feasible order)."""
    recs, _ = pool_ref.find(dem, dist, k, shard, n_shards, dedup=False)
    if len(recs) == 0:
        return np.zeros(0, np.int64)
    key = np.zeros(len(recs), np.int64)
    for q in range(k):
        key = (key << 14) | recs[:, q].astype(np.int64)
    cost = recs[:, 8].astype(np.int64)
    order = np.lexsort((cost, key))
    ks = key[order]
    first = np.ones(len(ks), bool)
    first[1:] = ks[1:] != ks[:-1]
    return cost[order][first]


def band_sizes(costs_per_slot, band0=BAND0, growth=GROWTH):
    """pool_select_kernel's band cut: per slot, the cumulative histogram of min(cost, 255) against targets that start at
    band0 and grow by `growth` x the running total; at most MAX_BANDS bands, the last one open-ended.  Returns the
    records of every band summed over the slots (the band-partitioned list)."""
    sizes = np.zeros(MAX_BANDS, np.int64)
    for costs in costs_per_slot:
        hist = np.bincount(np.minimum(np.asarray(costs, np.int64), BUCKETS - 1), minlength=BUCKETS)
        cum, target, in_band, band = 0, band0, 0, 0
        for bkt in range(BUCKETS):
            cum += int(hist[bkt])
            in_band += int(hist[bkt])
            if band < MAX_BANDS - 1 and bkt < BUCKETS - 1 and cum >= target:
                sizes[band] += in_band
                band, in_band, target = band + 1, 0, cum * growth
        sizes[band] += in_band
    return sizes


def key_bits(n):
    """cb: bits per customer in the repacked rank"""
    cb = 1
    while (1 << cb) < n:
        cb += 1
    return cb


def single_key_limit(n):
    """Costs below this fit beside the repacked rank in ONE 64-bit key (0: never)."""
    cost_bits = 64 - 4 * key_bits(n) - 5
    if cost_bits < 1:
        return 0
    return BUCKETS - 1 if cost_bits >= 31 else min(BUCKETS - 1, 1 << cost_bits)


def single_key(n, costs_per_slot):
    lim = single_key_limit(n)
    return all(len(c) == 0 or int(np.max(c)) < lim for c in costs_per_slot)


def fast_cap(n):
    """Rows the merge handles in shared memory (launch_merge)."""
    if n > 16384:
        return 0
    fc = MERGE_FAST
    while fc >= 256 and fc * 21 + n * 4 + 16 > 200 * 1024:
        fc >>= 1
    return fc if fc >= 256 else 0


def test_restated_limits():
    assert [single_key_limit(n) for n in (60, 4096, 4097, 8192, 8193, 16384)] == [255, 255, 128, 128, 8, 8]
    assert [fast_cap(n) for n in (0, 722, 8188, 8189, 10000, 16384)] == [8192, 8192, 8192, 4096, 4096, 4096]
    # growth 1: every bucket after the first band closes a band, empty ones too; the last band is open-ended
    assert band_sizes([[0, 0, 2, 5, 5, 9, 300]], band0=1, growth=1).tolist() == [2, 0, 1, 0, 0, 2, 0, 2]
    assert band_sizes([[3] * 10 + [7] * 30], band0=16, growth=2).tolist() == [40, 0, 0, 0, 0, 0, 0, 0]


# ---- inputs ------------------------------------------------------------------------------------------------------------
def random_table_case(k, seed, n=70, big=False):
    """test_pool_random_tables_vs_oracle's family (asymmetric random table, ragged waits / losses); big=True adds
    expensive legs so that plan costs reach past 255 (the open-ended bucket: two-level keys)."""
    rng = np.random.default_rng(seed)
    S = 23
    dist = rng.integers(0, 9, (S, S)).astype(np.int32)
    if big:
        dist += (rng.random((S, S)) < 0.35) * rng.integers(60, 260, (S, S)).astype(np.int32)
    np.fill_diagonal(dist, 0)
    waits = rng.integers(-1, 12, n)
    losses = rng.integers(0, 120, n) if not big else rng.integers(50, 400, n)
    dem = np.stack([np.arange(n), rng.integers(0, S, n), rng.integers(0, S, n), waits, losses], axis=1).astype(np.int32)
    return dem, dist


def k4_fuzz_case(seed):
    """test_pool_k4_pruning_bounds_fuzz's family: tables that break the triangle inequality in different ways"""
    rng = np.random.default_rng(seed)
    S = int(rng.integers(8, 30))
    n = 64
    kind = seed % 4
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
    fr = rng.integers(0, S, n)
    to = np.where(rng.random(n) < 0.1, fr, rng.integers(0, S, n))
    scale = max(1, int(dist.max()))
    dem = np.stack([np.arange(n), fr, to, rng.integers(0, 3 * scale + 1, n), rng.integers(0, 150, n)], axis=1).astype(np.int32)
    return dem, dist


FAMILIES = [(2, "table", False), (2, "table", True), (3, "table", False), (3, "table", True), (4, "table", True),
            (4, "fuzz", False)]


def family_case(k, kind, big, seed, even=False):
    """even: distances and waits doubled -- the same feasible plans at twice the cost, so every odd cost bucket is empty
    and growth 1 cuts empty bands between non-empty ones"""
    dem, dist = k4_fuzz_case(seed) if kind == "fuzz" else random_table_case(k, seed, n={2: 220, 3: 100}.get(k, 70), big=big)
    if even:
        dem[:, 3] *= 2
        dist = dist * 2
    return dem, dist


KNOBS = [(b0, gr, per_sm) for b0 in (1, 16, 256) for gr in (1, 2) for per_sm in (None, 1)]


def set_knobs(monkeypatch, band0, growth, per_sm):
    monkeypatch.setenv("TD_POOL_GRAPH", "0")
    monkeypatch.setenv("TD_SEL_BAND0", str(band0))
    monkeypatch.setenv("TD_SEL_GROWTH", str(growth))
    if per_sm is None:
        monkeypatch.delenv("TD_SEL_PER_SM", raising=False)
    else:
        monkeypatch.setenv("TD_SEL_PER_SM", str(per_sm))


def assert_same(got, gst, want, wst, where):
    assert {q: gst[q] for q in wst} == wst, where
    assert np.array_equal(got, want), where


# ---- 2. many bands on small inputs -------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k,kind,big", FAMILIES)
def test_select_many_bands_one_shard(td, monkeypatch, k, kind, big):
    """find_pool (one logical shard per call) with the band knobs: at least 4 non-empty bands every time, empty middle
    bands with growth 1, and (big) costs past 255 in the open-ended last band under two-level keys."""
    reached_empty_middle = reached_two_level = False
    for seed in (11, 12):
        dem, dist = family_case(k, kind, big, 100 * k + seed, even=seed == 12)
        n = len(dem)
        for n_shards, shard in ((1, 0), (3, 2)):
            want, wst = pool_ref.find(dem, dist, k, shard, n_shards)
            costs = [materialised_costs(dem, dist, k, shard, n_shards)]
            two_level = not single_key(n, costs)
            assert two_level == (big and int(costs[0].max()) >= 255)
            reached_two_level |= two_level
            for band0, growth, per_sm in KNOBS:
                sizes = band_sizes(costs, band0, growth)
                assert np.count_nonzero(sizes) >= 4, (sizes, band0, growth)
                nz = np.nonzero(sizes)[0]
                reached_empty_middle |= bool((sizes[nz[0]: nz[-1]] == 0).any())
                set_knobs(monkeypatch, band0, growth, per_sm)
                got, gst = td.find_pool(dem, dist, k, shard, n_shards)
                assert_same(got, gst, want, wst, (seed, n_shards, band0, growth, per_sm))
    assert reached_empty_middle
    assert reached_two_level == big


@gpu
@pytest.mark.parametrize("k,kind,big", FAMILIES)
def test_select_many_bands_many_slots(td, monkeypatch, k, kind, big):
    """find_pool_block: up to 64 logical shards in one selection launch with ragged n_shards (each slot has its own band
    bounds; the band segments hold the records of every slot; p0 / step through slot_of's reciprocal)."""
    dem, dist = family_case(k, kind, big, 700 + 10 * k + int(big))
    n = len(dem)
    for n_shards, begin, count in ((64, 0, 64), (37, 5, 30), (3, 1, 2)):
        want = [pool_ref.find(dem, dist, k, s, n_shards) for s in range(begin, begin + count)]
        costs = [materialised_costs(dem, dist, k, s, n_shards) for s in range(begin, begin + count)]
        assert single_key(n, costs) == (not big or max(int(c.max()) for c in costs if len(c)) < 255)
        for band0, growth, per_sm in KNOBS:
            if band0 == 256 and count > 2:
                continue                                  # a few hundred records per slot: one or two bands of 256
            sizes = band_sizes(costs, band0, growth)
            assert np.count_nonzero(sizes) >= 4, (sizes, n_shards, band0, growth)
            set_knobs(monkeypatch, band0, growth, per_sm)
            got = td.find_pool_block(dem, dist, k, begin, count, n_shards)
            for s in range(count):
                assert_same(got[s][0], got[s][1], want[s][0], want[s][1], (n_shards, begin + s, band0, growth, per_sm))


# ---- 3. cost windows with bands ----------------------------------------------------------------------------------------
@gpu
def test_select_cost_windows_with_bands(td, monkeypatch):
    """A record list far below the feasible count sends the call through cost windows: the first selection launch takes
    the cheapest plans, the later ones (first_pass = 0) start from the customers the earlier windows left free.  Combined
    with the band knobs, and with costs on both sides of 255 (the windows above 255 run on two-level keys).  The record
    list holds max_feasible plus a fixed slack of 1.2 M records, so the input has millions of materialised pairs; trips
    of every length on a line of stands make each window kill only the customers with short trips."""
    import torch
    eng = td.engine()
    rng = np.random.default_rng(2600)
    n, k, S = 2600, 2, 80
    dist = (np.abs(np.arange(S)[:, None] - np.arange(S)[None, :]) * 3 + rng.integers(0, 3, (S, S))).astype(np.int32)
    np.fill_diagonal(dist, 0)
    dem = np.stack([np.arange(n), rng.integers(0, S, n), rng.integers(0, S, n), rng.integers(150, 300, n),
                    rng.integers(100, 300, n)], axis=1).astype(np.int32)
    want, wst = pool_ref.find(dem, dist, k, 0, 1)
    costs = materialised_costs(dem, dist, k, 0, 1)
    assert len(costs) > 4_000_000 and int(costs.min()) < 255 <= int(costs.max())
    assert int(want[:, 8].max()) >= 255                   # the last window keeps plans on two-level keys
    dd, ds = torch.from_numpy(dem).cuda(), torch.from_numpy(dist).cuda()
    for band0, growth, per_sm in ((BAND0, GROWTH, None), (1, 1, 1), (16, 2, None), (256, 1, None)):
        set_knobs(monkeypatch, band0, growth, per_sm)
        out, cnt, st = eng.pool_find(dd, ds, k, 0, 1, max_feasible=100_000)
        assert st.passes >= 4, st.passes                  # overflowing passes + later windows
        got = out[: int(cnt.item())].cpu().numpy()
        assert_same(got, {"evaluated": st.evaluated, "feasible": st.feasible, "kept": st.kept}, want, wst,
                    (band0, growth, per_sm))


# ---- 4. key-width edges ------------------------------------------------------------------------------------------------
def key_edge_case(n, k, top, seed):
    """Pickup groups of k + 1 .. k + 3 customers on their own stands (waits 0-1, other pickup stands 50 away); in every
    group k or more customers ride to stand X and the others to stand Z, with D(s, X) = D(s, Z) = top - 1 and
    D(X, Z) = D(Z, X) = 1: a plan all-X or all-Z costs top - 1, a mixed one top.  The cheapest conflicting plans thus
    cost top - 1 and top; with top at the single-key limit the costlier one needs two-level keys."""
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
    S = G + 2
    dist = np.full((S, S), 50, np.int32)
    dist[:G, X] = dist[:G, Z] = top - 1
    dist[X, Z] = dist[Z, X] = 1
    np.fill_diagonal(dist, 0)
    fr = np.repeat(np.arange(G), sizes)
    to = np.empty(n, np.int64)
    at = 0
    for sz in sizes:
        nx = int(rng.integers(k, sz + 1)) if sz > k else sz
        to[at: at + sz] = rng.permutation([X] * nx + [Z] * (sz - nx))
        at += sz
    perm = rng.permutation(n)                             # groups interleave in customer order (and so in rank)
    fr, to = fr[perm], to[perm]
    dem = np.stack([np.arange(n), fr, to, rng.integers(0, 2, n), rng.integers(20, 100, n)], axis=1).astype(np.int32)
    return dem, dist


EDGES = [(n, k, top) for n in (4096, 4097, 8192, 8193, 16384) for k in (2, 3)
         for top in (single_key_limit(n) - 1, single_key_limit(n))]


@gpu
@pytest.mark.parametrize("n,k,top", EDGES)
def test_select_key_width_edges(td, n, k, top):
    dem, dist = key_edge_case(n, k, top, seed=n + 10 * k + top)
    shardings = ((1, 0), (2, 0), (2, 1)) if n == 16384 else ((1, 0),)
    for n_shards, shard in shardings:
        costs = materialised_costs(dem, dist, k, shard, n_shards)
        assert int(costs.max()) == top and int(costs.min()) == top - 1
        assert single_key(n, [costs]) == (top < single_key_limit(n))
        want, wst = pool_ref.find(dem, dist, k, shard, n_shards)
        assert {top - 1, top} <= set(want[:, 8].tolist())
        got, gst = td.find_pool(dem, dist, k, shard, n_shards)
        assert_same(got, gst, want, wst, (n_shards, shard))


@gpu
@pytest.mark.parametrize("n", [4097, 8193])
def test_pool_pairs_key_width_edges(td, n):
    """td_pool_pairs ranks all n^2 ordered pairs: at n = 4097 / 8193 the packed key has 7 / 3 cost bits.  The same stand
    layout as above with accept_all=False: pairs across groups fail the detour test, pairs inside cost limit - 1
    (same destination) or limit (mixed), so two-level keys decide the conflicts."""
    lim = single_key_limit(n)
    dem, dist = key_edge_case(n, 2, lim, seed=n)
    frm, to = dem[:, 1].copy(), dem[:, 2].copy()
    want = pool_ref.pairs(frm, to, dist, accept_all=False, max_loss=1.3)
    assert {lim - 1, lim} <= set(want[:, 3].tolist())     # candidates past the single-key limit: two-level keys
    got = td.find_pool_pairs(frm, to, dist, accept_all=False, max_loss=1.3)
    assert np.array_equal(got, want)


# ---- 5. the merge's general path ---------------------------------------------------------------------------------------
def synthetic_rows(rng, m, n, k, sort_runs, n_slots):
    """m rows of k distinct customers with costs 0..5 (many ties), cut into n_slots runs; sort_runs: every run ascends in
    cost (what pool_emit produces), else arbitrary order."""
    c = rng.integers(0, n, (m, k))
    while True:                                           # redraw rows that repeat a customer
        s = np.sort(c, axis=1)
        dup = (s[:, 1:] == s[:, :-1]).any(axis=1)
        if not dup.any():
            break
        c[dup] = rng.integers(0, n, (int(dup.sum()), k))
    rows = np.zeros((m, REC_W), np.int32)
    rows[:, :k] = c
    rows[:, 4: 4 + k] = c[:, ::-1]
    rows[:, 8] = rng.integers(0, 6, m)
    cuts = np.sort(rng.choice(np.arange(1, m), n_slots - 1, replace=False)) if n_slots > 1 else []
    runs = np.split(rows, cuts)
    if sort_runs:
        runs = [r[np.argsort(r[:, 8], kind="stable")] for r in runs]
    return runs


def padded(runs):
    cap = max(len(r) for r in runs)
    slots = np.full((len(runs), cap, REC_W), -7, np.int32)
    for s, r in enumerate(runs):
        slots[s, : len(r)] = r
    return slots, np.array([len(r) for r in runs], np.int32)


MERGE_CASES = [(k, n, extra) for k in (2, 3, 4) for n in (6000, 12000) for extra in (0, 1, 20000)]


@gpu
@pytest.mark.parametrize("k,n,extra", MERGE_CASES)
def test_merge_general_path_vs_oracle(td, k, n, extra):
    """m = fast_cap, fast_cap + 1 (the first row of the general path) and ~20 000 rows, on both sides of n = 8188 (fast_cap
    8192 / 4096), as one run (td_pool_merge) and as <= 64 / > 64 padded slots, sorted and unsorted runs."""
    import torch
    eng = td.engine()
    fc = fast_cap(n)
    m = 20000 if extra == 20000 else fc + extra
    assert (m > fc) == (extra > 0)
    rng = np.random.default_rng(k * 100000 + n + extra)
    for n_slots in (1, 40, 90):
        for sort_runs in (True, False):
            runs = synthetic_rows(rng, m, n, k, sort_runs, n_slots)
            want = pool_ref.merge(runs, n, k)
            if n_slots == 1:
                got = td.pool_merge(runs, n, k)
            else:
                slots, counts = padded(runs)
                merged, cnt = eng.pool_merge_padded(torch.from_numpy(slots).cuda(), torch.from_numpy(counts).cuda(), None, n, k)
                got = merged[: int(cnt.item())].cpu().numpy()
            assert np.array_equal(got, want), (n_slots, sort_runs)


@gpu
def test_find_pool_all_general_merge_path(td, monkeypatch):
    """find_pool_all end to end at n = 10 000 with more survivors than the merge's shared-memory capacity (4096 rows
    above n = 8188): the cost-window path (padded merge) and the asynchronous headed path (headed merge) both equal the
    oracle's shard-by-shard results merged by the restated findpool merge."""
    monkeypatch.setenv("TD_POOL_GRAPH", "0")
    n, k, n_shards = 10000, 2, 8
    rng = np.random.default_rng(10000)
    G = 4000
    fr = rng.integers(0, G, n)
    to = G + rng.integers(0, 3, n)
    S = G + 3
    dist = np.full((S, S), 9, np.int32)
    dist[:G, G:] = rng.integers(3, 8, (G, 3))
    dist[G:, G:] = rng.integers(0, 3, (3, 3))
    np.fill_diagonal(dist, 0)
    dem = np.stack([np.arange(n), fr, to, rng.integers(0, 2, n), rng.integers(30, 150, n)], axis=1).astype(np.int32)
    shards = [pool_ref.find(dem, dist, k, s, n_shards)[0] for s in range(n_shards)]
    survivors = sum(len(p) for p in shards)
    assert survivors > fast_cap(n) == 4096
    want = pool_ref.merge(shards, n, k)
    for rep in range(2):                                  # 0: cost-window path, 1: asynchronous headed blocks
        got, st = td.find_pool_all(dem, dist, k, n_shards)
        assert st["kept_per_shard"] == [len(p) for p in shards]
        assert np.array_equal(got, want), rep


# ---- 6. out-of-range customers in a caller's rows ----------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("k", [2, 4])
@pytest.mark.parametrize("m", [300, 9000])
def test_merge_rejects_customers_out_of_range(td, k, m):
    """A row naming customer n, -1 or 65 536 (which the fast path's 16-bit customer table would wrap to a valid one):
    both paths report count -1 and leave the output untouched, the wrappers raise TaxiDispatchError, and the same rows
    with the customer put back merge normally."""
    import ctypes
    import torch
    from taxidispatcher_b200 import TaxiDispatchError
    eng = td.engine()
    n = 6000
    assert (m > fast_cap(n)) == (m == 9000)
    rng = np.random.default_rng(m + k)
    rows = synthetic_rows(rng, m, n, k, True, 1)[0]
    for bad in (n, -1, 65536):
        for col in (0, k - 1):
            r = rows.copy()
            r[m // 2, col] = bad
            src = torch.from_numpy(r).cuda()
            out = torch.full((m, REC_W), -5, dtype=torch.int32, device="cuda")
            cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
            nbytes = eng.lib.td_pool_merge_workspace_bytes(m, n)
            ws = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            rc = eng.lib.td_pool_merge(ctypes.c_void_p(src.data_ptr()), m, n, k, ctypes.c_void_p(out.data_ptr()),
                                       ctypes.c_void_p(cnt.data_ptr()), ctypes.c_void_p(ws.data_ptr()), nbytes,
                                       ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert rc == 0 and int(cnt.item()) == -1, (bad, col)
            assert bool((out == -5).all()), (bad, col)
            with pytest.raises(TaxiDispatchError):
                td.pool_merge([r], n, k)
            slots, counts = padded([r[: m // 3], r[m // 3:]])
            with pytest.raises(TaxiDispatchError):
                eng.pool_merge_padded(torch.from_numpy(slots).cuda(), torch.from_numpy(counts).cuda(), None, n, k)
            blocks = np.zeros((2, slots.shape[1] + 1, REC_W), np.int32)
            blocks[:, 1:] = slots
            blocks[:, 0, 0] = counts
            with pytest.raises(TaxiDispatchError):
                eng.pool_merge_headed_packed(torch.from_numpy(blocks).cuda(), None, n, k)
            merged, hc = eng.pool_merge_headed(torch.from_numpy(blocks).cuda(), None, n, k)
            assert int(hc.item()) == -1
    # a row outside the valid count is never read: the same bad row past the count merges normally
    slots, counts = padded([rows[: m // 2], rows[m // 2:]])
    slots = np.concatenate([slots, np.full((2, 1, REC_W), -1, np.int32)], axis=1)
    merged, cnt = eng.pool_merge_padded(torch.from_numpy(slots).cuda(), torch.from_numpy(counts).cuda(), None, n, k)
    assert np.array_equal(merged[: int(cnt.item())].cpu().numpy(), pool_ref.merge([rows[: m // 2], rows[m // 2:]], n, k))
    assert np.array_equal(td.pool_merge([rows], n, k), pool_ref.merge([rows], n, k))
