"""Stand-derived assignment as S x S transportation problems: td_assign_stands_batch, tdh_assign_stands,
Engine.assign_stands_batch, pack_stands_batch, solve_stands_batch and solve_assignment_stands.

CPU: the transportation oracle (oracle/transport_ref.py) against scipy's linear_sum_assignment on the dense padded
matrix, HiGHS on the S x S LP and networkx's min-cost flow; its expansion rule, flow read-back and stand certificate;
the C ABI's argument checks and no-device return; pack_cost_matrices unchanged by the shared index packing.
GPU: objectives against the dense exact solver (0..2048 and up to 20 000 per side, both imbalances, with and without
cutoff, S = 1 / 50 / 128, negative and non-metric tables, fill below the real costs) and against the oracle at 10^6 and
10^7; permutation, cost_of_row and the expansion rule; td_assign_certify on the expanded duals; independence from
position / neighbours / n_max / repetition; withdrawal; the worst-case phase counts; a Simulator replay."""
import ctypes

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from oracle import transport_ref as T

BIG = 250000


def _dense(dist, ct, cf, fill, cutoff):
    C = T.arc_costs(dist, fill, cutoff)
    n = max(len(ct), len(cf))
    M = np.full((n, n), fill, np.int64)
    if len(ct) and len(cf):
        M[:len(ct), :len(cf)] = C[np.ix_(np.asarray(ct), np.asarray(cf))]
    return M


def _table(rng, S, kind):
    if kind == "uniform":
        return rng.integers(0, 60, (S, S))
    if kind == "negative":
        return rng.integers(-40, 40, (S, S))
    if kind == "line":                                   # metric
        return 3 * np.abs(np.subtract.outer(np.arange(S), np.arange(S)))
    if kind == "staircase":                              # squared offsets: many cancellations along paths
        return np.subtract.outer(np.arange(S), np.arange(S)) ** 2
    return rng.integers(0, 4, (S, S))                    # "ties"


KINDS = ("uniform", "negative", "line", "staircase", "ties")


# ---- CPU: the oracle --------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", KINDS)
def test_oracle_vs_linear_sum_assignment(kind):
    rng = np.random.default_rng(hash(kind) % 1000)
    for it in range(60):
        S = int(rng.integers(1, 9))
        dist = _table(rng, S, kind)
        ct, cf = rng.integers(0, S, int(rng.integers(0, 22))), rng.integers(0, S, int(rng.integers(0, 22)))
        fill = int((BIG, 5, -3)[it % 3])
        cutoff = (None, 10, 2)[it % 3 if kind != "negative" else 0]
        r = T.solve(dist, ct, cf, fill, cutoff)
        M = _dense(dist, ct, cf, fill, cutoff)
        n = M.shape[0]
        ref = int(M[linear_sum_assignment(M)].sum()) if n else 0
        assert r["objective"] == ref
        col, cost = T.expand(r["flow"], ct, cf, T.arc_costs(dist, fill, cutoff), fill)
        assert sorted(col.tolist()) == list(range(n))
        assert np.array_equal(cost, M[np.arange(n), col]) and int(cost.sum()) == ref
        assert np.array_equal(T.flows_from_cols(col, ct, cf, S), r["flow"])
        assert T.check_certificate(T.arc_costs(dist, fill, cutoff), T.stand_counts(ct, S), T.stand_counts(cf, S),
                                   r["flow"], r["u"], r["v"])


def test_oracle_vs_highs_lp():
    from scipy.optimize import linprog
    rng = np.random.default_rng(11)
    for it in range(30):
        S = int(rng.integers(2, 12))
        C = T.arc_costs(_table(rng, S, KINDS[it % 5]), BIG, None)
        s = rng.integers(0, 30, S)
        d = rng.integers(0, 30, S)
        F = min(s.sum(), d.sum())
        if F == 0:
            continue
        # min sum C f, row sums <= s, column sums <= d, total = min(sum s, sum d)
        A_ub = np.vstack([np.kron(np.eye(S), np.ones(S)), np.kron(np.ones(S), np.eye(S))])
        res = linprog(C.reshape(-1), A_ub=A_ub, b_ub=np.concatenate([s, d]), A_eq=np.ones((1, S * S)), b_eq=[F],
                      bounds=(0, None), method="highs")
        flow, u, v, _, _ = T.solve_counts(C, s.astype(np.int64), d.astype(np.int64))
        assert int((flow * C).sum()) == round(res.fun)
        assert T.check_certificate(C, s, d, flow, u, v)


def test_oracle_vs_networkx():
    nx = pytest.importorskip("networkx")
    rng = np.random.default_rng(12)
    for it in range(15):
        S = int(rng.integers(2, 10))
        C = T.arc_costs(_table(rng, S, KINDS[it % 5]), BIG, None)
        s, d = rng.integers(0, 20, S), rng.integers(0, 20, S)
        F = int(min(s.sum(), d.sum()))
        G = nx.DiGraph()
        G.add_node("src", demand=-F)
        G.add_node("dst", demand=F)
        for a in range(S):
            G.add_edge("src", ("a", a), capacity=int(s[a]), weight=0)
            G.add_edge(("b", a), "dst", capacity=int(d[a]), weight=0)
            for b in range(S):
                G.add_edge(("a", a), ("b", b), weight=int(C[a, b]))
        ref = nx.min_cost_flow_cost(G)
        flow, _, _, _, _ = T.solve_counts(C, s.astype(np.int64), d.astype(np.int64))
        assert int((flow * C).sum()) == ref


def test_oracle_worst_case_phases():
    """Staircase tables with one-stand clusters on both sides: every phase ends one stand's supply or demand, so the
    phase count stays at the number of stands (DESIGN section 17)."""
    for S in (8, 32, 128):
        dist = _table(None, S, "staircase")
        r = T.solve(dist, np.repeat(np.arange(S), 7), np.repeat(np.arange(S)[::-1], 5), BIG)
        assert r["phases"] <= 2 * S


# ---- CPU: the C ABI ---------------------------------------------------------------------------------------------------
def _stands_call(lib, batch=1, S=4, n_max=8, ws_bytes=None, null=()):
    p = lambda a, name: None if name in null else ctypes.c_void_p(a)   # noqa: E731
    if ws_bytes is None:
        ws_bytes = lib.td_assign_stands_workspace_bytes(max(batch, 0), S if 1 <= S <= 128 else 1, max(n_max, 0))
    return lib.td_assign_stands_batch(p(16, "dist"), S, BIG, -1, p(32, "cab_to"), p(48, "cab_off"), p(64, "n_c"),
                                      p(80, "cust_from"), p(96, "cust_off"), p(112, "n_d"), batch, n_max,
                                      p(128, "col"), None, p(160, "obj"), None, None, None, p(256, "ws"), ws_bytes, None)


def test_abi_validation_before_device():
    from taxidispatcher_b200 import _lib
    lib = _lib.lib()
    lib.td_launch_count_reset()
    assert _lib.STANDS_MAX_S == 128
    for kw in (dict(batch=-1), dict(S=0), dict(S=129), dict(n_max=-1), dict(null=("dist",)), dict(null=("cab_to",)),
               dict(null=("cust_off",)), dict(null=("n_d",)), dict(null=("col",)), dict(null=("obj",)),
               dict(null=("ws",))):
        assert _stands_call(lib, **kw) == _lib.TD_ERR_INVALID, kw
    assert _stands_call(lib, ws_bytes=16) == _lib.TD_ERR_WORKSPACE
    assert _stands_call(lib, batch=0, null=("dist", "cab_to", "col", "obj", "ws")) == _lib.TD_OK
    assert lib.td_launch_count() == 0
    assert lib.td_assign_stands_workspace_bytes(2, 50, 600) >= 2 * 600 * 4 + 3 * 2 * 50 * 50 * 4


def test_abi_no_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    from taxidispatcher_b200 import _lib
    lib = _lib.lib()
    lib.td_launch_count_reset()
    assert _stands_call(lib) == _lib.TD_ERR_NO_DEVICE
    dist = np.zeros((2, 2), np.int32)
    ct, cf = np.zeros(3, np.int32), np.ones(2, np.int32)
    col, obj = np.zeros(3, np.int32), np.zeros(1, np.int64)
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    assert lib.tdh_assign_stands(ptr(dist), 2, ptr(ct), 3, ptr(cf), 2, BIG, -1, ptr(col), None, ptr(obj), None, None,
                                 None) == _lib.TD_ERR_NO_DEVICE
    cf[0] = 5                                            # a stand outside the table is refused before the device
    assert lib.tdh_assign_stands(ptr(dist), 2, ptr(ct), 3, ptr(cf), 2, BIG, -1, ptr(col), None, ptr(obj), None, None,
                                 None) == _lib.TD_ERR_INVALID
    assert lib.td_launch_count() == 0


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _dense_objective(td, dist, ct, cf, fill, cutoff):
    import torch
    from taxidispatcher_b200 import dispatch
    n = max(len(ct), len(cf))
    if n == 0:
        return 0
    eng = dispatch.engine()
    dist_d = dispatch._h2d_i32(dist)
    e = torch.empty(0, dtype=torch.int32, device=eng.device)
    cost = eng.cost_matrix(dist_d, dispatch._h2d_i32(ct) if len(ct) else e, dispatch._h2d_i32(cf) if len(cf) else e,
                           fill, cutoff)
    _, obj, _, _ = eng.assign(cost, n_real_rows=max(len(ct), 1) if len(ct) < n else n,
                              n_real_cols=max(len(cf), 1) if len(cf) < n else n)
    return int(obj.item())


def _gpu_batch(instances, dist, fill=BIG, cutoff=None, n_max=None, want_cost=True, host_check=True):
    from taxidispatcher_b200 import dispatch
    if host_check:
        pk = dispatch.pack_stands_batch(instances, dist)
    else:                                                # stands outside the table reach the kernel
        pk = dispatch.pack_stands_batch(instances)
        pk["dist"] = dispatch._h2d_i32(dist)
    n_max = pk["n_max"] if n_max is None else n_max
    col, cost, obj, u, v, st = dispatch.engine().assign_stands_batch(
        pk["dist"], pk["cab_to"], pk["cab_off"], pk["n_c"], pk["cust_from"], pk["cust_off"], pk["n_d"], n_max, fill, cutoff,
        want_cost=want_cost, want_duals=True, want_stats=True)
    return (col.cpu().numpy(), cost.cpu().numpy() if cost is not None else None, obj.cpu().numpy(), u.cpu().numpy(),
            v.cpu().numpy(), st.cpu().numpy())


def _check_instance(k, inst, dist, fill, cutoff, res, ref_obj):
    col, cost, obj, u, v, st = res
    ct, cf = inst
    S = dist.shape[0]
    n = max(len(ct), len(cf))
    C = T.arc_costs(dist, fill, cutoff)
    assert int(obj[k]) == ref_obj
    c = col[k, :n].astype(np.int64)
    assert np.array_equal(np.sort(c), np.arange(n))
    assert np.all(col[k, n:] == -1)
    pc = T.padded_costs(c, ct, cf, C, fill) if n <= 50000 else None
    if pc is not None:
        assert np.array_equal(cost[k, :n], pc) and int(pc.sum()) == ref_obj
    F = T.flows_from_cols(c, ct, cf, S)
    if n <= 50000:
        assert np.array_equal(T.expand(F, ct, cf, C, fill)[0], c)
    assert T.check_certificate(C, T.stand_counts(ct, S), T.stand_counts(cf, S), F, u[k], v[k])


SIZES = [(0, 0), (0, 5), (7, 0), (1, 1), (3, 9), (9, 3), (64, 64), (218, 600), (600, 368), (333, 1000), (2048, 1500),
         (1111, 2048)]


@pytest.mark.gpu
@pytest.mark.parametrize("S", [1, 50, 128])
@pytest.mark.parametrize("cutoff", [None, 10])
def test_objective_vs_dense(td, S, cutoff):
    rng = np.random.default_rng(S * 7 + (cutoff or 0))
    for kind in KINDS:
        dist = _table(rng, S, kind).astype(np.int32)
        fill = BIG if kind != "ties" else 2                      # fill below the real costs
        insts = []
        for nc, nd in SIZES:
            ct, cf = rng.integers(0, S, nc).astype(np.int32), rng.integers(0, S, nd).astype(np.int32)
            if kind == "line" and nc:
                ct[:] = S - 1                                    # every cab on one stand
            if kind == "staircase" and nd:
                cf[:] = 0                                        # every customer on one stand
            insts.append((ct, cf))
        res = _gpu_batch(insts, dist, fill, cutoff)
        for k, (ct, cf) in enumerate(insts):
            if kind == "negative":   # the dense rect solver is not exact on negative tables: scipy is the reference here
                M = _dense(dist, ct, cf, fill, cutoff)
                ref = int(M[linear_sum_assignment(M)].sum()) if len(M) else 0
            else:
                ref = _dense_objective(td, dist, ct, cf, fill, cutoff)
            _check_instance(k, (ct, cf), dist, fill, cutoff, res, ref)
            assert res[5][k, 0] == T.solve(dist, ct, cf, fill, cutoff)["phases"]


@pytest.mark.gpu
@pytest.mark.parametrize("S", [50, 128])
def test_large_vs_dense(td, S):
    rng = np.random.default_rng(S)
    dist = _table(rng, S, "uniform").astype(np.int32)
    for nc, nd, cutoff in ((20000, 20000, None), (20000, 13000, 10), (9000, 20000, 25)):
        ct, cf = rng.integers(0, S, nc).astype(np.int32), rng.integers(0, S, nd).astype(np.int32)
        res = _gpu_batch([(ct, cf)], dist, BIG, cutoff)
        _check_instance(0, (ct, cf), dist, BIG, cutoff, res, _dense_objective(td, dist, ct, cf, BIG, cutoff))


@pytest.mark.gpu
@pytest.mark.parametrize("n", [10**6, 10**7])
def test_huge_vs_oracle(td, n):
    rng = np.random.default_rng(n % 97)
    S = 128
    dist = _table(rng, S, "uniform").astype(np.int32)
    ct = rng.integers(0, S, n).astype(np.int32)
    cf = rng.integers(0, S, n - n // 7).astype(np.int32)
    ref = T.solve(dist, ct, cf, BIG, 30)
    res = _gpu_batch([(ct, cf)], dist, BIG, 30)
    _check_instance(0, (ct, cf), dist, BIG, 30, res, ref["objective"])
    assert np.array_equal(T.flows_from_cols(res[0][0].astype(np.int64), ct, cf, S), ref["flow"])


@pytest.mark.gpu
def test_independence_and_withdrawal(td):
    rng = np.random.default_rng(3)
    S = 50
    dist = _table(rng, S, "uniform").astype(np.int32)
    insts = [(rng.integers(0, S, a).astype(np.int32), rng.integers(0, S, b).astype(np.int32))
             for a, b in ((600, 300), (12, 40), (0, 3), (250, 250))]
    base = _gpu_batch(insts, dist, BIG, 10)
    for perm, n_max in (([3, 2, 1, 0], 700), ([1, 0, 3, 2], 600), ([0, 1, 2, 3], 4096)):
        got = _gpu_batch([insts[p] for p in perm], dist, BIG, 10, n_max=n_max)
        for k, p in enumerate(perm):
            n = max(len(insts[p][0]), len(insts[p][1]))
            assert np.array_equal(got[0][k, :n], base[0][p, :n]) and got[2][k] == base[2][p]
            assert np.array_equal(got[3][k], base[3][p]) and np.array_equal(got[4][k], base[4][p])
    again = _gpu_batch(insts, dist, BIG, 10)
    assert all(np.array_equal(a, b) for a, b in zip(again, base))
    bad = list(insts)
    bad[1] = (np.array([0, 51, 2], np.int32), insts[1][1])      # a stand outside the table
    with pytest.raises(IndexError):
        _gpu_batch(bad, dist, BIG, 10, n_max=600)
    got = _gpu_batch(bad, dist, BIG, 10, n_max=600, host_check=False)
    assert got[2][1] == -(1 << 63) and np.all(got[0][1] == -1) and not got[3][1].any() and not got[4][1].any()
    for k in (0, 2, 3):
        n = max(len(insts[k][0]), len(insts[k][1]))
        assert np.array_equal(got[0][k, :n], base[0][k, :n]) and got[2][k] == base[2][k]
    got = _gpu_batch(insts, dist, BIG, 10, n_max=300)            # n_b > n_max withdraws only that instance
    assert got[2][0] == -(1 << 63) and got[2][1] == base[2][1] and got[2][3] == base[2][3]


@pytest.mark.gpu
def test_certify_expanded_duals(td):
    import torch
    from taxidispatcher_b200 import dispatch
    rng = np.random.default_rng(8)
    eng = dispatch.engine()
    for S, nc, nd, cutoff, kind in ((50, 600, 300, 10, "uniform"), (128, 700, 1400, None, "line"),
                                    (17, 500, 500, 4, "ties"), (50, 2000, 1999, None, "staircase")):
        dist = _table(rng, S, kind).astype(np.int32)
        ct, cf = rng.integers(0, S, nc).astype(np.int32), rng.integers(0, S, nd).astype(np.int32)
        col, _, obj, u, v, _ = _gpu_batch([(ct, cf)], dist, BIG, cutoff)
        n = max(nc, nd)
        nr, ncol = (nc if nc < n else n), (nd if nd < n else n)
        dist_d = dispatch._h2d_i32(dist)
        cost = eng.cost_matrix(dist_d, dispatch._h2d_i32(ct), dispatch._h2d_i32(cf), BIG, cutoff)
        uu = np.zeros(n, np.int64); uu[:nc] = u[0][ct]
        vv = np.zeros(n, np.int64); vv[:nd] = v[0][cf]
        cert = eng.assign_certify(cost, torch.from_numpy(col[0, :n].copy()).cuda(), torch.from_numpy(uu).cuda(),
                                  torch.from_numpy(vv).cuda(), nr, ncol)
        assert cert["optimal"], cert
        assert cert["dual_objective"] + (n - min(nc, nd)) * BIG == int(obj[0])


@pytest.mark.gpu
def test_worst_case_phases(td):
    """Staircase tables with one-stand clusters: the phase / augmentation counts equal the oracle's and stay within the
    bound DESIGN section 17 states (at most 2S)."""
    for S in (8, 64, 128):
        dist = _table(None, S, "staircase").astype(np.int32)
        insts = [(np.repeat(np.arange(S), 7).astype(np.int32), np.repeat(np.arange(S)[::-1], 5).astype(np.int32)),
                 (np.zeros(900, np.int32), np.arange(S, dtype=np.int32).repeat(3)),
                 (np.arange(S, dtype=np.int32).repeat(4), np.full(1000, S - 1, np.int32))]
        res = _gpu_batch(insts, dist)
        for k, (ct, cf) in enumerate(insts):
            r = T.solve(dist, ct, cf, BIG)
            assert int(res[2][k]) == r["objective"]
            assert tuple(res[5][k]) == (r["phases"], r["augmentations"])
            assert r["phases"] <= 2 * S


@pytest.mark.gpu
def test_host_functions(td):
    from taxidispatcher_b200 import _lib, dispatch
    rng = np.random.default_rng(9)
    S = 50
    dist = _table(rng, S, "uniform").astype(np.int32)
    dist_d = dispatch._h2d_i32(dist)
    for nc, nd in ((600, 218), (600, 368), (5, 9), (0, 4)):
        ct, cf = rng.integers(0, S, nc).astype(np.int32), rng.integers(0, S, nd).astype(np.int32)
        n, col, cost = td.solve_assignment_stands(dist_d, ct, cf, BIG, 10)
        n2, col2, cost2 = dispatch.solve_assignment(dist_d, ct, cf, BIG, 10)
        assert n == n2 and int(cost.sum()) == int(cost2.sum())
        assert np.array_equal(cost, T.padded_costs(col, ct, cf, T.arc_costs(dist, BIG, 10), BIG))
    with pytest.raises(IndexError):
        td.solve_assignment_stands(dist_d, [1, 2], [3, 99])
    insts = [(rng.integers(0, S, 600), rng.integers(0, S, m)) for m in (218, 300, 368)]
    for (ct, cf), (col, obj, u, v) in zip(insts, td.solve_stands_batch(dist, insts, cutoff=10, want_duals=True)):
        assert obj == _dense_objective(td, dist, ct, cf, BIG, 10) and len(u) == S
    # the host twin
    lib = _lib.lib()
    ct, cf = rng.integers(0, S, 70).astype(np.int32), rng.integers(0, S, 40).astype(np.int32)
    col, cost, obj = np.zeros(70, np.int32), np.zeros(70, np.int32), np.zeros(1, np.int64)
    u, v, st = np.zeros(S, np.int64), np.zeros(S, np.int64), np.zeros(2, np.int32)
    ptr = lambda a: a.ctypes.data_as(ctypes.c_void_p)   # noqa: E731
    assert lib.tdh_assign_stands(ptr(dist), S, ptr(ct), 70, ptr(cf), 40, BIG, -1, ptr(col), ptr(cost), ptr(obj), ptr(u),
                                 ptr(v), ptr(st)) == 0
    assert int(obj[0]) == _dense_objective(td, dist, ct, cf, BIG, None) == int(cost.astype(np.int64).sum())


@pytest.mark.gpu
def test_pack_cost_matrices_unchanged_and_pack_stands(td):
    from taxidispatcher_b200 import dispatch
    rng = np.random.default_rng(10)
    S = 30
    dist = _table(rng, S, "uniform").astype(np.int32)
    dist_d = dispatch._h2d_i32(dist)
    insts = [(rng.integers(0, S, a), rng.integers(0, S, b)) for a, b in ((5, 9), (0, 3), (40, 12))]
    packed, sizes, offsets, n_max, ns = dispatch.pack_cost_matrices(dist_d, insts, BIG, 10)
    p = packed.cpu().numpy()
    assert ns == [9, 3, 40] and n_max == 40 and sizes.cpu().tolist() == ns
    for b, (ct, cf) in enumerate(insts):
        o = int(offsets[b])
        assert np.array_equal(p[o: o + ns[b] ** 2].reshape(ns[b], ns[b]), _dense(dist, ct, cf, BIG, 10))
    pk = dispatch.pack_stands_batch(insts, dist)
    assert pk["n_c"].cpu().tolist() == [5, 0, 40] and pk["n_d"].cpu().tolist() == [9, 3, 12] and pk["ns"] == ns
    idx = pk["cab_to"].cpu().numpy()
    for b, (ct, cf) in enumerate(insts):
        co, uo = int(pk["cab_off"][b]), int(pk["cust_off"][b])
        assert np.array_equal(idx[co: co + len(ct)], ct) and np.array_equal(idx[uo: uo + len(cf)], cf)
    assert np.array_equal(pk["dist"].cpu().numpy(), dist)


@pytest.mark.gpu
def test_simulator_replay_stands(td):
    """120 Simulator steps through a CudaBackend that records the stand arrays cost() receives: at every solver step
    solve_assignment_stands gives the dense objective.  The backend returns the dense results, so the replay is
    unchanged."""
    import gzip
    import os
    from conftest import GOLDEN
    from taxidispatcher_b200 import dispatch, formats
    from taxidispatcher_b200.simulator import BIG_COST, DROP_TIME, CudaBackend, Simulator

    class Recording(CudaBackend):
        def __init__(self):
            super().__init__()
            self.seen, self.checked = {}, 0

        def cost(self, dist, cab_to, cust_from):
            host = super().cost(dist, cab_to, cust_from)
            self.seen[id(host)] = (host, np.asarray(dist), np.array(cab_to, np.int32), np.array(cust_from, np.int32))
            return host

        def solve(self, n, cost, n_cabs=None, n_cust=None):
            x = super().solve(n, cost, n_cabs, n_cust)
            rec = self.seen.get(id(cost))
            if rec is not None and rec[0] is cost and n:
                _, dist, ct, cf = rec
                dense = int((np.asarray(cost, np.int64).reshape(-1) * np.asarray(x).reshape(-1)).sum())
                _, _, c = dispatch.solve_assignment_stands(dispatch._h2d_i32(dist), ct, cf, BIG_COST, DROP_TIME)
                assert int(c.astype(np.int64).sum()) == dense
                self.checked += 1
            return x

    rows = formats.read_taxi_demand(gzip.open(os.path.join(GOLDEN, "taxi_demand.txt.gz"), "rt").read())
    be = Recording()
    log, _ = Simulator(rows, backend=be).run(120)
    ref, _ = Simulator(rows).run(120)
    assert log == ref and be.checked > 0
