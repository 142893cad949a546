"""Exact 2-passenger pool: td_pool_pairs_exact_batch (minimum-cost maximum-cardinality pair matching, one CTA per
instance), the dispatch helpers on top of it, the greedy-vs-optimum experiment (pool_opt_min.py; the paper, p.5,
reports the greedy within 3 % of the optimum, 2 % on average) and the Simulator's exact_pool option.

CPU: argument validation and the no-device return of the C ABI; the C oracle against networkx and scipy's MILP on the
reference's equality ILP; structural invariants of the oracle's rows; the experiment and the Simulator with oracles.
GPU: counts and totals against the oracle from n = 0 to 1445, batches (one launch, ragged, poisoned gaps, withdrawn
instances, position / n_max independence, repeatability) and the Simulator replay with exact pooling."""
import ctypes
import gzip
import os

import numpy as np
import pytest

from conftest import GOLDEN
from oracle import pairs_ref, pool_ref
from taxidispatcher_b200 import experiments as ex

MAX_N = 4096
D50 = np.abs(np.subtract.outer(np.arange(50), np.arange(50))).astype(np.int32)


def rand_instance(rng, n, removed=0.0, one_stand=False):
    f = rng.integers(0, 50, n).astype(np.int32)
    t = rng.integers(0, 50, n).astype(np.int32)
    if one_stand:
        f[:] = 7
        t[:] = 7
    if removed and n:
        f[rng.random(n) < removed] = -1
    return f, t


# ---- CPU: the C ABI refuses bad arguments before it looks for a device -----------------------------------------------
def _abi():
    from taxidispatcher_b200 import _lib
    return _lib, _lib.lib()


def _call(lib, frm=16, to=32, sizes=48, offsets=64, batch=1, n_max=4, dist=80, n_stands=50, accept_all=1,
          max_loss=1.01, rows=96, npairs=112, cost=128, ws=144, ws_bytes=None):
    p = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    if ws_bytes is None:
        ws_bytes = lib.td_pool_pairs_exact_workspace_bytes(max(batch, 0), min(max(n_max, 0), MAX_N))
    return lib.td_pool_pairs_exact_batch(p(frm), p(to), p(sizes), p(offsets), batch, n_max, p(dist), n_stands, accept_all,
                                         max_loss, p(rows), p(npairs), p(cost), p(ws), ws_bytes, None)


def test_pairs_exact_abi_argument_validation():
    _lib, lib = _abi()
    INV = _lib.TD_ERR_INVALID
    launches = lib.td_launch_count()
    assert _call(lib, batch=-1) == INV
    assert _call(lib, n_max=-1) == INV
    assert _call(lib, n_max=MAX_N + 1) == INV
    assert _call(lib, n_stands=0) == INV
    assert _call(lib, n_stands=129) == INV
    assert _call(lib, accept_all=0, max_loss=float("nan")) == INV
    assert _call(lib, accept_all=0, max_loss=float("inf")) == INV
    for name in ("frm", "to", "sizes", "offsets", "dist", "rows", "npairs", "cost"):
        assert _call(lib, **{name: None}) == INV, name
    assert _call(lib, ws=None) == _lib.TD_ERR_WORKSPACE
    assert _call(lib, ws_bytes=lib.td_pool_pairs_exact_workspace_bytes(1, 4) - 1) == _lib.TD_ERR_WORKSPACE
    assert _call(lib, batch=0, n_max=MAX_N + 1) == INV
    assert lib.td_pool_pairs_exact_workspace_bytes(-1, 4) == 0 and lib.td_pool_pairs_exact_workspace_bytes(1, MAX_N + 1) == 0
    # the host twin checks the stand table and the rows itself
    f = np.array([0, 1], np.int32)
    d = np.ascontiguousarray(D50)
    out, npairs, tot = np.zeros((1, 4), np.int32), ctypes.c_int32(0), ctypes.c_int64(0)
    twin = lambda frm, dist, S: lib.tdh_pool_pairs_exact(frm.ctypes.data, frm.ctypes.data, len(frm), dist.ctypes.data, S, 1,  # noqa: E731
                                                         1.01, out.ctypes.data, ctypes.byref(npairs), ctypes.byref(tot))
    assert twin(np.array([0, 50], np.int32), d, 50) == INV
    bad = d.copy()
    bad[3, 4] = (1 << 22) + 1
    assert twin(f, bad, 50) == INV
    assert lib.td_launch_count() == launches


def test_pairs_exact_abi_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    _lib, lib = _abi()
    launches = lib.td_launch_count()
    assert _call(lib) == _lib.TD_ERR_NO_DEVICE
    assert _call(lib, batch=0) == _lib.TD_ERR_NO_DEVICE
    assert _call(lib, n_max=MAX_N, ws_bytes=lib.td_pool_pairs_exact_workspace_bytes(1, MAX_N)) == _lib.TD_ERR_NO_DEVICE
    f = np.array([0, 1, 2], np.int32)
    d = np.ascontiguousarray(D50)
    out, npairs, tot = np.zeros((1, 4), np.int32), ctypes.c_int32(0), ctypes.c_int64(0)
    assert lib.tdh_pool_pairs_exact(f.ctypes.data, f.ctypes.data, 3, d.ctypes.data, 50, 1, 1.01, out.ctypes.data,
                                    ctypes.byref(npairs), ctypes.byref(tot)) == _lib.TD_ERR_NO_DEVICE
    assert lib.td_launch_count() == launches


# ---- CPU: the oracle --------------------------------------------------------------------------------------------------
def _cand(f, t, D, A, B, accept_all, max_loss):
    if A == B or f[A] < 0 or f[B] < 0:
        return None
    c1 = int(D[f[A], f[B]] + D[f[B], t[A]] + D[t[A], t[B]])
    c2 = int(D[f[A], f[B]] + D[f[B], t[B]] + D[t[B], t[A]])
    ok = accept_all or (D[f[B], t[A]] + D[t[A], t[B]] < D[f[B], t[B]] * max_loss and
                        D[f[A], f[B]] + D[f[B], t[A]] < D[f[A], t[A]] * max_loss) or c2 < D[f[A], t[A]] * max_loss
    return (min(c1, c2), A * len(f) + B, 1 if c1 < c2 else 0) if ok else None


def edges(f, t, D, accept_all, max_loss):
    """{(i, j): preferred candidate row [A, B, plan, cost]} for i < j, straight from the definition."""
    n, out = len(f), {}
    for i in range(n):
        for j in range(i + 1, n):
            cs = [c for c in (_cand(f, t, D, i, j, accept_all, max_loss), _cand(f, t, D, j, i, accept_all, max_loss)) if c]
            if cs:
                cost, key, plan = min(cs)
                out[(i, j)] = [key // n, key % n, plan, cost]
    return out


def check_rows(rows, f, t, D, accept_all, max_loss):
    """Disjoint pairs, each the preferred candidate of its pair, in (cost, A*n+B) order."""
    rows = np.asarray(rows).reshape(-1, 4)
    n = len(f)
    custs = rows[:, :2].reshape(-1)
    assert len(set(custs.tolist())) == len(custs)
    e = edges(f, t, D, accept_all, max_loss) if n <= 120 else None
    for A, B, plan, cost in rows.tolist():
        if e is not None:
            assert e[(min(A, B), max(A, B))] == [A, B, plan, cost]
        else:
            c = [x for x in (_cand(f, t, D, A, B, accept_all, max_loss), _cand(f, t, D, B, A, accept_all, max_loss)) if x]
            assert c and min(c) == (cost, A * n + B, plan)
    keys = [(c, a * n + b) for a, b, _, c in rows.tolist()]
    assert keys == sorted(keys)


def oracle_cases():
    rng = np.random.default_rng(2024)
    cases = []
    for k in range(220):
        n = int(rng.integers(0, 61))
        accept_all = k % 2 == 0
        max_loss = (1.01, 1.1, 1.3)[k % 3]
        f, t = rand_instance(rng, n, removed=0.2 if k % 5 == 0 else 0.0, one_stand=k % 11 == 0)
        cases.append((f, t, accept_all, max_loss))
    return cases


def test_oracle_matches_networkx():
    nx = pytest.importorskip("networkx")
    for f, t, accept_all, max_loss in oracle_cases():
        G = nx.Graph()
        G.add_nodes_from(range(len(f)))
        for (i, j), r in edges(f, t, D50, accept_all, max_loss).items():
            G.add_edge(i, j, neg=-r[3], cost=r[3])
        M = nx.max_weight_matching(G, maxcardinality=True, weight="neg")
        rows, m, total = pairs_ref.pairs_exact(f, t, D50, accept_all, max_loss)
        assert (m, total) == (len(M), sum(G[u][v]["cost"] for u, v in M))
        check_rows(rows, f, t, D50, accept_all, max_loss)
        g = pool_ref.pairs(f, t, D50, accept_all=accept_all, max_loss=max_loss)
        gm, gt = len(g), int(g[:, 3].sum()) if len(g) else 0
        assert m >= gm and (m > gm or total <= gt)


def test_oracle_matches_milp_equality_ilp():
    """pool_opt_min.py's model: x_ij per ordered accepted pair, sum_i x_ij + sum_i x_ji = 1 for every customer."""
    opt = pytest.importorskip("scipy.optimize")
    from scipy.sparse import lil_matrix
    rng = np.random.default_rng(5)
    for _ in range(3):
        f, t = rand_instance(rng, 100)
        cand = [(A, B, _cand(f, t, D50, A, B, True, 1.01)[0]) for A in range(100) for B in range(100) if A != B]
        Aeq = lil_matrix((100, len(cand)))
        for k, (A, B, _) in enumerate(cand):
            Aeq[A, k] += 1
            Aeq[B, k] += 1
        res = opt.milp(np.array([c for _, _, c in cand], float), integrality=np.ones(len(cand)), bounds=opt.Bounds(0, 1),
                       constraints=opt.LinearConstraint(Aeq.tocsr(), 1, 1))
        assert res.status == 0
        _, m, total = pairs_ref.pairs_exact(f, t, D50, True)
        assert m == 50 and total == round(res.fun)


def test_pool_greedy_vs_optimum_with_oracles():
    rng = np.random.default_rng(11)
    inst = [rand_instance(rng, 100) for _ in range(20)]
    res = ex.pool_greedy_vs_optimum(inst, D50, True, 1.01, greedy=lambda f, t, d, a, ml: pool_ref.pairs(f, t, d, a, ml),
                                    exact=lambda ins, d, a, ml: [pairs_ref.pairs_exact(f, t, d, a, ml)[0] for f, t in ins])
    assert len(res) == 20
    for (f, t), (gc, gcost, oc, ocost) in zip(inst, res):
        g = pool_ref.pairs(f, t, D50)
        _, m, total = pairs_ref.pairs_exact(f, t, D50)
        assert (gc, gcost, oc, ocost) == (len(g), int(g[:, 3].sum()), m, total)
        assert oc == gc == 50 and ocost <= gcost
    gap = sum(g for _, g, _, _ in res) / sum(o for _, _, _, o in res) - 1
    assert 0 <= gap < 0.2


class Recording:
    """Wraps a Simulator backend and keeps (frm, to, rows) of every pool step."""

    def __init__(self, inner):
        self.inner, self.pools = inner, []

    def pool_pairs(self, frm, to, dist):
        r = self.inner.pool_pairs(frm, to, dist)
        self.pools.append((np.array(frm), np.array(to), np.asarray(r).reshape(-1, 4).copy()))
        return r

    def __getattr__(self, name):
        return getattr(self.inner, name)


def _demand():
    from taxidispatcher_b200 import formats
    return formats.read_taxi_demand(gzip.open(os.path.join(GOLDEN, "taxi_demand.txt.gz"), "rt").read())


def test_simulator_exact_pool_oracle_backend():
    from taxidispatcher_b200.simulator import Simulator
    rec = Recording(pairs_ref.OracleBackend(exact_pool=True))
    sim = Simulator(_demand(), backend=rec)
    sim.run(4)
    assert rec.pools
    for f, t, rows in rec.pools:
        g = pool_ref.pairs(f, t, sim.dist)
        assert len(rows) == len(f) // 2
        assert int(rows[:, 3].sum()) <= int(g[:, 3].sum())


# ---- GPU ----------------------------------------------------------------------------------------------------------------
SIZES = (0, 1, 2, 3, 5, 16, 99, 100, 101, 232, 500, 1000, 1445)


@pytest.mark.gpu
def test_single_instances_match_oracle(td):
    rng = np.random.default_rng(7)
    for n in SIZES:
        for accept_all in (True, False):
            f, t = rand_instance(rng, n, removed=0.1 if n % 2 else 0.0)
            rows = td.find_pool_pairs_exact(f, t, D50, accept_all=accept_all, max_loss=1.05)
            _, m, total = pairs_ref.pairs_exact(f, t, D50, accept_all, 1.05)
            assert (len(rows), int(rows[:, 3].astype(np.int64).sum()) if len(rows) else 0) == (m, total), (n, accept_all)
            check_rows(rows, f, t, D50, accept_all, 1.05)


@pytest.mark.gpu
def test_batch_one_launch_matches_oracle(td):
    from taxidispatcher_b200 import _lib, dispatch
    rng = np.random.default_rng(8)
    for accept_all in (True, False):
        inst = [rand_instance(rng, 100) for _ in range(1000)]
        lib = _lib.lib()
        dispatch.find_pool_pairs_exact_batch(inst[:2], D50, accept_all)          # warm the workspace and staging
        before = lib.td_launch_count()
        res = dispatch.find_pool_pairs_exact_batch(inst, D50, accept_all, 1.05)
        assert lib.td_launch_count() - before == 1
        for (f, t), rows in zip(inst, res):
            _, m, total = pairs_ref.pairs_exact(f, t, D50, accept_all, 1.05)
            assert (len(rows), int(rows[:, 3].sum())) == (m, total)


@pytest.mark.gpu
def test_batch_ragged_poisoned_withdrawn_and_deterministic(td):
    import torch
    from taxidispatcher_b200 import dispatch
    rng = np.random.default_rng(9)
    inst = [rand_instance(rng, n, removed=0.15) for n in (37, 0, 120, 1, 64, 201, 2, 90)]
    ref = [pairs_ref.pairs_exact(f, t, D50, True) for f, t in inst]
    res = dispatch.find_pool_pairs_exact_batch(inst, D50)
    for r, (_, m, total) in zip(res, ref):
        assert (len(r), int(r[:, 3].sum()) if len(r) else 0) == (m, total)
    # poisoned gaps: stands far outside the table between the instances change nothing
    eng = dispatch.engine()
    sizes = [len(f) for f, _ in inst]
    offs = np.cumsum([0] + [s + 5 for s in sizes[:-1]]).astype(np.int64)
    total = int(offs[-1] + sizes[-1] + 5)
    fr, to = np.full(total, 10**6, np.int32), np.full(total, -10**6, np.int32)
    for (f, t), o in zip(inst, offs):
        fr[o: o + len(f)] = f
        to[o: o + len(t)] = t
    dev = lambda a, dt=torch.int32: torch.from_numpy(np.ascontiguousarray(a)).to(dtype=dt, device="cuda")  # noqa: E731
    rows, npairs, cost = eng.pool_pairs_exact_batch(dev(fr), dev(to), dev(np.array(sizes, np.int32)), dev(offs, torch.int64),
                                                    max(sizes), dev(D50))
    rows, npairs, cost = rows.cpu().numpy(), npairs.cpu().numpy(), cost.cpu().numpy()
    for b, r in enumerate(res):
        assert npairs[b] == len(r) and np.array_equal(rows[b, : len(r)], r) and cost[b] == int(r[:, 3].sum() if len(r) else 0)
    # withdrawn instances next to valid ones: bad size, bad offset, stand outside the table
    bad_sizes = np.array(sizes, np.int32)
    bad_offs = offs.copy()
    bad_sizes[1] = max(sizes) + 1
    bad_offs[3] = -1
    fr2 = fr.copy()
    fr2[offs[4] + 2] = 50
    rows, npairs, cost = eng.pool_pairs_exact_batch(dev(fr2), dev(to), dev(bad_sizes), dev(bad_offs, torch.int64), max(sizes),
                                                    dev(D50))
    rows, npairs, cost = rows.cpu().numpy(), npairs.cpu().numpy(), cost.cpu().numpy()
    for b, r in enumerate(res):
        if b in (1, 3, 4):
            assert npairs[b] == -1 and cost[b] == np.iinfo(np.int64).min and (rows[b] == -1).all()
        else:
            assert npairs[b] == len(r) and np.array_equal(rows[b, : len(r)], r)
    # the same instance at other positions, next to other neighbours and under a larger n_max: identical rows
    f, t = inst[5]
    big = rand_instance(rng, 700)
    for batch in ([(f, t)], [big, (f, t)], [inst[0], inst[2], (f, t), big]):
        out = dispatch.find_pool_pairs_exact_batch(batch, D50)
        assert np.array_equal(out[[i for i, x in enumerate(batch) if x[0] is f][0]], res[5])
    # repeated calls are byte-identical
    again = dispatch.find_pool_pairs_exact_batch(inst, D50)
    assert all(np.array_equal(a, b) for a, b in zip(again, res))


@pytest.mark.gpu
def test_pool_greedy_vs_optimum_on_gpu(td):
    rng = np.random.default_rng(12)
    inst = [rand_instance(rng, 100) for _ in range(50)]
    res = ex.pool_greedy_vs_optimum(inst, D50)
    for (f, t), (gc, gcost, oc, ocost) in zip(inst, res):
        g = pool_ref.pairs(f, t, D50)
        _, m, total = pairs_ref.pairs_exact(f, t, D50)
        assert (gc, gcost, oc, ocost) == (len(g), int(g[:, 3].sum()), m, total)


@pytest.mark.gpu
def test_simulator_replay_exact_pool(td):
    from taxidispatcher_b200.simulator import CudaBackend, Simulator
    rec = Recording(CudaBackend(exact_pool=True))
    sim = Simulator(_demand(), backend=rec)
    sim.run(60)
    assert len(rec.pools) >= 50
    for f, t, rows in rec.pools:
        _, m, total = pairs_ref.pairs_exact(f, t, sim.dist, True)
        assert (len(rows), int(rows[:, 3].astype(np.int64).sum()) if len(rows) else 0) == (m, total)
