"""Greedy 2-passenger pool, batched: td_pool_pairs_batch (Simulator.findPool over many instances, one CTA per instance),
its host twin tdh_pool_pairs, find_pool_pairs_batch and the two-launch pool_greedy_vs_optimum.

CPU: argument validation and the no-device return of the C ABI, the twin's own checks, the experiment with oracles.
GPU: rows byte for byte against both find_pool_pairs (td_pool_pairs) and the C oracle from n = 0 to 4096, one launch for
1000 instances, ragged / poisoned / withdrawn batches, position / n_max independence, repeatability, the two-launch
experiment and the pool inputs of a Simulator replay."""
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
          max_loss=1.01, rows=96, npairs=112, cost=128):
    p = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    return lib.td_pool_pairs_batch(p(frm), p(to), p(sizes), p(offsets), batch, n_max, p(dist), n_stands, accept_all,
                                   max_loss, p(rows), p(npairs), p(cost), None)


def _twin(lib, frm, to, dist, n_stands, accept_all=1, max_loss=1.01):
    out, npairs, tot = np.zeros((max(len(frm) // 2, 1), 4), np.int32), ctypes.c_int32(0), ctypes.c_int64(0)
    rc = lib.tdh_pool_pairs(frm.ctypes.data, to.ctypes.data, len(frm), dist.ctypes.data, n_stands, accept_all, max_loss,
                            out.ctypes.data, ctypes.byref(npairs), ctypes.byref(tot))
    return rc, out[: max(npairs.value, 0)], tot.value


def test_pairs_batch_abi_argument_validation():
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
    assert _call(lib, accept_all=0, max_loss=float("-inf")) == INV
    for name in ("frm", "to", "sizes", "offsets", "dist", "rows", "npairs", "cost"):
        assert _call(lib, **{name: None}) == INV, name
    assert _call(lib, batch=0, n_max=MAX_N + 1) == INV
    assert _call(lib, batch=0, n_stands=0) == INV
    # the host twin checks the stand table and the rows itself
    f = np.array([0, 1], np.int32)
    d = np.ascontiguousarray(D50)
    assert _twin(lib, np.array([0, 50], np.int32), f, d, 50)[0] == INV           # live row, stand outside the table
    assert _twin(lib, f, np.array([0, -1], np.int32), d, 50)[0] == INV
    bad = d.copy()
    bad[3, 4] = (1 << 22) + 1
    assert _twin(lib, f, f, bad, 50)[0] == INV
    bad[3, 4] = -1
    assert _twin(lib, f, f, bad, 50)[0] == INV
    assert _twin(lib, f, f, d, 129)[0] == INV
    assert _twin(lib, f, f, d, 50, accept_all=0, max_loss=float("nan"))[0] == INV
    assert lib.td_launch_count() == launches


def test_pairs_batch_abi_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    _lib, lib = _abi()
    launches = lib.td_launch_count()
    assert _call(lib) == _lib.TD_ERR_NO_DEVICE
    assert _call(lib, batch=0) == _lib.TD_ERR_NO_DEVICE
    assert _call(lib, n_max=MAX_N) == _lib.TD_ERR_NO_DEVICE
    f = np.array([0, 1, 2], np.int32)
    # a removed row's `to` is not checked: it is never read
    assert _twin(lib, np.array([0, -1, 2], np.int32), np.array([0, 99, 2], np.int32), np.ascontiguousarray(D50), 50)[0] == \
        _lib.TD_ERR_NO_DEVICE
    assert _twin(lib, f, f, np.ascontiguousarray(D50), 50)[0] == _lib.TD_ERR_NO_DEVICE
    assert lib.td_launch_count() == launches


def test_pool_greedy_vs_optimum_with_injected_oracles():
    rng = np.random.default_rng(21)
    inst = [rand_instance(rng, n, removed=0.1 if n % 2 else 0.0) for n in (0, 1, 2, 3, 37, 100, 100, 151)]
    greedy = lambda f, t, d, a, ml: pool_ref.pairs(f, t, d, a, ml)   # noqa: E731
    exact = lambda ins, d, a, ml: [pairs_ref.pairs_exact(f, t, d, a, ml)[0] for f, t in ins]   # noqa: E731
    for accept_all in (True, False):
        res = ex.pool_greedy_vs_optimum(inst, D50, accept_all, 1.05, greedy=greedy, exact=exact)
        for (f, t), r in zip(inst, res):
            g = pool_ref.pairs(f, t, D50, accept_all, 1.05)
            _, m, total = pairs_ref.pairs_exact(f, t, D50, accept_all, 1.05)
            assert r == (len(g), int(g[:, 3].sum()) if len(g) else 0, m, total)


# ---- GPU ----------------------------------------------------------------------------------------------------------------
SIZES = (0, 1, 2, 3, 5, 16, 99, 100, 101, 232, 500, 1000, 1445, 4096)
ONE_STAND = (2, 5, 100, 500, 1445)


def _same(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes()


@pytest.mark.gpu
def test_rows_equal_find_pool_pairs_and_oracle(td):
    rng = np.random.default_rng(31)
    inst = [rand_instance(rng, n, removed=0.1 if n % 2 else 0.0) for n in SIZES]
    inst += [rand_instance(rng, n, one_stand=True) for n in ONE_STAND]
    for accept_all in (True, False):
        for max_loss in (1.01, 1.05):
            res = td.find_pool_pairs_batch(inst, D50, accept_all, max_loss)
            for (f, t), rows in zip(inst, res):
                dev = td.find_pool_pairs(f, t, D50, accept_all, max_loss)
                ref = pool_ref.pairs(f, t, D50, accept_all, max_loss)
                assert _same(rows, dev), (len(f), accept_all, max_loss)
                assert np.array_equal(rows, ref), (len(f), accept_all, max_loss)


@pytest.mark.gpu
def test_host_twin_equals_oracle(td):
    _lib, lib = _abi()
    rng = np.random.default_rng(32)
    for n in (0, 1, 7, 100, 1445):
        f, t = rand_instance(rng, n, removed=0.1)
        rc, rows, total = _twin(lib, f, t, np.ascontiguousarray(D50), 50, 0, 1.05)
        ref = pool_ref.pairs(f, t, D50, False, 1.05)
        assert rc == 0 and np.array_equal(rows, ref) and total == (int(ref[:, 3].sum()) if len(ref) else 0)


@pytest.mark.gpu
def test_batch_1000x100_one_launch(td):
    from taxidispatcher_b200 import _lib, dispatch
    lib = _lib.lib()
    rng = np.random.default_rng(33)
    for accept_all in (True, False):
        inst = [rand_instance(rng, 100) for _ in range(1000)]
        dispatch.find_pool_pairs_batch(inst[:2], D50, accept_all)               # warm the staging buffers
        before = lib.td_launch_count()
        res = dispatch.find_pool_pairs_batch(inst, D50, accept_all, 1.01)
        assert lib.td_launch_count() - before == 1
        for (f, t), rows in zip(inst, res):
            assert np.array_equal(rows, pool_ref.pairs(f, t, D50, accept_all, 1.01))


@pytest.mark.gpu
def test_batch_ragged_poisoned_withdrawn_and_deterministic(td):
    import torch
    from taxidispatcher_b200 import dispatch
    rng = np.random.default_rng(34)
    inst = [rand_instance(rng, n, removed=0.15) for n in (37, 0, 120, 1, 64, 201, 2, 90)]
    res = dispatch.find_pool_pairs_batch(inst, D50)
    for (f, t), r in zip(inst, res):
        assert _same(r, dispatch.find_pool_pairs(f, t, D50))
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
    rows, npairs, cost = eng.pool_pairs_batch(dev(fr), dev(to), dev(np.array(sizes, np.int32)), dev(offs, torch.int64),
                                              max(sizes), dev(D50))
    rows, npairs, cost = rows.cpu().numpy(), npairs.cpu().numpy(), cost.cpu().numpy()
    for b, r in enumerate(res):
        assert npairs[b] == len(r) and _same(rows[b, : len(r)], r) and (rows[b, len(r):] == -1).all()
        assert cost[b] == int(r[:, 3].astype(np.int64).sum())
    # withdrawn instances next to valid ones: bad size, bad offset, a live stand outside the table
    bad_sizes = np.array(sizes, np.int32)
    bad_offs = offs.copy()
    bad_sizes[1] = max(sizes) + 1
    bad_sizes[6] = -1
    bad_offs[3] = -1
    fr2 = fr.copy()
    fr2[offs[4] + 2] = 50 if fr[offs[4] + 2] >= 0 else 0
    to2 = to.copy()
    to2[offs[4] + 2] = 50
    rows, npairs, cost = eng.pool_pairs_batch(dev(fr2), dev(to2), dev(bad_sizes), dev(bad_offs, torch.int64), max(sizes),
                                              dev(D50))
    rows, npairs, cost = rows.cpu().numpy(), npairs.cpu().numpy(), cost.cpu().numpy()
    for b, r in enumerate(res):
        if b in (1, 3, 4, 6):
            assert npairs[b] == -1 and cost[b] == np.iinfo(np.int64).min and (rows[b] == -1).all()
        else:
            assert npairs[b] == len(r) and _same(rows[b, : len(r)], r)
    # the same instance at other positions, next to other neighbours and under a larger n_max: identical rows
    f, t = inst[5]
    big = rand_instance(rng, 700)
    for batch in ([(f, t)], [big, (f, t)], [inst[0], inst[2], (f, t), big]):
        out = dispatch.find_pool_pairs_batch(batch, D50)
        assert _same(out[[i for i, x in enumerate(batch) if x[0] is f][0]], res[5])
    # repeated calls are byte-identical
    again = dispatch.find_pool_pairs_batch(inst, D50)
    assert all(_same(a, b) for a, b in zip(again, res))


@pytest.mark.gpu
def test_table_entry_above_limit_withdraws_every_instance(td):
    from taxidispatcher_b200 import dispatch
    rng = np.random.default_rng(35)
    inst = [rand_instance(rng, n) for n in (0, 5, 40)]
    d = D50.copy()
    d[10, 11] = (1 << 22) + 1
    assert dispatch.find_pool_pairs_batch(inst, d) == [None, None, None]
    d[10, 11] = 1 << 22                                                # the limit itself is a valid entry
    for (f, t), rows in zip(inst, dispatch.find_pool_pairs_batch(inst, d)):
        assert np.array_equal(rows, pool_ref.pairs(f, t, d))


@pytest.mark.gpu
def test_pool_greedy_vs_optimum_two_launches(td):
    from taxidispatcher_b200 import _lib, dispatch
    lib = _lib.lib()
    rng = np.random.default_rng(36)
    inst = [rand_instance(rng, 100) for _ in range(1000)]
    ex.pool_greedy_vs_optimum(inst[:2], D50)                                    # warm the workspace and staging
    before = lib.td_launch_count()
    res = ex.pool_greedy_vs_optimum(inst, D50)
    assert lib.td_launch_count() - before == 2
    old = ex.pool_greedy_vs_optimum(inst, D50, greedy=dispatch.find_pool_pairs)
    assert res == old


class Recording:
    """Wraps a Simulator backend and keeps (frm, to, rows) of every pool step."""

    def __init__(self, inner):
        self.inner, self.pools = inner, []

    def pool_pairs(self, frm, to, dist):
        r = self.inner.pool_pairs(frm, to, dist)
        self.pools.append((np.array(frm), np.array(to), np.asarray(r).copy()))
        return r

    def __getattr__(self, name):
        return getattr(self.inner, name)


@pytest.mark.gpu
def test_simulator_replay_pools_in_one_batch(td):
    from taxidispatcher_b200 import formats
    from taxidispatcher_b200.simulator import MAX_LOSS, CudaBackend, Simulator
    demand = formats.read_taxi_demand(gzip.open(os.path.join(GOLDEN, "taxi_demand.txt.gz"), "rt").read())
    rec = Recording(CudaBackend())
    sim = Simulator(demand, backend=rec)
    sim.run(60)
    assert len(rec.pools) >= 50 and max(len(f) for f, _, _ in rec.pools) <= 1445
    res = td.find_pool_pairs_batch([(f, t) for f, t, _ in rec.pools], sim.dist, True, MAX_LOSS)
    for (f, t, rows), got in zip(rec.pools, res):
        assert _same(got, rows)
