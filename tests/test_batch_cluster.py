"""Batches of mid-size instances (n <= 640) on thread-block clusters: td_assign_exact_batch_cluster /
td_lcm_batch_cluster, the size routing of run_batch, and the paper's split / hybrid experiment (PDF p.5-6, 1000 cases of
400 x 400 over 4000 stands) batched through split_hybrid_vs_optimum.

CPU: argument validation and the no-device return of the C ABI; split_hybrid_vs_optimum fed with oracles against the
per-case flow of tests/test_experiments.py.
GPU: ragged batches with K = 2, 4 and 8 CTAs per cluster against scipy, the dual certificate and (n <= 232) the
single-CTA batch kernel bit for bit; independence from n_max / position / repetition; isolation; every LCM variant
against the literal C oracle; routing; the paper's experiment at full size."""
import ctypes

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from oracle import assign_ref, cost_ref, gen_inputs as g, lcm_ref
from taxidispatcher_b200 import experiments as ex

I32_MAX = 2**31 - 1
MAX_N = 640
SMALL_N = 232
# the published means over 1000 cases and their tolerances (as in tests/test_experiments.py)
PAPER = {"split": (1.16, 0.04), "lcm": (1.20, 0.04), "best": (1.14, 0.04), "hybrid": (1.024, 0.008), "n2": (146, 10)}


# ---- CPU: the C ABI refuses bad arguments before it looks for a device -----------------------------------------------
def _abi():
    from taxidispatcher_b200 import _lib
    return _lib, _lib.lib()


def _assign_call(lib, costs=16, sizes=32, offsets=48, batch=1, n_max=4, col=64, obj=80, u=None, v=None):
    p = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    return lib.td_assign_exact_batch_cluster(p(costs), p(sizes), p(offsets), batch, n_max, p(col), p(obj), p(u), p(v), None)


def _lcm_call(lib, _lib, costs=16, sizes=32, offsets=48, batch=1, n_max=4, params=True, rows=64, cols=80, npairs=96,
              total=112, last=None):
    p = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    prm = _lib.LcmParams(100, I32_MAX, I32_MAX, I32_MAX, 0, -1)
    return lib.td_lcm_batch_cluster(p(costs), p(sizes), p(offsets), batch, n_max, ctypes.byref(prm) if params else None,
                                    p(rows), p(cols), p(npairs), p(total), p(last), None)


def test_cluster_batch_abi_argument_validation():
    _lib, lib = _abi()
    INV = _lib.TD_ERR_INVALID
    launches = lib.td_launch_count()
    for call in (lambda **kw: _assign_call(lib, **kw), lambda **kw: _lcm_call(lib, _lib, **kw)):
        assert call(batch=-1) == INV
        assert call(n_max=-1) == INV
        assert call(n_max=MAX_N + 1) == INV
        assert call(costs=20) == INV                       # costs must be 16-byte aligned
        assert call(costs=None) == INV
        assert call(sizes=None) == INV
        assert call(offsets=None) == INV
        assert call(batch=0, costs=None, sizes=None, offsets=None) == _lib.TD_OK   # nothing to do, nothing launched
        assert call(batch=0, n_max=MAX_N + 1) == INV
    assert _assign_call(lib, col=None) == INV
    assert _assign_call(lib, obj=None) == INV
    assert _lcm_call(lib, _lib, params=False) == INV
    assert _lcm_call(lib, _lib, rows=None) == INV
    assert _lcm_call(lib, _lib, cols=None) == INV
    assert _lcm_call(lib, _lib, npairs=None) == INV
    assert _lcm_call(lib, _lib, total=None) == INV
    assert lib.td_launch_count() == launches
    # the single-CTA entry points keep their limit
    assert lib.td_assign_exact_batch(ctypes.c_void_p(16), ctypes.c_void_p(32), ctypes.c_void_p(48), 1, SMALL_N + 1,
                                     ctypes.c_void_p(64), ctypes.c_void_p(80), None, None, None) == INV


def test_cluster_batch_abi_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    _lib, lib = _abi()
    launches = lib.td_launch_count()
    for n_max in (0, 232, 233, 400, MAX_N):
        assert _assign_call(lib, n_max=n_max) == _lib.TD_ERR_NO_DEVICE
        assert _lcm_call(lib, _lib, n_max=n_max) == _lib.TD_ERR_NO_DEVICE
    assert _assign_call(lib, u=96, v=112) == _lib.TD_ERR_NO_DEVICE
    assert _lcm_call(lib, _lib, last=128) == _lib.TD_ERR_NO_DEVICE
    assert lib.td_launch_count() == launches


# ---- the paper's split / hybrid experiment: batched flow == per-case flow ---------------------------------------------
def oracle_solver(distances, demand, cabs):
    n, cost = cost_ref.calculate_cost(distances, demand, cabs)
    if n == 0:
        return 0, [], 0
    _, col = assign_ref.solve_scipy(np.asarray(cost))
    return n, assign_ref.x_from_cols(col), np.asarray(cost)


def oracle_lcm_greedy(n, c, threshold):
    tot, sup, dem = lcm_ref.lcm_greedy_opt(n, c, threshold)
    return int(tot), sup, dem


def oracle_solver_batch(costs):
    out = []
    for c in costs:
        c = np.asarray(c)
        _, col = assign_ref.solve_scipy(c)
        col = np.asarray(col, dtype=np.int32)
        out.append((col, int(c.astype(np.int64)[np.arange(len(col)), col].sum())))
    return out


def _lcm_oracle(c, kw):
    return lcm_ref.lcm_c(c, kw["mask_value"], kw.get("stop_above", I32_MAX), kw.get("stop_at_value", I32_MAX),
                         kw.get("sum_below", I32_MAX), kw.get("residual_size", 0), kw.get("max_iters", -1))


def oracle_lcm_batch(costs, **kw):
    return [_lcm_oracle(np.asarray(c, dtype=np.int32), kw) for c in costs]


def paper_cases(count, seed=56, n_size=400, n_stands=4000):
    rng = np.random.default_rng(seed)
    return [(g.rand_list(rng, n_size, n_stands), g.rand_list(rng, n_size, n_stands)) for _ in range(count)]


def per_case_flow(dist, demand, cabs, threshold=10):
    """what tests/test_experiments.py::degradation_statistics computes for one case, with the oracles"""
    nn, opt, n2, hyb = ex.greedy_then_solve(dist, demand, cabs, threshold=threshold, solver=oracle_solver,
                                            lcm=oracle_lcm_greedy)
    split = ex.solve_split(len(dist), dist, demand, cabs, solver=oracle_solver)
    n, cost = cost_ref.calculate_cost(dist, demand, cabs)
    lcm_total = int(lcm_ref.lcm_split(n, np.asarray(cost).T)[0])
    return opt, split, lcm_total, hyb, n2


def test_split_hybrid_batched_equals_the_per_case_flow_cpu():
    dist = g.stand_distances(4000)
    cases = paper_cases(10)
    got = ex.split_hybrid_vs_optimum(dist, cases, threshold=10, solver_batch=oracle_solver_batch,
                                     lcm_batch=oracle_lcm_batch)
    assert len(got) == len(cases)
    for (demand, cabs), row in zip(cases, got):
        assert row == per_case_flow(dist, demand, cabs)


def test_split_hybrid_small_shapes_cpu():
    """unbalanced cases, ranges with one side only, tiny sizes: still the per-case flow"""
    dist = g.stand_distances(40)
    rng = np.random.default_rng(8)
    cases = [(g.rand_list(rng, nd, 40), g.rand_list(rng, nc, 40)) for nd, nc in ((30, 20), (5, 50), (60, 60), (3, 2))]
    cases.append(([(0, 1, 2), (1, 12, 3)], [(0, 2, 35), (1, 3, 36), (2, 4, 37)]))      # ranges with one side only
    got = ex.split_hybrid_vs_optimum(dist, cases, threshold=3, solver_batch=oracle_solver_batch,
                                     lcm_batch=oracle_lcm_batch)
    for (demand, cabs), row in zip(cases, got):
        assert row == per_case_flow(dist, demand, cabs, threshold=3)


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _engine():
    from taxidispatcher_b200 import dispatch
    return dispatch, dispatch.engine()


def _case(rng, n, kind, dist):
    if kind == 0:
        c = rng.integers(1, 40, (n, n))
    elif kind == 1 and n > 1:                    # stand-derived with big_cost padding rows (fewer cabs than customers)
        n_cabs = max(1, n - 1 - int(rng.integers(0, max(1, n // 10))))
        _, c = cost_ref.calculate_cost_np(dist, rng.integers(0, len(dist), n_cabs), rng.integers(0, len(dist), n))
    elif kind == 2:
        c = rng.integers(0, 3, (n, n))           # many ties
    else:
        c = rng.integers(-2**30, 2**30, (n, n))
    return np.ascontiguousarray(c, dtype=np.int32)


def _ragged(n_max, seed):
    rng = np.random.default_rng(seed)
    dist = g.stand_distances(300)
    sizes = [0, 1, 2, 3, 31, 100, 232, 233, n_max] + [int(s) for s in rng.integers(1, n_max + 1, 9)]
    if n_max == MAX_N:
        sizes += [400, 600, 639]
    return [_case(rng, n, k % 4, dist) for k, n in enumerate(sizes)]


def _run_assign(eng, packed, sizes, offs, n_max):
    return [t.cpu().numpy() for t in eng.assign_batch(packed, sizes, offs, n_max, want_duals=True)]


def _small_reference(dispatch, eng, cases):
    """td_assign_exact_batch (one CTA per instance) on the instances up to 232"""
    small = [c for c in cases if c.shape[0] <= SMALL_N]
    packed, sizes, offs, n_max = dispatch.pack_batch(small)
    return small, _run_assign(eng, packed, sizes, offs, n_max)


@pytest.mark.gpu
@pytest.mark.parametrize("n_max", [300, 400, 640])
def test_cluster_assign_ragged_against_scipy_duals_and_the_small_kernel(td, n_max):
    dispatch, eng = _engine()
    cases = _ragged(n_max, n_max)
    packed, sizes, offs, nm = dispatch.pack_batch(cases)
    assert nm == n_max
    lib = eng.lib
    l0 = lib.td_launch_count()
    col, obj, u, v = _run_assign(eng, packed, sizes, offs, nm)
    assert lib.td_launch_count() == l0 + 1
    small, (scol, sobj, su, sv) = _small_reference(dispatch, eng, cases)
    k = 0
    for b, c in enumerate(cases):
        n = c.shape[0]
        assert (col[b, n:] == -1).all() and (u[b, n:] == 0).all() and (v[b, n:] == 0).all()
        if n == 0:
            assert obj[b] == 0
        else:
            cb, ub, vb = col[b, :n], u[b, :n], v[b, :n]
            r, cc = linear_sum_assignment(c)
            want = int(c.astype(np.int64)[r, cc].sum())
            assert int(obj[b]) == want, (n_max, b, n)
            assert sorted(cb.tolist()) == list(range(n))
            red = c.astype(np.int64) - ub[:, None] - vb[None, :]
            assert red.min() >= 0 and (red[np.arange(n), cb] == 0).all()
            assert int(ub.sum() + vb.sum()) == want == int(c.astype(np.int64)[np.arange(n), cb].sum())
        if n <= SMALL_N:                                    # the same algorithm as the single-CTA kernel, bit for bit
            assert np.array_equal(col[b, :n], scol[k, :n]) and obj[b] == sobj[k], (n_max, b, n)
            assert np.array_equal(u[b, :n], su[k, :n]) and np.array_equal(v[b, :n], sv[k, :n]), (n_max, b, n)
            k += 1


@pytest.mark.gpu
def test_cluster_assign_kats_inside_a_k8_batch(td, golden):
    dispatch, eng = _engine()
    gold = golden("assign.json")
    a1 = np.array(gold["A1_python_py"]["cost"], dtype=np.int32).reshape(4, 4)        # python.py:7
    a3 = np.array(gold["A3_procedure_py"]["cost"], dtype=np.int32)                   # procedure.py
    a3 = a3.reshape(int(round(a3.size ** 0.5)), -1)
    rng = np.random.default_rng(3)
    cases = [rng.integers(1, 40, (640, 640)).astype(np.int32), a1, rng.integers(1, 40, (500, 500)).astype(np.int32), a3]
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    col, obj, _, _ = eng.assign_batch(packed, sizes, offs, n_max)
    col, obj = col.cpu().numpy(), obj.cpu().numpy()
    assert int(obj[1]) == 101 and int(obj[3]) == 17
    assert col[1, :4].tolist() in gold["A1_python_py"]["optimal_perms"]
    for b in (0, 2):
        assert int(obj[b]) == assign_ref.solve_scipy(cases[b])[0]


@pytest.mark.gpu
def test_cluster_assign_is_independent_of_n_max_position_and_repetition(td):
    dispatch, eng = _engine()
    rng = np.random.default_rng(17)
    dist = g.stand_distances(300)
    probe = [_case(rng, n, k, dist) for k, n in enumerate((237, 180, 1, 233))]
    alone = []
    for c in probe:
        packed, sizes, offs, n_max = dispatch.pack_batch([c])
        alone.append(_run_assign(eng, packed, sizes, offs, n_max))
    fillers = [_case(rng, n, 0, dist) for n in (240, 400, 640)]
    for filler in fillers:                      # n_max 240 / 400 / 640 (K = 2 / 4 / 8), the probes at both ends
        for order in (probe + [filler], [filler] + probe[::-1]):
            packed, sizes, offs, n_max = dispatch.pack_batch(order)
            for rep in range(2):
                col, obj, u, v = _run_assign(eng, packed, sizes, offs, n_max)
                for b, c in enumerate(order):
                    if c is filler:
                        continue
                    a = alone[[id(x) for x in probe].index(id(c))]
                    n = c.shape[0]
                    assert np.array_equal(col[b, :n], a[0][0, :n]) and obj[b] == a[1][0], (n_max, n, rep)
                    assert np.array_equal(u[b, :n], a[2][0, :n]) and np.array_equal(v[b, :n], a[3][0, :n]), (n_max, n)


def _poisoned_pack(cases, gaps):
    import torch
    chunks, offsets, pos = [], [], 0
    for c, gap in zip(cases, gaps):
        chunks.append(np.full(gap, np.iinfo(np.int32).min, np.int32))
        pos += gap
        offsets.append(pos)
        flat = np.ascontiguousarray(c, dtype=np.int32).reshape(-1)
        pad = (-flat.size) % 4
        chunks.append(np.concatenate([flat, np.full(pad, np.iinfo(np.int32).min, np.int32)]))
        pos += flat.size + pad
    chunks.append(np.full(8, np.iinfo(np.int32).min, np.int32))
    packed = torch.from_numpy(np.concatenate(chunks)).cuda()
    sizes = torch.tensor([c.shape[0] for c in cases], dtype=torch.int32, device="cuda")
    offs = torch.tensor(offsets, dtype=torch.int64, device="cuda")
    return packed, sizes, offs, max(c.shape[0] for c in cases)


@pytest.mark.gpu
def test_cluster_instances_are_isolated_and_bad_ones_withdrawn(td):
    dispatch, eng = _engine()
    cases = _ragged(MAX_N, 11)
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    ref = _run_assign(eng, packed, sizes, offs, n_max)
    ref_lcm = [t.cpu().numpy() for t in eng.lcm_batch(packed, sizes, offs, n_max, mask_value=100)]
    rng = np.random.default_rng(5)
    ppacked, psizes, poffs, _ = _poisoned_pack(cases, [4 * int(k) for k in rng.integers(1, 9, len(cases))])
    got = _run_assign(eng, ppacked, psizes, poffs, n_max)
    for a, b in zip(ref, got):
        assert np.array_equal(a, b)
    for a, b in zip(ref_lcm, [t.cpu().numpy() for t in eng.lcm_batch(ppacked, psizes, poffs, n_max, mask_value=100)]):
        assert np.array_equal(a, b)
    # withdrawn: a size above n_max and an offset that is not a multiple of 4
    sizes2, offs2 = sizes.clone(), offs.clone()
    sizes2[1] = n_max + 1
    offs2[4] += 2
    col, obj, u, v = _run_assign(eng, packed, sizes2, offs2, n_max)
    rows, cols, npairs, total, last = [t.cpu().numpy() for t in eng.lcm_batch(packed, sizes2, offs2, n_max, mask_value=100)]
    for b in range(len(cases)):
        if b in (1, 4):
            assert obj[b] == np.iinfo(np.int64).min and (col[b] == -1).all() and (u[b] == 0).all() and (v[b] == 0).all()
            assert npairs[b] == -1 and total[b] == np.iinfo(np.int64).min and last[b] == np.iinfo(np.int32).min
            assert (rows[b] == -1).all() and (cols[b] == -1).all()
        else:
            assert np.array_equal(col[b], ref[0][b]) and obj[b] == ref[1][b]
            assert np.array_equal(u[b], ref[2][b]) and np.array_equal(v[b], ref[3][b])
            assert npairs[b] == ref_lcm[2][b] and total[b] == ref_lcm[3][b] and np.array_equal(rows[b], ref_lcm[0][b])


@pytest.mark.gpu
def test_cluster_many_waves_one_launch_each(td):
    """600 instances of 400 x 400 (K = 4: 2400 CTAs, several waves) against the single-instance calls"""
    dispatch, eng = _engine()
    rng = np.random.default_rng(2000)
    cases = [rng.integers(1, 40, (400, 400)).astype(np.int32) for _ in range(600)]
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    lib = eng.lib
    l0 = lib.td_launch_count()
    col, obj, _, _ = eng.assign_batch(packed, sizes, offs, n_max)
    assert lib.td_launch_count() == l0 + 1
    lcm = eng.lcm_batch(packed, sizes, offs, n_max, mask_value=100)
    assert lib.td_launch_count() == l0 + 2
    obj = obj.cpu().numpy()
    col = col.cpu().numpy()
    rows, totals = lcm[0].cpu().numpy(), lcm[3].cpu().numpy()
    offs = offs.cpu().numpy()
    for b in range(0, len(cases), 7):
        d = packed[offs[b]: offs[b] + 160000].view(400, 400)
        _, sobj = eng.assign(d)[:2]
        r = dispatch.Engine.lcm_host_view(*eng.lcm(d, 100))
        assert int(obj[b]) == int(sobj.item()), b
        assert sorted(col[b].tolist()) == list(range(400))
        assert int(totals[b]) == r["total"] and np.array_equal(rows[b, :r["n_pairs"]], r["rows"]), b


LCM_VARIANTS = {
    "heuristic": dict(mask_value=100),
    "split": dict(mask_value=g.BIG_COST, sum_below=g.BIG_COST),
    "greedy_opt": dict(mask_value=g.BIG_COST, stop_above=10, sum_below=g.BIG_COST),
    "java": dict(mask_value=g.BIG_COST, stop_at_value=g.BIG_COST, residual_size=20),
    "max_iters": dict(mask_value=100, max_iters=15),
    "mask_tail": dict(mask_value=45),
}


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(LCM_VARIANTS))
def test_cluster_lcm_matches_the_literal_algorithm(td, variant):
    dispatch, eng = _engine()
    kw = LCM_VARIANTS[variant]
    cases = _ragged(MAX_N, 21)
    rng = np.random.default_rng(22)
    if variant == "mask_tail":                      # every cost >= the mask: masked cells win the argmin (trap 4)
        cases += [rng.integers(45, 60, (n, n)).astype(np.int32) for n in (1, 3, 240, 401)] + [np.full((300, 300), 45, np.int32)]
        c = rng.integers(1, 40, (500, 500)).astype(np.int32)
        c[0, :] = 50                                # row 0 expensive: the (0, min masked column) pick
        cases.append(c)
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    rows, cols, npairs, total, last = [t.cpu().numpy() for t in eng.lcm_batch(packed, sizes, offs, n_max, **kw)]
    for b, c in enumerate(cases):
        o = _lcm_oracle(c, kw)
        k = o["n_pairs"]
        assert npairs[b] == k and total[b] == o["total"] and last[b] == o["last_min"], (variant, b, c.shape)
        assert np.array_equal(rows[b, :k], o["rows"]) and np.array_equal(cols[b, :k], o["cols"]), (variant, b)
        assert (rows[b, k:] == -1).all() and (cols[b, k:] == -1).all()
        if c.shape[0] > SMALL_N and b % 3 == 0:     # and the single-instance kernel
            s = dispatch.LCM(c.shape[0], c, **kw)
            assert s["n_pairs"] == k and s["total"] == o["total"] and np.array_equal(s["rows"], o["rows"])


@pytest.mark.gpu
def test_run_batch_routes_by_size(td):
    dispatch, eng = _engine()
    rng = np.random.default_rng(300)
    sizes = (700, 12, 400, 233, 0, 640)
    cases = [rng.integers(1, 40, (n, n)).astype(np.int32) for n in sizes]
    lib = eng.lib
    l0 = lib.td_launch_count()
    res = dispatch.solve_batch(cases, want_duals=True)
    launched = lib.td_launch_count() - l0
    l1 = lib.td_launch_count()
    dispatch.solve_batch([cases[0]], want_duals=True)
    single = lib.td_launch_count() - l1
    assert launched == 2 + single                       # one launch for {12, 0}, one for {400, 233, 640}, 700 alone
    for c, (col, obj, u, v) in zip(cases, res):
        n = c.shape[0]
        assert obj == (assign_ref.solve_scipy(c)[0] if n else 0)
        assert sorted(col.tolist()) == list(range(n)) and len(u) == n and len(v) == n
        if n:
            red = c.astype(np.int64) - u[:, None] - v[None, :]
            assert red.min() >= 0 and int(u.sum() + v.sum()) == obj
    more = cases + [rng.integers(1, 40, (n, n)).astype(np.int32) for n in (300, 500)]    # 5 mid-size instances
    assert dispatch.LCM_CLUSTER_MIN_BATCH > 3 and dispatch.LCM_CLUSTER_MIN_BATCH <= 5
    for kw in (LCM_VARIANTS["heuristic"], LCM_VARIANTS["java"]):
        def single_launches(cs):
            l1 = lib.td_launch_count()
            for c in cs:
                dispatch.LCM(c.shape[0], c, **kw)
            return lib.td_launch_count() - l1
        l0 = lib.td_launch_count()
        got = dispatch.LCM_batch(cases, **kw)
        launched = lib.td_launch_count() - l0
        # one launch for {12, 0}; three mid-size instances are fewer than LCM_CLUSTER_MIN_BATCH: single calls
        assert launched == 1 + single_launches([c for c in cases if c.shape[0] > SMALL_N])
        l0 = lib.td_launch_count()
        got_more = dispatch.LCM_batch(more, **kw)
        assert lib.td_launch_count() - l0 == 2 + single_launches([cases[0]])      # {12, 0}, one cluster launch, 700
        for c, r in zip(more, got_more):
            o = _lcm_oracle(c, kw)
            assert r["n_pairs"] == o["n_pairs"] and r["total"] == o["total"] and np.array_equal(r["rows"], o["rows"])
        for c, r in zip(cases, got):
            o = _lcm_oracle(c, kw)
            assert r["n_pairs"] == o["n_pairs"] and r["total"] == o["total"] and r["last_min"] == o["last_min"]
            assert np.array_equal(r["rows"], o["rows"]) and np.array_equal(r["cols"], o["cols"])


@pytest.mark.gpu
def test_pack_cost_matrices_equals_calculate_cost(td):
    import torch
    dispatch, eng = _engine()
    rng = np.random.default_rng(12)
    dist = g.stand_distances(4000)
    dist[rng.integers(0, 4000, 50), rng.integers(0, 4000, 50)] += 7          # not symmetric
    insts = [(rng.integers(0, 4000, nc), rng.integers(0, 4000, nd)) for nc, nd in ((400, 400), (3, 5), (0, 4), (233, 200))]
    dist_d = dispatch._h2d_i32(dist)
    for transpose in (False, True):
        packed, sizes, offs, n_max, ns = dispatch.pack_cost_matrices(dist_d.t().contiguous() if transpose else dist_d, insts,
                                                                     transpose=transpose)
        assert ns == [400, 5, 4, 233] and n_max == 400 and sizes.cpu().tolist() == ns
        p, o = packed.cpu().numpy(), offs.cpu().numpy()
        for b, (c, d) in enumerate(insts):
            n = ns[b]
            _, want = cost_ref.calculate_cost_np(dist, c, d)
            got = p[o[b]: o[b] + n * n].reshape(n, n)
            assert np.array_equal(got, want.T if transpose else want), (b, transpose)
    assert torch.cuda.is_available()


@pytest.mark.gpu
def test_split_hybrid_paper_experiment_at_full_size(td):
    """1000 cases of 400 x 400 over 4000 stands, threshold 10 (PDF p.5-6).  Optimum, LCM-split, hybrid and n2 are unique
    and equal the oracle flow case by case (first 100 cases); split depends on which optimum a range solve returns and is
    checked statistically and against the optimum."""
    dist = g.stand_distances(4000)
    cases = paper_cases(1000)
    got = ex.split_hybrid_vs_optimum(dist, cases, threshold=10)
    assert len(got) == 1000
    ref = ex.split_hybrid_vs_optimum(dist, cases[:100], threshold=10, solver_batch=oracle_solver_batch,
                                     lcm_batch=oracle_lcm_batch)
    for a, b in zip(got[:100], ref):
        assert (a[0], a[2], a[3], a[4]) == (b[0], b[2], b[3], b[4])
    for opt, split, lcm_total, hyb, n2 in got:
        assert split >= opt and lcm_total >= opt and hyb >= opt
    stats = {"split": np.mean([r[1] / r[0] for r in got]), "lcm": np.mean([r[2] / r[0] for r in got]),
             "best": np.mean([min(r[1], r[2]) / r[0] for r in got]), "hybrid": np.mean([r[3] / r[0] for r in got]),
             "n2": np.mean([r[4] for r in got])}
    for k, (want, tol) in PAPER.items():
        assert abs(stats[k] - want) <= tol, (k, stats[k], want)
