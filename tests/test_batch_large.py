"""Batches of large instances (641 <= n <= 2048) on thread-block clusters that read the matrix from global memory:
td_assign_exact_batch_large / td_lcm_batch_large, the size routing of run_batch, and the batched experiments at the
reference's large sizes (heuristic.py's 2000 x 2000, the Simulator's 1300-row LCM model).

CPU: argument validation and the no-device return of the C ABI; the host-side grouping and minimum-batch rule.
GPU: ragged batches against scipy and the dual certificate; n <= 640 instances inside the large kernel bit for bit
against the DSMEM cluster and single-CTA kernels; independence from n_max / position / repetition; isolation and
withdrawal; every LCM variant against single td_lcm calls and the literal C oracle; Simulator-shaped 1300 x 1300
instances; routing by launch counts; split_hybrid_vs_optimum against the per-case flow."""
import ctypes

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from oracle import cost_ref, gen_inputs as g, lcm_ref

I32_MAX = 2**31 - 1
MAX_N = 2048
CLUSTER_N = 640
SMALL_N = 232
LCM_VARIANTS = {
    "heuristic": dict(mask_value=100),
    "split": dict(mask_value=g.BIG_COST, sum_below=g.BIG_COST),
    "greedy_opt": dict(mask_value=g.BIG_COST, stop_above=10, sum_below=g.BIG_COST),
    "java": dict(mask_value=g.BIG_COST, stop_at_value=g.BIG_COST, residual_size=20),
    "max_iters": dict(mask_value=100, max_iters=15),
    "mask_tail": dict(mask_value=45),
}


# ---- CPU: the C ABI refuses bad arguments before it looks for a device -----------------------------------------------
def _abi():
    from taxidispatcher_b200 import _lib
    return _lib, _lib.lib()


def _assign_call(lib, costs=16, sizes=32, offsets=48, batch=1, n_max=4, col=64, obj=80, u=None, v=None):
    p = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    return lib.td_assign_exact_batch_large(p(costs), p(sizes), p(offsets), batch, n_max, p(col), p(obj), p(u), p(v), None)


def _lcm_call(lib, _lib, costs=16, sizes=32, offsets=48, batch=1, n_max=4, params=True, rows=64, cols=80, npairs=96,
              total=112, last=None):
    p = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    prm = _lib.LcmParams(100, I32_MAX, I32_MAX, I32_MAX, 0, -1)
    return lib.td_lcm_batch_large(p(costs), p(sizes), p(offsets), batch, n_max, ctypes.byref(prm) if params else None,
                                  p(rows), p(cols), p(npairs), p(total), p(last), None)


def test_large_batch_abi_argument_validation():
    _lib, lib = _abi()
    INV = _lib.TD_ERR_INVALID
    assert _lib.BATCH_LARGE_MAX_N == MAX_N
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
        assert call(batch=0, n_max=MAX_N) == _lib.TD_OK
        assert call(batch=0, n_max=MAX_N + 1) == INV
    assert _assign_call(lib, col=None) == INV
    assert _assign_call(lib, obj=None) == INV
    assert _lcm_call(lib, _lib, params=False) == INV
    assert _lcm_call(lib, _lib, rows=None) == INV
    assert _lcm_call(lib, _lib, cols=None) == INV
    assert _lcm_call(lib, _lib, npairs=None) == INV
    assert _lcm_call(lib, _lib, total=None) == INV
    # the DSMEM cluster entry points keep their limit
    assert lib.td_assign_exact_batch_cluster(ctypes.c_void_p(16), ctypes.c_void_p(32), ctypes.c_void_p(48), 1,
                                             CLUSTER_N + 1, ctypes.c_void_p(64), ctypes.c_void_p(80), None, None,
                                             None) == INV
    assert lib.td_launch_count() == launches


def test_large_batch_abi_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    _lib, lib = _abi()
    launches = lib.td_launch_count()
    for n_max in (0, 232, 640, 641, 1024, 1025, MAX_N):
        assert _assign_call(lib, n_max=n_max) == _lib.TD_ERR_NO_DEVICE
        assert _lcm_call(lib, _lib, n_max=n_max) == _lib.TD_ERR_NO_DEVICE
    assert _assign_call(lib, u=96, v=112) == _lib.TD_ERR_NO_DEVICE
    assert _lcm_call(lib, _lib, last=128) == _lib.TD_ERR_NO_DEVICE
    assert lib.td_launch_count() == launches


def test_kernel_choice_by_n_max():
    from taxidispatcher_b200 import dispatch
    pick = dispatch.Engine._batch_kernel
    assert pick(232, "td_lcm_batch") == "td_lcm_batch"
    assert pick(233, "td_lcm_batch") == "td_lcm_batch_cluster"
    assert pick(640, "td_assign_exact_batch") == "td_assign_exact_batch_cluster"
    assert pick(641, "td_assign_exact_batch") == "td_assign_exact_batch_large"
    assert pick(MAX_N, "td_lcm_batch") == "td_lcm_batch_large"
    with pytest.raises(ValueError):
        pick(MAX_N + 1, "td_assign_exact_batch")


def test_batch_routes_groups_and_minimum_batches():
    from taxidispatcher_b200 import dispatch
    ns = [100, 300, 700, 2048, 2049, 5000, 641, 640, 0]
    assert dispatch.size_groups(ns) == ([0, 8], [1, 7], [2, 3, 6], [4, 5])
    la, ll = dispatch.ASSIGN_LARGE_MIN_BATCH, dispatch.LCM_LARGE_MIN_BATCH
    assert la >= 1 and ll >= 2                         # a lone large LCM: one whole-GPU td_lcm call
    for count in sorted({1, la - 1, la, ll - 1, ll, ll + 1} - {0}):
        ns = [700 + k for k in range(count)] + [3000]
        groups, single_a, single_l = dispatch.batch_routes(ns)
        large = list(range(count))
        want_a, want_l = count >= la, count >= ll
        assert groups == ([(large, want_a, want_l)] if want_a or want_l else []), count
        assert single_a == ([] if want_a else large) + [count]       # above 2048: always a single call
        assert single_l == ([] if want_l else large) + [count]
        groups, single_a, single_l = dispatch.batch_routes(ns, assign=True, lcm=False)
        assert groups == ([(large, True, False)] if want_a else []) and single_l == []
        groups, single_a, single_l = dispatch.batch_routes(ns, assign=False, lcm=True)
        assert groups == ([(large, False, True)] if want_l else []) and single_a == []
    # the smaller groups keep their rules
    groups, single_a, single_l = dispatch.batch_routes([10, 300, 300], assign=True, lcm=True)
    assert groups == [([0], True, True), ([1, 2], True, dispatch.LCM_CLUSTER_MIN_BATCH <= 2)]
    assert single_a == [] and single_l == ([] if dispatch.LCM_CLUSTER_MIN_BATCH <= 2 else [1, 2])


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


def _large_assign(eng, packed, sizes, offs, n_max):
    """td_assign_exact_batch_large at any n_max (Engine.assign_batch picks it above 640 only)"""
    import torch
    B = int(sizes.numel())
    col = torch.empty((B, max(n_max, 1)), dtype=torch.int32, device="cuda")
    obj = torch.empty(B, dtype=torch.int64, device="cuda")
    u = torch.empty((B, max(n_max, 1)), dtype=torch.int64, device="cuda")
    v = torch.empty((B, max(n_max, 1)), dtype=torch.int64, device="cuda")
    p = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731
    rc = eng.lib.td_assign_exact_batch_large(p(packed), p(sizes), p(offs), B, int(n_max), p(col), p(obj), p(u), p(v), None)
    assert rc == 0
    return [t.cpu().numpy() for t in (col, obj, u, v)]


def _large_lcm(eng, packed, sizes, offs, n_max, kw):
    import torch
    from taxidispatcher_b200 import _lib
    B = int(sizes.numel())
    rows = torch.empty((B, max(n_max, 1)), dtype=torch.int32, device="cuda")
    cols = torch.empty((B, max(n_max, 1)), dtype=torch.int32, device="cuda")
    npairs = torch.empty(B, dtype=torch.int32, device="cuda")
    total = torch.empty(B, dtype=torch.int64, device="cuda")
    last = torch.empty(B, dtype=torch.int32, device="cuda")
    prm = _lib.LcmParams(kw["mask_value"], kw.get("stop_above", I32_MAX), kw.get("stop_at_value", I32_MAX),
                         kw.get("sum_below", I32_MAX), kw.get("residual_size", 0), kw.get("max_iters", -1))
    p = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731
    rc = eng.lib.td_lcm_batch_large(p(packed), p(sizes), p(offs), B, int(n_max), ctypes.byref(prm), p(rows), p(cols),
                                    p(npairs), p(total), p(last), None)
    assert rc == 0
    return [t.cpu().numpy() for t in (rows, cols, npairs, total, last)]


def _check_certificate(c, col, obj, u, v):
    n = c.shape[0]
    c64 = c.astype(np.int64)
    assert sorted(col.tolist()) == list(range(n))
    assert int(obj) == int(c64[np.arange(n), col].sum())
    red = c64 - u[:, None] - v[None, :]
    assert red.min() >= 0 and (red[np.arange(n), col] == 0).all()
    assert int(u.sum() + v.sum()) == int(obj)


@pytest.mark.gpu
def test_large_assign_ragged_against_scipy_and_the_dual_certificate(td):
    dispatch, eng = _engine()
    rng = np.random.default_rng(641)
    dist = g.stand_distances(4000)
    sizes = [641, 700, 1024, 1025, 1300, 2000, 2048] + [int(s) for s in rng.integers(641, MAX_N + 1, 3)]
    cases = [_case(rng, n, k % 2, dist) for k, n in enumerate(sizes)]
    cases.append(g.config2_stand(2000))                  # greedy_opt.py's stand-derived config 2
    packed, sizes_d, offs, n_max = dispatch.pack_batch(cases)
    assert n_max == MAX_N
    l0 = eng.lib.td_launch_count()
    col, obj, u, v = [t.cpu().numpy() for t in eng.assign_batch(packed, sizes_d, offs, n_max, want_duals=True)]
    assert eng.lib.td_launch_count() == l0 + 1
    for b, c in enumerate(cases):
        n = c.shape[0]
        assert (col[b, n:] == -1).all() and (u[b, n:] == 0).all() and (v[b, n:] == 0).all()
        _check_certificate(c, col[b, :n], obj[b], u[b, :n], v[b, :n])
        if b in (0, 3, 5, len(cases) - 1):               # scipy on a subset (seconds per 2000 x 2000 instance)
            r, cc = linear_sum_assignment(c)
            assert int(obj[b]) == int(c.astype(np.int64)[r, cc].sum()), (b, n)


def _ragged_small(rng, dist):
    sizes = [0, 1, 2, 3, 31, 100, 232, 233, 300, 400, 600, 639, 640] + [int(s) for s in rng.integers(1, CLUSTER_N + 1, 5)]
    return [_case(rng, n, k % 4, dist) for k, n in enumerate(sizes)]


@pytest.mark.gpu
@pytest.mark.parametrize("n_max", [640, 1024, 1025, 2048])
def test_large_assign_small_instances_equal_the_cluster_and_single_cta_kernels(td, n_max):
    dispatch, eng = _engine()
    rng = np.random.default_rng(n_max)
    dist = g.stand_distances(300)
    cases = _ragged_small(rng, dist)
    packed, sizes, offs, nm = dispatch.pack_batch(cases)
    assert nm == CLUSTER_N
    ref = [t.cpu().numpy() for t in eng.assign_batch(packed, sizes, offs, nm, want_duals=True)]       # DSMEM cluster
    small = [c for c in cases if c.shape[0] <= SMALL_N]
    sp, ss, so, snm = dispatch.pack_batch(small)
    sref = [t.cpu().numpy() for t in eng.assign_batch(sp, ss, so, snm, want_duals=True)]              # one CTA each
    col, obj, u, v = _large_assign(eng, packed, sizes, offs, n_max)
    k = 0
    for b, c in enumerate(cases):
        n = c.shape[0]
        assert np.array_equal(col[b, :n], ref[0][b, :n]) and obj[b] == ref[1][b], (n_max, b, n)
        assert np.array_equal(u[b, :n], ref[2][b, :n]) and np.array_equal(v[b, :n], ref[3][b, :n]), (n_max, b, n)
        assert (col[b, n:] == -1).all() and (u[b, n:] == 0).all() and (v[b, n:] == 0).all()
        if n <= SMALL_N:
            assert np.array_equal(col[b, :n], sref[0][k, :n]) and obj[b] == sref[1][k]
            assert np.array_equal(u[b, :n], sref[2][k, :n]) and np.array_equal(v[b, :n], sref[3][k, :n])
            k += 1


@pytest.mark.gpu
def test_large_assign_is_independent_of_n_max_position_and_repetition(td):
    dispatch, eng = _engine()
    rng = np.random.default_rng(23)
    dist = g.stand_distances(4000)
    probe = [_case(rng, n, k, dist) for k, n in enumerate((700, 233, 1, 1300))]
    alone = []
    for c in probe:
        packed, sizes, offs, n_max = dispatch.pack_batch([c])
        alone.append(_large_assign(eng, packed, sizes, offs, n_max))
    for fn in (1024, 1025, 2048):               # K = 4 / 8 / 8, the probes at both ends
        filler = _case(rng, fn, 0, dist)
        for order in (probe + [filler], [filler] + probe[::-1]):
            packed, sizes, offs, n_max = dispatch.pack_batch(order)
            for rep in range(2):
                col, obj, u, v = _large_assign(eng, packed, sizes, offs, n_max)
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
def test_large_instances_are_isolated_and_bad_ones_withdrawn(td):
    dispatch, eng = _engine()
    rng = np.random.default_rng(31)
    dist = g.stand_distances(4000)
    cases = [_case(rng, n, k % 4, dist) for k, n in enumerate((0, 5, 700, 1500, 233, 1025, 2048, 900))]
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    kw = LCM_VARIANTS["heuristic"]
    ref = _large_assign(eng, packed, sizes, offs, n_max)
    ref_lcm = _large_lcm(eng, packed, sizes, offs, n_max, kw)
    ppacked, psizes, poffs, _ = _poisoned_pack(cases, [4 * int(k) for k in rng.integers(1, 9, len(cases))])
    for a, b in zip(ref, _large_assign(eng, ppacked, psizes, poffs, n_max)):
        assert np.array_equal(a, b)
    for a, b in zip(ref_lcm, _large_lcm(eng, ppacked, psizes, poffs, n_max, kw)):
        assert np.array_equal(a, b)
    # withdrawn: a size above n_max, an offset that is not a multiple of 4, a negative offset
    sizes2, offs2 = sizes.clone(), offs.clone()
    sizes2[2] = n_max + 1
    offs2[3] += 2
    offs2[5] = -4
    col, obj, u, v = _large_assign(eng, packed, sizes2, offs2, n_max)
    rows, cols, npairs, total, last = _large_lcm(eng, packed, sizes2, offs2, n_max, kw)
    for b in range(len(cases)):
        if b in (2, 3, 5):
            assert obj[b] == np.iinfo(np.int64).min and (col[b] == -1).all() and (u[b] == 0).all() and (v[b] == 0).all()
            assert npairs[b] == -1 and total[b] == np.iinfo(np.int64).min and last[b] == np.iinfo(np.int32).min
            assert (rows[b] == -1).all() and (cols[b] == -1).all()
        else:
            assert np.array_equal(col[b], ref[0][b]) and obj[b] == ref[1][b]
            assert np.array_equal(u[b], ref[2][b]) and np.array_equal(v[b], ref[3][b])
            assert npairs[b] == ref_lcm[2][b] and total[b] == ref_lcm[3][b] and last[b] == ref_lcm[4][b]
            assert np.array_equal(rows[b], ref_lcm[0][b]) and np.array_equal(cols[b], ref_lcm[1][b])


def _lcm_oracle(c, kw):
    return lcm_ref.lcm_c(c, kw["mask_value"], kw.get("stop_above", I32_MAX), kw.get("stop_at_value", I32_MAX),
                         kw.get("sum_below", I32_MAX), kw.get("residual_size", 0), kw.get("max_iters", -1))


def _assert_trace(rows, cols, npairs, total, last, want, what):
    k = want["n_pairs"]
    assert (npairs, total, last) == (k, want["total"], want["last_min"]), what
    assert np.array_equal(rows[:k], want["rows"]) and np.array_equal(cols[:k], want["cols"]), what
    assert (rows[k:] == -1).all() and (cols[k:] == -1).all(), what


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(LCM_VARIANTS))
def test_large_lcm_matches_single_td_lcm(td, variant):
    dispatch, eng = _engine()
    kw = LCM_VARIANTS[variant]
    rng = np.random.default_rng(77)
    dist = g.stand_distances(4000)
    cases = [_case(rng, n, k % 4, dist) for k, n in enumerate((641, 900, 1024, 1025, 1300, 2048, 1, 233, 600))]
    if variant == "mask_tail":                      # every cost >= the mask: masked cells win the argmin (trap 4)
        cases += [rng.integers(45, 60, (n, n)).astype(np.int32) for n in (700, 1500)] + [np.full((1100, 1100), 45, np.int32)]
        c = rng.integers(1, 40, (800, 800)).astype(np.int32)
        c[0, :] = 50                                # row 0 expensive: the (0, min masked column) pick
        cases.append(c)
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    rows, cols, npairs, total, last = [t.cpu().numpy() for t in eng.lcm_batch(packed, sizes, offs, n_max, **kw)]
    for b, c in enumerate(cases):
        want = dispatch.LCM(c.shape[0], c, **kw)
        _assert_trace(rows[b], cols[b], npairs[b], total[b], last[b], want, (variant, b, c.shape))


@pytest.mark.gpu
def test_large_lcm_near_2048_matches_the_literal_c_oracle(td):
    dispatch, eng = _engine()
    rng = np.random.default_rng(2047)
    cases = [g.config2(2000), rng.integers(1, 40, (2047, 2047)).astype(np.int32)]
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    for kw in (LCM_VARIANTS["heuristic"], LCM_VARIANTS["split"]):
        rows, cols, npairs, total, last = [t.cpu().numpy() for t in eng.lcm_batch(packed, sizes, offs, n_max, **kw)]
        for b, c in enumerate(cases):
            _assert_trace(rows[b], cols[b], npairs[b], total[b], last[b], _lcm_oracle(c, kw), (kw, b))


@pytest.mark.gpu
def test_large_lcm_simulator_shaped_instances(td):
    """1300 x 1300 matrices of Simulator.java's LCM model: 50 stands, cutoff 10, big_cost fill, residual 600"""
    dispatch, eng = _engine()
    rng = np.random.default_rng(1300)
    dist = g.stand_distances(50)
    insts = [(rng.integers(0, 50, nc), rng.integers(0, 50, 1300)) for nc in (1300, 1250, 1100, 1300, 700)]
    dist_d = dispatch._h2d_i32(dist)
    packed, sizes, offs, n_max, ns = dispatch.pack_cost_matrices(dist_d, insts, fill=g.BIG_COST, cutoff=10)
    assert n_max == 1300
    kw = dict(mask_value=g.BIG_COST, stop_at_value=g.BIG_COST, residual_size=600)
    rows, cols, npairs, total, last = [t.cpu().numpy() for t in eng.lcm_batch(packed, sizes, offs, n_max, **kw)]
    o = offs.cpu().numpy()
    for b, n in enumerate(ns):
        m = packed[int(o[b]): int(o[b]) + n * n].view(n, n)
        _, want = cost_ref.calculate_cost_np(dist, *insts[b], fill=g.BIG_COST, cutoff=10)
        assert np.array_equal(m.cpu().numpy(), want)
        single = dispatch.Engine.lcm_host_view(*eng.lcm(m, **kw))
        _assert_trace(rows[b], cols[b], npairs[b], total[b], last[b], single, b)
        assert single["n_pairs"] > 0


@pytest.mark.gpu
def test_run_batch_routes_large_instances(td):
    dispatch, eng = _engine()
    rng = np.random.default_rng(900)
    sizes = [100, 300, 700, 2100, 5, 1300] + [800 + k for k in range(max(dispatch.LCM_LARGE_MIN_BATCH,
                                                                          dispatch.ASSIGN_LARGE_MIN_BATCH))]
    cases = [rng.integers(1, 40, (n, n)).astype(np.int32) for n in sizes]
    lib = eng.lib

    def launches(fn):
        l0 = lib.td_launch_count()
        out = fn()
        return lib.td_launch_count() - l0, out

    ns = [c.shape[0] for c in cases]
    groups, single_a, single_l = dispatch.batch_routes(ns)
    assert groups == [([0, 4], True, True), ([1], True, False), ([2, 5] + list(range(6, len(ns))), True, True)]
    assert single_a == [3] and single_l == [1, 3]
    # assignment: one launch per size group (<= 232, 233-640, 641-2048), the 2100-row instance alone
    got_a, res = launches(lambda: dispatch.solve_batch(cases, want_duals=True))
    lone = launches(lambda: dispatch.solve_batch([cases[3]], want_duals=True))[0]
    assert got_a == 3 + lone
    for b in (0, 1, 2, 3, 5):
        c = cases[b]
        col, obj, u, v = res[b]
        r, cc = linear_sum_assignment(c)
        assert obj == int(c.astype(np.int64)[r, cc].sum())
        _check_certificate(c, col, obj, u, v)
    # LCM: the large group in one launch once it reaches LCM_LARGE_MIN_BATCH; the mid group alone is below its minimum
    for kw in (LCM_VARIANTS["heuristic"], LCM_VARIANTS["java"]):
        def singles(idx):
            l0 = lib.td_launch_count()
            for b in idx:
                dispatch.LCM(cases[b].shape[0], cases[b], **kw)
            return lib.td_launch_count() - l0
        got_l, res_l = launches(lambda: dispatch.LCM_batch(cases, **kw))
        assert got_l == 2 + singles(single_l)
        for b, c in enumerate(cases):
            want = dispatch.LCM(c.shape[0], c, **kw)
            assert (res_l[b]["n_pairs"], res_l[b]["total"], res_l[b]["last_min"]) == \
                (want["n_pairs"], want["total"], want["last_min"])
            assert np.array_equal(res_l[b]["rows"], want["rows"]) and np.array_equal(res_l[b]["cols"], want["cols"])
        # a lone large LCM goes through a single call
        got1, _ = launches(lambda: dispatch.LCM_batch([cases[2]], **kw))
        assert got1 == singles([2])


@pytest.mark.gpu
def test_lcm_vs_optimum_at_config2_size(td):
    """heuristic.py's experiment on 2000 x 2000 instances: the batched flow against single calls"""
    dispatch, eng = _engine()
    from taxidispatcher_b200 import experiments as ex
    rng = np.random.default_rng(2)
    cases = [g.config2(2000)] + [rng.integers(1, 40, (n, n)).astype(np.int32) for n in (2000, 1500, 1000, 700)]
    got = ex.lcm_vs_optimum(cases)
    for c, (lcm_total, opt) in zip(cases, got):
        assert lcm_total == dispatch.LCM(c.shape[0], c, mask_value=100)["total"]
        assert opt == int(eng.assign(dispatch._h2d_i32(c))[1].item()) and opt <= lcm_total


@pytest.mark.gpu
def test_split_hybrid_up_to_2048_rows_equals_the_per_case_flow(td):
    dispatch, eng = _engine()
    from oracle import assign_ref
    from taxidispatcher_b200 import experiments as ex
    dist = g.stand_distances(4000)
    rng = np.random.default_rng(56)
    cases = [(g.rand_list(rng, nd, 4000), g.rand_list(rng, nc, 4000))
             for nd, nc in ((700, 690), (1300, 1300), (2048, 2000), (300, 320), (1100, 900))]
    got = ex.split_hybrid_vs_optimum(dist, cases, threshold=10)

    def solver(distances, demand, cabs):
        n, cost = cost_ref.calculate_cost(distances, demand, cabs)
        if n == 0:
            return 0, [], 0
        cost = np.asarray(cost, dtype=np.int32)
        packed, sizes, offs, n_max = dispatch.pack_batch([cost])       # the batch kernel of the instance's size
        col = dispatch.run_packed(packed, sizes, offs, n_max, [n])[0][0][0]
        return n, assign_ref.x_from_cols(col), cost

    def lcm_greedy(n, c, threshold):
        return dispatch.LCM_greedy_opt(n, np.asarray(c, dtype=np.int32), threshold)

    for (demand, cabs), row in zip(cases, got):
        nn, opt, n2, hyb = ex.greedy_then_solve(dist, demand, cabs, threshold=10, solver=solver, lcm=lcm_greedy)
        split = ex.solve_split(len(dist), dist, demand, cabs, solver=solver)
        n, cost = cost_ref.calculate_cost(dist, demand, cabs)
        lcm_total = dispatch.LCM_split(n, np.ascontiguousarray(np.asarray(cost, dtype=np.int32).T))
        assert row == (opt, split, lcm_total, hyb, n2), len(demand)
