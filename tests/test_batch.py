"""Batches of small independent instances: td_assign_exact_batch / td_lcm_batch (one CTA per instance, one launch per
call), the dispatch helpers on top of them, and the heuristic.py:20-40 experiment (LCM against the optimum on 1000
random 100 x 100 cases; the paper, p.4, reports LCM 78 % above the optimum).

CPU: argument validation and the no-device return of the C ABI, and lcm_vs_optimum fed with the oracles.
GPU: every instance against scipy / the single-instance solver / the literal LCM oracle, isolation between instances,
withdrawn instances, more than one wave of CTAs, and the mixed path for instances above TD_BATCH_MAX_N."""
import ctypes

import numpy as np
import pytest
from scipy.optimize import linear_sum_assignment

from oracle import assign_ref, cost_ref, gen_inputs as g, lcm_ref
from taxidispatcher_b200 import experiments as ex

I32_MAX = 2**31 - 1
MAX_N = 232


# ---- CPU: the C ABI refuses bad arguments before it looks for a device -----------------------------------------------
def _abi():
    from taxidispatcher_b200 import _lib
    return _lib, _lib.lib()


def _assign_call(lib, costs=16, sizes=32, offsets=48, batch=1, n_max=4, col=64, obj=80, u=None, v=None):
    p = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    return lib.td_assign_exact_batch(p(costs), p(sizes), p(offsets), batch, n_max, p(col), p(obj), p(u), p(v), None)


def _lcm_call(lib, _lib, costs=16, sizes=32, offsets=48, batch=1, n_max=4, params=True, rows=64, cols=80, npairs=96,
              total=112, last=None):
    p = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    prm = _lib.LcmParams(100, I32_MAX, I32_MAX, I32_MAX, 0, -1)
    return lib.td_lcm_batch(p(costs), p(sizes), p(offsets), batch, n_max, ctypes.byref(prm) if params else None, p(rows),
                            p(cols), p(npairs), p(total), p(last), None)


def test_batch_abi_argument_validation():
    _lib, lib = _abi()
    INV = _lib.TD_ERR_INVALID
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


def test_batch_abi_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    _lib, lib = _abi()
    launches = lib.td_launch_count()
    assert _assign_call(lib, n_max=MAX_N) == _lib.TD_ERR_NO_DEVICE
    assert _assign_call(lib, u=96, v=112) == _lib.TD_ERR_NO_DEVICE
    assert _lcm_call(lib, _lib, n_max=0) == _lib.TD_ERR_NO_DEVICE
    assert _lcm_call(lib, _lib, last=128) == _lib.TD_ERR_NO_DEVICE
    assert lib.td_launch_count() == launches


# ---- CPU: heuristic.py:20-40 with the oracles --------------------------------------------------------------------------
def heuristic_cases(seed, cases=1000, n=100):
    rng = np.random.default_rng(seed)
    return [rng.integers(1, 40, (n, n)).astype(np.int32) for _ in range(cases)]


def oracle_solver_batch(costs):
    out = []
    for c in costs:
        r, col = linear_sum_assignment(c)
        out.append((col.astype(np.int32), int(np.asarray(c)[r, col].sum())))
    return out


def oracle_lcm_batch(costs):
    return [lcm_ref.lcm_c(c, 100) for c in costs]


def test_lcm_vs_optimum_matches_the_paper_cpu():
    res = ex.lcm_vs_optimum(heuristic_cases(24), solver_batch=oracle_solver_batch, lcm_batch=oracle_lcm_batch)
    assert len(res) == 1000
    assert all(opt <= lcm for lcm, opt in res)              # heuristic.py:40
    ratio = float(np.mean([lcm / opt for lcm, opt in res]))
    assert abs(ratio - 1.78) <= 0.02, ratio                 # PDF p.4: LCM is 78 % worse than the optimum


# ---- GPU ---------------------------------------------------------------------------------------------------------------
def _ragged_cases(seed=7):
    """U[1,39], stand-derived with big_cost padding rows, all-equal and +-2^30 costs over sizes 0..232"""
    rng = np.random.default_rng(seed)
    sizes = [0, 1, 2, 3, 31, 32, 33, 100, 200, 232] + [int(s) for s in rng.integers(1, MAX_N + 1, 14)]
    dist = g.stand_distances(50)
    cases = []
    for k, n in enumerate(sizes):
        kind = k % 4
        if kind == 0:
            c = rng.integers(1, 40, (n, n))
        elif kind == 1 and n > 1:                       # gen_inputs.config1b shape: fewer cabs than customers
            n_cabs = max(1, n - 1 - int(rng.integers(0, max(1, n // 10))))
            _, c = cost_ref.calculate_cost_np(dist, rng.integers(0, 50, n_cabs), rng.integers(0, 50, n))
        elif kind == 2:
            c = np.full((n, n), 7)
        else:
            c = rng.integers(-2**30, 2**30, (n, n))
        cases.append(np.ascontiguousarray(c, dtype=np.int32))
    return cases


def _engine(td):
    from taxidispatcher_b200 import dispatch
    return dispatch, dispatch.engine()


def _assign_all(td, costs, want_duals=True):
    dispatch, eng = _engine(td)
    packed, sizes, offsets, n_max = dispatch.pack_batch(costs)
    col, obj, u, v = eng.assign_batch(packed, sizes, offsets, n_max, want_duals=want_duals)
    return (col.cpu().numpy(), obj.cpu().numpy(), None if u is None else u.cpu().numpy(),
            None if v is None else v.cpu().numpy())


def _single_col(eng, c):
    import torch
    col, obj, _, _ = eng.assign(torch.from_numpy(np.ascontiguousarray(c, dtype=np.int32)).cuda())
    return col.cpu().numpy(), int(obj.item())


@pytest.mark.gpu
def test_assign_batch_ragged_against_scipy_single_path_and_duals(td):
    dispatch, eng = _engine(td)
    cases = _ragged_cases()
    col, obj, u, v = _assign_all(td, cases)
    n_max = max(c.shape[0] for c in cases)
    assert col.shape == (len(cases), n_max)
    for b, c in enumerate(cases):
        n = c.shape[0]
        assert (col[b, n:] == -1).all() and (u[b, n:] == 0).all() and (v[b, n:] == 0).all()
        if n == 0:
            assert obj[b] == 0
            continue
        cb, ub, vb = col[b, :n], u[b, :n].astype(np.int64), v[b, :n].astype(np.int64)
        assert int(obj[b]) == assign_ref.solve_scipy(c)[0], (b, n)
        assert sorted(cb.tolist()) == list(range(n))
        scol, sobj = _single_col(eng, c)
        assert np.array_equal(cb, scol) and sobj == int(obj[b]), (b, n)      # the very same routine
        su, sv = eng.assign_duals(n)
        assert np.array_equal(ub, su.cpu().numpy()) and np.array_equal(vb, sv.cpu().numpy()), (b, n)
        red = c.astype(np.int64) - ub[:, None] - vb[None, :]
        assert red.min() >= 0 and (red[np.arange(n), cb] == 0).all()
        assert int(ub.sum() + vb.sum()) == int(obj[b]) == int(c.astype(np.int64)[np.arange(n), cb].sum())


@pytest.mark.gpu
def test_assign_batch_kats_inside_a_batch(td, golden):
    gold = golden("assign.json")
    a1 = np.array(gold["A1_python_py"]["cost"], dtype=np.int32).reshape(4, 4)        # python.py:7
    a3 = np.array(gold["A3_procedure_py"]["cost"], dtype=np.int32)                   # procedure.py
    a3 = a3.reshape(int(round(a3.size ** 0.5)), -1)
    rng = np.random.default_rng(3)
    cases = [rng.integers(1, 40, (50, 50)), a1, rng.integers(0, 3, (17, 17)), a3, rng.integers(1, 40, (5, 5))]
    col, obj, _, _ = _assign_all(td, cases, want_duals=False)
    assert int(obj[1]) == 101 and int(obj[3]) == 17
    assert col[1, :4].tolist() in gold["A1_python_py"]["optimal_perms"]
    for b in (0, 2, 4):
        assert int(obj[b]) == assign_ref.solve_scipy(cases[b])[0]


def _poisoned_pack(cases, gaps):
    """packed buffer with INT32_MIN-filled gaps of the given lengths (multiples of 4) before every instance and after
    the last one"""
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
def test_batch_instances_are_isolated_from_poisoned_gaps(td):
    dispatch, eng = _engine(td)
    cases = _ragged_cases(11)
    ref_col, ref_obj, ref_u, ref_v = _assign_all(td, cases)
    ref_lcm = dispatch.LCM_batch(cases, mask_value=100)
    rng = np.random.default_rng(5)
    packed, sizes, offs, n_max = _poisoned_pack(cases, [4 * int(k) for k in rng.integers(1, 9, len(cases))])
    col, obj, u, v = eng.assign_batch(packed, sizes, offs, n_max, want_duals=True)
    assert np.array_equal(col.cpu().numpy(), ref_col) and np.array_equal(obj.cpu().numpy(), ref_obj)
    assert np.array_equal(u.cpu().numpy(), ref_u) and np.array_equal(v.cpu().numpy(), ref_v)
    rows, cols, npairs, total, last = [t.cpu().numpy() for t in eng.lcm_batch(packed, sizes, offs, n_max, mask_value=100)]
    for b, r in enumerate(ref_lcm):
        k = r["n_pairs"]
        assert npairs[b] == k and total[b] == r["total"] and last[b] == r["last_min"]
        assert np.array_equal(rows[b, :k], r["rows"]) and np.array_equal(cols[b, :k], r["cols"])


@pytest.mark.gpu
def test_batch_withdraws_bad_instances_only(td):
    dispatch, eng = _engine(td)
    rng = np.random.default_rng(9)
    cases = [rng.integers(1, 40, (n, n)).astype(np.int32) for n in (30, 40, 50, 60, 70)]
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    sizes = sizes.clone()
    offs = offs.clone()
    sizes[1] = n_max + 1                   # larger than the call's n_max
    offs[3] += 2                           # not a multiple of 4
    col, obj, _, _ = eng.assign_batch(packed, sizes, offs, n_max)
    col, obj = col.cpu().numpy(), obj.cpu().numpy()
    rows, cols, npairs, total, last = [t.cpu().numpy() for t in eng.lcm_batch(packed, sizes, offs, n_max, mask_value=100)]
    for b in (1, 3):
        assert obj[b] == np.iinfo(np.int64).min and (col[b] == -1).all()
        assert npairs[b] == -1 and total[b] == np.iinfo(np.int64).min and (rows[b] == -1).all() and (cols[b] == -1).all()
    for b in (0, 2, 4):
        n = cases[b].shape[0]
        assert int(obj[b]) == assign_ref.solve_scipy(cases[b])[0]
        assert np.array_equal(col[b, :n], _single_col(eng, cases[b])[0])
        o = lcm_ref.lcm_c(cases[b], 100)
        assert npairs[b] == o["n_pairs"] and total[b] == o["total"] and np.array_equal(rows[b, :n], o["rows"])


@pytest.mark.gpu
def test_batch_many_waves_equal_single_calls_and_one_launch_each(td):
    dispatch, eng = _engine(td)
    rng = np.random.default_rng(2000)
    cases = [rng.integers(1, 40, (100, 100)).astype(np.int32) for _ in range(2000)]
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    lib = eng.lib
    l0 = lib.td_launch_count()
    col, obj, _, _ = eng.assign_batch(packed, sizes, offs, n_max)
    assert lib.td_launch_count() == l0 + 1
    lcm = eng.lcm_batch(packed, sizes, offs, n_max, mask_value=100)
    assert lib.td_launch_count() == l0 + 2
    col, obj = col.cpu().numpy(), obj.cpu().numpy()
    totals = lcm[3].cpu().numpy()
    offs = offs.cpu().numpy()
    for b in range(len(cases)):
        d = packed[offs[b]: offs[b] + 10000].view(100, 100)
        scol, sobj = eng.assign(d)[:2]
        rows, cols, scal = eng.lcm(d, 100)
        assert np.array_equal(col[b], scol.cpu().numpy()) and int(obj[b]) == int(sobj.item()), b
        assert int(totals[b]) == _lcm_total(scal), b


def _lcm_total(scal):
    s = scal.cpu().numpy()
    return int(np.frombuffer(s[:2].tobytes(), dtype=np.int64)[0])


LCM_VARIANTS = {
    "heuristic": dict(mask_value=100),
    "split": dict(mask_value=g.BIG_COST, sum_below=g.BIG_COST),
    "greedy_opt": dict(mask_value=g.BIG_COST, stop_above=10, sum_below=g.BIG_COST),
    "java": dict(mask_value=g.BIG_COST, stop_at_value=g.BIG_COST, residual_size=20),
    "max_iters": dict(mask_value=100, max_iters=15),
    "mask_tail": dict(mask_value=45),
}


def _lcm_oracle(c, kw):
    return lcm_ref.lcm_c(c, kw["mask_value"], kw.get("stop_above", I32_MAX), kw.get("stop_at_value", I32_MAX),
                         kw.get("sum_below", I32_MAX), kw.get("residual_size", 0), kw.get("max_iters", -1))


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(LCM_VARIANTS))
def test_lcm_batch_matches_the_literal_algorithm(td, variant):
    dispatch, eng = _engine(td)
    kw = LCM_VARIANTS[variant]
    cases = _ragged_cases(21)
    rng = np.random.default_rng(22)
    if variant == "mask_tail":                      # every cost >= the mask: masked cells win the argmin (trap 4)
        cases += [rng.integers(45, 60, (n, n)).astype(np.int32) for n in (1, 3, 40, 101)] + [np.full((20, 20), 45, np.int32)]
        c = rng.integers(1, 40, (80, 80)).astype(np.int32)
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


@pytest.mark.gpu
def test_solve_batch_and_lcm_batch_mix_small_and_large(td):
    dispatch, eng = _engine(td)
    rng = np.random.default_rng(300)
    cases = [rng.integers(1, 40, (n, n)).astype(np.int32) for n in (300, 12, 232, 300, 0, 77)]
    res = dispatch.solve_batch(cases, want_duals=True)
    for c, (col, obj, u, v) in zip(cases, res):
        n = c.shape[0]
        assert obj == (assign_ref.solve_scipy(c)[0] if n else 0)
        assert sorted(col.tolist()) == list(range(n)) and len(u) == n and len(v) == n
        if n:
            red = c.astype(np.int64) - u[:, None] - v[None, :]
            assert red.min() >= 0 and int(u.sum() + v.sum()) == obj
        if 0 < n <= MAX_N:
            assert np.array_equal(col, _single_col(eng, c)[0])
    for kw in (LCM_VARIANTS["heuristic"], LCM_VARIANTS["java"]):
        for c, r in zip(cases, dispatch.LCM_batch(cases, **kw)):
            o = _lcm_oracle(c, kw)
            assert r["n_pairs"] == o["n_pairs"] and r["total"] == o["total"] and r["last_min"] == o["last_min"]
            assert np.array_equal(r["rows"], o["rows"]) and np.array_equal(r["cols"], o["cols"])


@pytest.mark.gpu
def test_lcm_vs_optimum_on_the_device_equals_the_oracle_flow(td):
    cases = heuristic_cases(0)
    got = ex.lcm_vs_optimum(cases)
    want = ex.lcm_vs_optimum(cases, solver_batch=oracle_solver_batch, lcm_batch=oracle_lcm_batch)
    assert got == want                                      # LCM totals and optima are unique: exact, case by case
    ratio = float(np.mean([lcm / opt for lcm, opt in got]))
    assert abs(ratio - 1.78) <= 0.02, ratio
