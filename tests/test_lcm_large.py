"""The whole-GPU LCM (td_lcm) above 2000 rows and on both of its round kernels, against a reference that scales: the
sorted walk of oracle/lcm_ref.py (lcm_sort_keys + lcm_walk), which tests/test_oracle.py pins to the literal C oracle.

td_lcm picks its round kernel by size: lcm_rounds_smem_kernel while the replicated state fits 200 KB of shared memory
(n <= 7873), lcm_rounds_kernel (the "generic" kernel: state in global memory, two grid barriers per round, pick slots
from atomics) above that, or at any n when TD_LCM_GENERIC is set.  The library does not report which one ran, so the
size rule is restated below and the boundary sizes are derived from it; setting TD_LCM_GENERIC is what guarantees the
generic kernel at the smaller sizes.

CPU: the restated rule; argument validation and the no-device return of the C ABI.
GPU: the generic kernel at the shapes of the K3 parity tests; sizes from 2001 to 20000 on both kernels (scalar and
vectorised scans, misaligned bases, determinism of the generic kernel); flat indices above 2^31 at n = 65535; the
route of LCM_batch above 2048 rows; extreme values through every LCM entry point; the 0-row call.  Every comparison is
bit-exact on rows, cols, n_pairs, total and last_min."""
import ctypes

import numpy as np
import pytest

from oracle import cost_ref, gen_inputs as g, lcm_ref

I32_MIN, I32_MAX = -2**31, 2**31 - 1
MAX_N = 65535                     # the flat index n * n - 1 must fit the 32-bit half of the key
BIG = g.BIG_COST

# ---- which round kernel td_lcm runs (csrc/td_lcm.cu), restated ---------------------------------------------------------
SMEM_LIMIT = 200 * 1024


def smem_kernel_bytes(n):
    """row and column minima (16 n), free flags (2 round16(n)), the stale-line list (8 n) and 64 bytes of slack"""
    return 16 * n + 2 * ((n + 15) & ~15) + 8 * n + 64


def runs_smem_kernel(n):
    return smem_kernel_bytes(n) <= SMEM_LIMIT


LAST_SMEM_N = max(n for n in range(1, 10000) if runs_smem_kernel(n))
FIRST_GENERIC_N = LAST_SMEM_N + 1


def test_restated_size_rule():
    assert (LAST_SMEM_N, FIRST_GENERIC_N) == (7873, 7874)
    assert all(runs_smem_kernel(n) for n in (1, 600, 2000, 2048, 4001, LAST_SMEM_N))
    assert not any(runs_smem_kernel(n) for n in (FIRST_GENERIC_N, 7876, 12000, 20000, MAX_N))
    # both kernels see both scans at the sizes below: odd n and n % 4 == 2 scan scalar, n % 4 == 0 vectorised
    assert {n % 4 for n in SIZES if n <= LAST_SMEM_N} >= {0, 1} and {n % 4 for n in SIZES if n > LAST_SMEM_N} >= {0, 2, 3}


# ---- CPU: the C ABI refuses bad arguments before it looks for a device -------------------------------------------------
def _abi():
    from taxidispatcher_b200 import _lib
    return _lib, _lib.lib()


def _params(_lib, kw):
    return _lib.LcmParams(kw["mask_value"], kw.get("stop_above", I32_MAX), kw.get("stop_at_value", I32_MAX),
                          kw.get("sum_below", I32_MAX), kw.get("residual_size", 0), kw.get("max_iters", -1))


def _td_lcm_call(lib, _lib, n, params=True, cost=16, rows=32, cols=48, npairs=64, total=80, last=96, ws=128,
                 ws_bytes=1 << 40):
    p = lambda a: None if a is None else ctypes.c_void_p(a)   # noqa: E731
    prm = _params(_lib, dict(mask_value=100))
    return lib.td_lcm(p(cost), n, ctypes.byref(prm) if params else None, p(rows), p(cols), p(npairs), p(total), p(last),
                      p(ws), ws_bytes, None)


def test_lcm_abi_argument_validation():
    _lib, lib = _abi()
    INV = _lib.TD_ERR_INVALID
    launches = lib.td_launch_count()
    assert _td_lcm_call(lib, _lib, MAX_N + 1) == INV
    assert _td_lcm_call(lib, _lib, -1) == INV
    assert _td_lcm_call(lib, _lib, 100, params=False) == INV
    assert _td_lcm_call(lib, _lib, 100, npairs=None) == INV
    assert _td_lcm_call(lib, _lib, 100, total=None) == INV
    assert lib.td_launch_count() == launches
    # the host wrapper answers a 0-row call itself: no pairs, total 0, last_min INT32_MAX (no iteration ran)
    prm = _params(_lib, dict(mask_value=100))
    npairs, total, last = ctypes.c_int32(-7), ctypes.c_int64(-7), ctypes.c_int32(-7)
    assert lib.tdh_lcm(None, 0, ctypes.byref(prm), None, None, ctypes.byref(npairs), ctypes.byref(total),
                       ctypes.byref(last)) == _lib.TD_OK
    assert (npairs.value, total.value, last.value) == (0, 0, I32_MAX)
    assert lib.td_launch_count() == launches


def test_lcm_abi_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    _lib, lib = _abi()
    launches = lib.td_launch_count()
    for n in (0, 1, LAST_SMEM_N, FIRST_GENERIC_N, MAX_N):
        assert _td_lcm_call(lib, _lib, n) == _lib.TD_ERR_NO_DEVICE, n
    assert lib.td_launch_count() == launches


# ---- GPU helpers -------------------------------------------------------------------------------------------------------
def _engine():
    from taxidispatcher_b200 import dispatch
    return dispatch, dispatch.engine()


def _oracle(c, kw):
    return lcm_ref.lcm_c(c, kw["mask_value"], kw.get("stop_above", I32_MAX), kw.get("stop_at_value", I32_MAX),
                         kw.get("sum_below", I32_MAX), kw.get("residual_size", 0), kw.get("max_iters", -1))


def _run(eng, cost_d, kw):
    """td_lcm through Engine.lcm on a device matrix (any view: its data pointer is passed as it is)"""
    from taxidispatcher_b200 import dispatch
    return dispatch.Engine.lcm_host_view(*eng.lcm(cost_d, **kw))


def _same(got, want, what):
    assert (got["n_pairs"], got["total"], got["last_min"]) == (want["n_pairs"], want["total"], want["last_min"]), what
    assert np.array_equal(got["rows"], want["rows"]) and np.array_equal(got["cols"], want["cols"]), what


def _generic(monkeypatch, fn):
    """fn() with the generic round kernel forced, twice: its pick slots come from atomics, its results must not"""
    monkeypatch.setenv("TD_LCM_GENERIC", "1")
    try:
        a, b = fn(), fn()
    finally:
        monkeypatch.delenv("TD_LCM_GENERIC")
    _same(a, b, "generic kernel, second run")
    return a


# ---- GPU: the generic kernel at the shapes of the K3 parity tests -------------------------------------------------------
def _parity_shapes():
    """(matrix, params) of test_gpu_parity.py's K3 tests"""
    out = []
    for n in (1, 2, 3, 31, 100, 257, 600):
        out.append((np.random.default_rng(n).integers(1, 40, (n, n)).astype(np.int32), dict(mask_value=100)))
    for n in (1, 5, 64, 130):
        out.append((np.full((n, n), 7, np.int32), dict(mask_value=100)))
        out.append((np.zeros((n, n), np.int32), dict(mask_value=BIG, sum_below=BIG)))
    out.append((np.random.default_rng(3).integers(0, 3, (90, 90)).astype(np.int32), dict(mask_value=100)))
    dist, cab_to, cust_from = g.config1b()
    split = dict(mask_value=BIG, sum_below=BIG)
    out.append((cost_ref.calculate_cost_np(dist, cab_to, cust_from)[1], split))
    out.append((cost_ref.calculate_cost_np(dist, cab_to[:150], cust_from)[1], split))
    out.append((cost_ref.calculate_cost_np(dist, cab_to, cust_from[:120], cutoff=10)[1], split))
    c = np.random.default_rng(8).integers(1, 40, (80, 80)).astype(np.int32)
    out += [(c, dict(mask_value=m)) for m in (20, 1, 0, 39, 40)]
    c = c.copy()
    c[0, :] = 50
    out += [(c, dict(mask_value=45)), (c, dict(mask_value=45, max_iters=60))]
    cost = cost_ref.calculate_cost_np(dist, cab_to, cust_from, cutoff=10)[1]
    out += [(cost, dict(mask_value=BIG, stop_above=thr, sum_below=BIG)) for thr in (0, 3, 10, 20)]
    out += [(cost, dict(mask_value=BIG, stop_at_value=BIG, residual_size=res)) for res in (0, 150, 199, 1, 500)]
    return out


@pytest.mark.gpu
def test_generic_kernel_at_the_parity_shapes(td, monkeypatch):
    dispatch, eng = _engine()
    for i, (c, kw) in enumerate(_parity_shapes()):
        cd = dispatch._h2d_i32(c)
        _same(_generic(monkeypatch, lambda: _run(eng, cd, kw)), _oracle(c, kw), (i, c.shape, kw))


def _finalize_cases():
    """A stop rule trips on a cell the last round left free, below a cell that round picked.  3 x 3: round 0 picks
    (0,0) = 1 and (2,2) = 7 (both dominant); (1,1) = 5 is not (its column holds 3 at (0,1)) and stays free when row 0
    goes.  With stop_above 4 the literal loop stops on 5, so last_min is 5, not 7.  The random cases put the same
    pattern at scale: a stop rule inside the value range."""
    c = np.array([[1, 3, 9], [9, 5, 9], [9, 9, 7]], np.int32)
    out = [(c, dict(mask_value=100, stop_above=4)), (c, dict(mask_value=100, stop_at_value=5)),
           (c, dict(mask_value=6, stop_above=4))]
    for n in (2, 3, 5, 8, 31, 100, 600):
        rng = np.random.default_rng(31 + n)
        u = rng.integers(1, 40, (n, n)).astype(np.int32)
        out += [(u, dict(mask_value=100, stop_above=10)), (u, dict(mask_value=100, stop_at_value=20)),
                (u, dict(mask_value=BIG, stop_above=25, sum_below=BIG))]
    return out


@pytest.mark.gpu
def test_stop_rule_below_a_last_round_pick(td, monkeypatch):
    dispatch, eng = _engine()
    cases = _finalize_cases()
    assert _oracle(*cases[0])["last_min"] == 5
    for i, (c, kw) in enumerate(cases):
        want = _oracle(c, kw)
        cd = dispatch._h2d_i32(c)
        _same(_run(eng, cd, kw), want, ("smem", i, c.shape, kw))
        _same(_generic(monkeypatch, lambda: _run(eng, cd, kw)), want, ("generic", i, c.shape, kw))


# ---- GPU: sizes above 2000 rows on both kernels ------------------------------------------------------------------------
HEUR = dict(mask_value=100)                                           # heuristic.py, config 2
STOP10 = dict(mask_value=100, stop_above=10)                          # a stop rule inside U[1,39]
SPLIT = dict(mask_value=BIG, sum_below=BIG)                           # split.py: the big_cost tail (trap 4)
GREEDY10 = dict(mask_value=BIG, stop_above=10, sum_below=BIG)         # greedy_opt.py
JAVA600 = dict(mask_value=BIG, stop_at_value=BIG, residual_size=600)  # Simulator.java, MAX_NON_LCM 600
JAVA1300 = dict(mask_value=BIG, stop_at_value=BIG, residual_size=1300)
TIESTOP = dict(mask_value=100, stop_at_value=1)
MAXIT = "max_iters n/3"                                               # HEUR with max_iters = n // 3


def _matrix(kind, n):
    rng = np.random.default_rng(n * 10 + len(kind))
    if kind == "u39":
        return g.config2(n, seed=n)                                   # config 2's shape: U[1,39]
    if kind == "ties":
        return rng.integers(0, 3, (n, n)).astype(np.int32)
    if kind == "above":                                               # every cost >= the mask: masked cells win at t = 1
        return rng.integers(100, 131, (n, n)).astype(np.int32)
    assert kind == "stand"                                            # big_cost dummy rows, cutoff 10 holes
    n_cabs = n - n // 20
    return cost_ref.calculate_cost_np(g.stand_distances(500), rng.integers(0, 500, n_cabs), rng.integers(0, 500, n),
                                      cutoff=10)[1]


# n -> [(matrix kind, [params])]: a tail case (SPLIT, "above") and a stop-rule case on each side of the kernel boundary
SIZES = {
    2001: [("u39", [HEUR, STOP10]), ("stand", [SPLIT, GREEDY10, JAVA600])],
    4000: [("u39", [HEUR, MAXIT])],
    4001: [("ties", [HEUR, TIESTOP]), ("above", [HEUR])],
    LAST_SMEM_N - 1: [("stand", [SPLIT, GREEDY10, JAVA1300]), ("u39", [STOP10])],
    LAST_SMEM_N: [("stand", [SPLIT, GREEDY10, JAVA600]), ("u39", [HEUR, MAXIT])],
    FIRST_GENERIC_N: [("stand", [SPLIT, GREEDY10, JAVA1300]), ("u39", [STOP10])],
    FIRST_GENERIC_N + 1: [("ties", [HEUR, TIESTOP]), ("above", [HEUR])],
    FIRST_GENERIC_N + 2: [("u39", [HEUR, MAXIT])],
    12000: [("ties", [HEUR, MAXIT])],
    16384: [("u39", [HEUR, STOP10])],
    20000: [("stand", [SPLIT, GREEDY10, JAVA600, JAVA1300])],
}


def _misaligned(c):
    """the same matrix as an (n, n) view that starts one element into a flat device buffer: not 16-byte aligned"""
    import torch
    n = c.shape[0]
    buf = torch.empty(n * n + 4, dtype=torch.int32, device="cuda")
    buf[1: 1 + n * n] = torch.from_numpy(c.reshape(-1)).cuda()
    view = buf[1: 1 + n * n].view(n, n)
    assert view.data_ptr() % 16 != 0
    return view


@pytest.mark.gpu
@pytest.mark.parametrize("n", sorted(SIZES))
def test_sizes_above_2000_rows_on_both_kernels(td, monkeypatch, n):
    dispatch, eng = _engine()
    for ci, (kind, variants) in enumerate(SIZES[n]):
        c = _matrix(kind, n)
        keys = lcm_ref.lcm_sort_keys(c)
        cd = dispatch._h2d_i32(c)
        views = [("aligned", cd)] + ([("misaligned", _misaligned(c))] if n % 4 == 0 and ci == 0 else [])
        for kw in variants:
            kw = dict(HEUR, max_iters=n // 3) if kw is MAXIT else kw
            want = lcm_ref.lcm_walk(keys, n, **kw)
            for name, view in views:
                what = (n, kind, kw, name)
                got = _run(eng, view, kw)
                _same(got, want, what + ("smem" if runs_smem_kernel(n) else "generic",))
                if runs_smem_kernel(n):
                    _same(_generic(monkeypatch, lambda: _run(eng, view, kw)), got, what + ("generic",))
                else:
                    _same(_run(eng, view, kw), got, what + ("generic, second run",))
            if kw in (SPLIT, HEUR) and kind in ("stand", "above"):   # every masked pick repeats a picked column
                assert want["n_pairs"] == n and len(np.unique(want["cols"])) < n, "the tail reaches the masked picks"
            if kw in (STOP10, GREEDY10, TIESTOP):
                assert want["n_pairs"] < n, "the stop rule ends the walk early"
        del cd, keys


# ---- GPU: flat indices above 2^31 --------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_flat_index_above_2_31_at_the_largest_n(td):
    """n = 65535: row i holds one cheap cell w_i in [0, 4) at column pi(i), every other cell is big_cost.  Every cheap
    cell is the minimum of its row and of its column, so round 0 picks all of them, and the trace is those cells in
    (w_i, i * n + pi(i)) order -- an int64 sort on the host.  About half of them lie past flat index 2^31."""
    import torch
    from taxidispatcher_b200 import _lib
    n = MAX_N
    free, _ = torch.cuda.mem_get_info()
    if free < 40 * 2**30:
        pytest.skip("needs 40 GB of free device memory (cost and its transpose are 17 GB each), %.1f GB free" %
                    (free / 2**30))
    _, eng = _engine()
    rng = np.random.default_rng(65535)
    pi = rng.permutation(n)
    w = rng.integers(0, 4, n).astype(np.int32)
    idx = np.arange(n, dtype=np.int64) * n + pi
    order = np.lexsort((idx, w))
    cost = ws = None
    try:
        cost = torch.full((n, n), BIG, dtype=torch.int32, device="cuda")
        cost[torch.arange(n, device="cuda"), torch.from_numpy(pi).cuda()] = torch.from_numpy(w).cuda()
        ws_bytes = eng.lib.td_lcm_workspace_bytes(n)
        ws = torch.empty(ws_bytes, dtype=torch.uint8, device="cuda")     # not the engine's grow-only workspace
        rows = torch.empty(n, dtype=torch.int32, device="cuda")
        cols = torch.empty(n, dtype=torch.int32, device="cuda")
        scal = torch.zeros(4, dtype=torch.int32, device="cuda")
        for iters in (n, n // 2):
            prm = _params(_lib, dict(mask_value=BIG, sum_below=BIG, max_iters=iters))
            scal.fill_(-7)
            p = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731
            base = scal.data_ptr()
            rc = eng.lib.td_lcm(p(cost), n, ctypes.byref(prm), p(rows), p(cols), ctypes.c_void_p(base + 8),
                                ctypes.c_void_p(base), ctypes.c_void_p(base + 12), p(ws), ws_bytes,
                                ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
            assert rc == 0
            from taxidispatcher_b200 import dispatch
            got = dispatch.Engine.lcm_host_view(rows, cols, scal)
            sel = order[:iters]
            assert (idx[sel] >= 2**31).sum() > iters // 3
            want = {"n_pairs": iters, "total": int(w[sel].astype(np.int64).sum()), "last_min": int(w[sel[-1]]),
                    "rows": sel.astype(np.int32), "cols": pi[sel].astype(np.int32)}
            _same(got, want, ("n = 65535", iters))
    finally:
        del cost, ws
        torch.cuda.synchronize()
        torch.cuda.empty_cache()


# ---- GPU: LCM_batch above 2048 rows ------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_lcm_batch_routes_instances_above_2048_rows(td):
    """Instances above the batch kernels' 2048 rows take whole-GPU td_lcm calls inside LCM_batch; they are checked
    against the sorted walk, the batch-sized ones against the literal oracle."""
    from test_batch_large import LCM_VARIANTS
    dispatch, _ = _engine()
    rng = np.random.default_rng(2100)
    cases = [rng.integers(1, 40, (n, n)).astype(np.int32) for n in (100, 2100, 5, 300, 4000, 700)]
    keys = {b: lcm_ref.lcm_sort_keys(c) for b, c in enumerate(cases) if c.shape[0] > 2048}
    for kw in (LCM_VARIANTS["heuristic"], LCM_VARIANTS["java"]):
        res = dispatch.LCM_batch(cases, **kw)
        for b, c in enumerate(cases):
            n = c.shape[0]
            want = lcm_ref.lcm_walk(keys[b], n, **kw) if b in keys else _oracle(c, kw)
            _same(res[b], want, (kw, b, n))


# ---- GPU: extreme values through every LCM entry point -----------------------------------------------------------------
EXTREME_PARAMS = [dict(mask_value=I32_MAX), dict(mask_value=I32_MIN), dict(mask_value=0),
                  dict(mask_value=I32_MAX, stop_above=I32_MAX - 1), dict(mask_value=0, stop_above=I32_MAX - 1),
                  dict(mask_value=100, max_iters=0), dict(mask_value=I32_MIN, residual_size=200),
                  dict(mask_value=BIG, stop_at_value=BIG, residual_size=101, sum_below=I32_MIN)]


def _extreme_cases():
    rng = np.random.default_rng(2**31 - 1)
    vals = np.array([I32_MIN, I32_MIN + 1, -1, 0, 1, 100, I32_MAX - 1, I32_MAX], np.int64)
    out = [np.zeros((0, 0), np.int32)]
    for n in (1, 2, 5, 33, 100):
        out.append(rng.choice(vals, (n, n)).astype(np.int32))
    out.append(np.full((17, 17), I32_MAX, np.int32))
    out.append(np.full((18, 18), I32_MIN, np.int32))
    return out


def _batch_call(eng, name, packed, sizes, offs, n_max, kw):
    import torch
    from taxidispatcher_b200 import _lib
    B = int(sizes.numel())
    rows = torch.empty((B, max(n_max, 1)), dtype=torch.int32, device="cuda")
    cols = torch.empty((B, max(n_max, 1)), dtype=torch.int32, device="cuda")
    npairs = torch.empty(B, dtype=torch.int32, device="cuda")
    total = torch.empty(B, dtype=torch.int64, device="cuda")
    last = torch.empty(B, dtype=torch.int32, device="cuda")
    prm = _params(_lib, kw)
    p = lambda t: ctypes.c_void_p(t.data_ptr())   # noqa: E731
    rc = getattr(eng.lib, name)(p(packed), p(sizes), p(offs), B, int(n_max), ctypes.byref(prm), p(rows), p(cols),
                                p(npairs), p(total), p(last), None)
    assert rc == 0, name
    rows, cols, npairs, total, last = [t.cpu().numpy() for t in (rows, cols, npairs, total, last)]
    return [{"rows": rows[b, :npairs[b]], "cols": cols[b, :npairs[b]], "n_pairs": int(npairs[b]),
             "total": int(total[b]), "last_min": int(last[b])} for b in range(B)]


@pytest.mark.gpu
def test_extreme_values_on_every_lcm_entry_point(td, monkeypatch):
    import torch
    dispatch, eng = _engine()
    cases = _extreme_cases()
    packed, sizes, offs, n_max = dispatch.pack_batch(cases)
    for kw in EXTREME_PARAMS:
        want = [_oracle(c, kw) for c in cases]
        for name, nm in (("td_lcm_batch", n_max), ("td_lcm_batch_cluster", 640), ("td_lcm_batch_large", 2048)):
            for b, got in enumerate(_batch_call(eng, name, packed, sizes, offs, nm, kw)):
                _same(got, want[b], (name, kw, b))
        for b, c in enumerate(cases):
            cd = torch.from_numpy(c).cuda()
            _same(_run(eng, cd, kw), want[b], ("td_lcm", kw, b))
            _same(_generic(monkeypatch, lambda: _run(eng, cd, kw)), want[b], ("td_lcm generic", kw, b))


# ---- GPU: the 0-row call -----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_zero_rows_report_last_min_int32_max(td):
    import torch
    from taxidispatcher_b200 import _lib
    dispatch, eng = _engine()
    scal = torch.full((4,), -7, dtype=torch.int32, device="cuda")   # [total lo, total hi, n_pairs, last_min]
    prm = _params(_lib, dict(mask_value=100))
    base = scal.data_ptr()
    rc = eng.lib.td_lcm(None, 0, ctypes.byref(prm), None, None, ctypes.c_void_p(base + 8), ctypes.c_void_p(base),
                        ctypes.c_void_p(base + 12), None, 0, None)
    assert rc == 0
    torch.cuda.synchronize()
    assert scal.cpu().tolist() == [0, 0, 0, I32_MAX]
    got = dispatch.Engine.lcm_host_view(*eng.lcm(torch.empty((0, 0), dtype=torch.int32, device="cuda"), mask_value=100))
    assert (got["n_pairs"], got["total"], got["last_min"]) == (0, 0, I32_MAX)
    want = dispatch.LCM(0, np.zeros((0, 0), np.int32), mask_value=100)     # answered on the host
    assert (want["n_pairs"], want["total"], want["last_min"]) == (0, 0, I32_MAX)
