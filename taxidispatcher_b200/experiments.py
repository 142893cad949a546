"""Host-side orchestration of the reference's two composite experiments on top of the dispatch kernels
(SURVEY.md section 8(f)-3):

  solve_split        split.py:61-119   stands cut into size/4-wide ranges, one exact solve per range, then a
                                       last solve over the customers and cabs the ranges left unserved
  greedy_then_solve  greedy_opt.py:131-163   LCM prefix with a distance threshold, exact solve on the rest
  lcm_vs_optimum     heuristic.py:20-40      LCM (mask 100) against the exact optimum on many small instances
  split_hybrid_vs_optimum  split.py:186-212, greedy_opt.py:129-163   the paper's split / LCM / hybrid degradation over
                                       many cases at once (batched stages)
  pool_greedy_vs_optimum  pool_opt_min.py      the Simulator's greedy 2-passenger pool against the optimal pairing

Every range of solve_split is an independent K1 + K2 instance: with a process group the ranges are spread
over the ranks (parallel.instances_for_rank), the unserved ids are gathered, and the leftover solve runs
once.  `solver` / `lcm` (and the batch functions) are injectable so that the host logic can be checked on CPU (tests only).
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np

BIG_COST = 250000


def _default_solver():
    from . import dispatch
    return dispatch.solve_dispatch


def count_sum(nn: int, cost, res, demand, supply, distances, total=0):
    """split.py:20-28: adds dist[cab.to][customer.from] of every real (non big_cost) assignment."""
    if nn == 0:
        return total
    x = np.asarray(res).reshape(nn, nn)
    c = np.asarray(cost)
    for taxi, trip in zip(*np.nonzero(x == 1)):
        if c[taxi][trip] < BIG_COST:
            total = total + int(distances[supply[taxi][2]][demand[trip][1]])
    return total


def filter_rows(rows: Sequence[Tuple[int, int, int]], wanted, element: int):
    """split.py:31-38 (`filter`): keeps rows whose field `element` is in `wanted` (a range or a list of ids)."""
    w = wanted if isinstance(wanted, range) else set(wanted)
    return [r for r in rows if r[element] in w]


def filter_out(rows, allocated: Sequence[int], element: int = 0):
    """greedy_opt.py:32-37: drops rows whose field `element` is in `allocated`."""
    a = set(int(v) for v in allocated)
    return [r for r in rows if r[element] not in a]


def _solve_range(solver, distances, split_demand, split_cabs):
    """One range of split.py:77-105.  Returns (range total, unserved customer ids, unused cab ids)."""
    nb_cust, nb_cabs = len(split_demand), len(split_cabs)
    rest_cust, rest_cabs = [], []
    s = 0
    if nb_cust > 0 and nb_cabs > 0:
        nb, x4, c = solver(distances, split_demand, split_cabs)
        xm = np.asarray(x4).reshape(nb, nb)
        cm = np.asarray(c)
        for taxi, trip in zip(*np.nonzero(xm == 1)):
            if cm[taxi][trip] == BIG_COST:                      # split.py:89 -- not served
                if nb_cabs > nb_cust:
                    rest_cabs.append(split_cabs[taxi][0])
                else:
                    rest_cust.append(split_demand[trip][0])
            else:
                s += int(distances[split_cabs[taxi][2]][split_demand[trip][1]])
    elif nb_cust > 0:
        rest_cust = [d[0] for d in split_demand]
    else:
        rest_cabs = [c[0] for c in split_cabs]
    return s, rest_cust, rest_cabs


def _solve_split_device(size: int, distances, demand, cabs, distributed: bool):
    """solve_split on the engine without the host in the loop: the stand table is uploaded once, every range is a
    boolean mask over the demand / cab arrays (split.py:31-38 `filter`), K1 and K2 run back to back on the device and
    only the matching (n column indices + n picked costs per range) comes back -- the reference-shaped solver interface
    would ship the n x n cost matrix and the n^2 solution vector to the host for every range."""
    from . import dispatch
    dem = np.asarray(demand, dtype=np.int64).reshape(-1, 3)
    cab = np.asarray(cabs, dtype=np.int64).reshape(-1, 3)
    dist_d = dispatch._h2d_i32(distances)
    split_size = int(size / 4)
    starts = list(range(0, size, split_size)) if split_size > 0 else []
    rank, world = 0, 1
    if distributed:
        from . import parallel
        rank, world = parallel.world()

    def solve_block(d_rows, c_rows):
        """(range total, unserved customer ids, unused cab ids) -- split.py:77-105"""
        nb_cust, nb_cabs = len(d_rows), len(c_rows)
        if nb_cust > 0 and nb_cabs > 0:
            nb, col, picked = dispatch.solve_assignment(dist_d, c_rows[:, 2], d_rows[:, 1])
            unserved = picked == BIG_COST                                        # split.py:89
            s = int(picked[~unserved].astype(np.int64).sum())
            if nb_cabs > nb_cust:                                                # there is always just one side dissatisfied
                return s, np.zeros(0, np.int64), c_rows[np.nonzero(unserved)[0], 0]
            return s, d_rows[col[unserved], 0], np.zeros(0, np.int64)
        if nb_cust > 0:
            return 0, d_rows[:, 0], np.zeros(0, np.int64)
        return 0, np.zeros(0, np.int64), c_rows[:, 0]

    results = {}
    for idx, start in enumerate(starts):
        if idx % world != rank:
            continue
        d_rows = dem[(dem[:, 1] >= start) & (dem[:, 1] < start + split_size)]
        c_rows = cab[(cab[:, 2] >= start) & (cab[:, 2] < start + split_size)]
        results[idx] = solve_block(d_rows, c_rows)
    if distributed and world > 1:
        import torch.distributed as dist
        gathered = [None] * world
        dist.all_gather_object(gathered, results)            # a few hundred ids: latency, not bandwidth
        results = {k: v for part in gathered for k, v in part.items()}
    total = 0
    rest_cust, rest_cabs = [], []
    for idx in range(len(starts)):                            # range order, like the reference's while loop
        s, rc, rb = results[idx]
        total += s
        rest_cust.append(np.asarray(rc, dtype=np.int64))
        rest_cabs.append(np.asarray(rb, dtype=np.int64))
    rest_cust = np.concatenate(rest_cust) if rest_cust else np.zeros(0, np.int64)
    rest_cabs = np.concatenate(rest_cabs) if rest_cabs else np.zeros(0, np.int64)
    rest_demand = dem[np.isin(dem[:, 0], rest_cust)]         # split.py:109-111: `filter` keeps the original order
    rest_supply = cab[np.isin(cab[:, 0], rest_cabs)]
    if len(rest_demand) == 0 and len(rest_supply) == 0:
        return total
    # the fifth run (split.py:113-119); count_sum adds every pairing below big_cost
    nn, col, picked = dispatch.solve_assignment(dist_d, rest_supply[:, 2], rest_demand[:, 1])
    return total + int(picked[picked < BIG_COST].astype(np.int64).sum())


def solve_split(size: int, distances, demand, cabs, solver: Optional[Callable] = None, distributed: bool = False):
    """split.py:61-119.  Returns the total cost of the split solution, or None when there is no demand or no
    supply (split.py:62-64).  distributed=True spreads the ranges over the ranks of the current process group.
    Without an injected `solver` the device path runs (_solve_split_device); a reference-shaped solver
    (distances, demand, cabs) -> (n, x, cost) takes the literal restatement below (tests, oracle back ends)."""
    if len(demand) == 0 or len(cabs) == 0:
        return None
    if solver is None:
        return _solve_split_device(size, distances, demand, cabs, distributed)
    split_size = int(size / 4)
    ranges = []
    start = 0
    while start < size:
        ranges.append(range(start, start + split_size))
        start += split_size
    rank, world = 0, 1
    if distributed:
        from . import parallel
        rank, world = parallel.world()
    results = {}
    for idx, r in enumerate(ranges):
        if idx % world != rank:
            continue
        results[idx] = _solve_range(solver, distances, filter_rows(demand, r, 1), filter_rows(cabs, r, 2))
    if distributed and world > 1:
        import torch.distributed as dist
        gathered = [None] * world
        dist.all_gather_object(gathered, results)            # a few hundred ids: latency, not bandwidth
        results = {k: v for part in gathered for k, v in part.items()}
    total, rest_cust, rest_cabs = 0, [], []
    for idx in range(len(ranges)):                            # range order, like the reference's while loop
        s, rc, rb = results[idx]
        total += s
        rest_cust += rc
        rest_cabs += rb
    rest_demand = filter_rows(demand, rest_cust, 0)
    rest_supply = filter_rows(cabs, rest_cabs, 0)
    if len(rest_demand) == 0 and len(rest_supply) == 0:
        return total
    nn, x5, c_table = solver(distances, rest_demand, rest_supply)
    return count_sum(nn, c_table, x5, rest_demand, rest_supply, distances, total)


def greedy_then_solve(distances, demand, cabs, threshold: int = 10, solver: Optional[Callable] = None,
                      lcm: Optional[Callable] = None):
    """greedy_opt.py:131-163: returns (nn, optimum, n2, hybrid total) -- the two pairs the script logs."""
    if solver is None or lcm is None:
        from . import dispatch
        solver = solver or dispatch.solve_dispatch
        lcm = lcm or dispatch.LCM_greedy_opt
    nn, x, cost_table = solver(distances, demand, cabs)
    res = count_sum(nn, cost_table, x, demand, cabs, distances, 0)
    # greedy_opt.py:146 hands LCM `matrix(cost_table).T`; cvxopt's matrix() of a list of rows is already the
    # transpose, so numpy sees the row-major cost[cab][cust] again (SURVEY.md section 4 trap 5)
    lcm_total, allocated_cabs, allocated_cust = lcm(nn, np.asarray(cost_table), threshold)
    rest_demand = filter_out(demand, allocated_cust, 0)
    rest_cabs = filter_out(cabs, allocated_cabs, 0)
    n2, x2, cost_table2 = solver(distances, rest_demand, rest_cabs)
    res2 = count_sum(n2, cost_table2, x2, rest_demand, rest_cabs, distances, 0)
    return nn, res, n2, res2 + int(lcm_total)


def lcm_vs_optimum(costs: Sequence, solver_batch: Optional[Callable] = None, lcm_batch: Optional[Callable] = None):
    """heuristic.py:20-40: every square matrix of `costs` goes through LCM (mask 100, every value summed, :24-33) and
    through the exact solver (:37).  Returns [(lcm_total, optimum)] per case; optimum <= lcm_total always holds (:40).
    solver_batch(costs) -> [(col_of_row, objective)] and lcm_batch(costs) -> [LCM dict] are injectable (tests feed
    oracles).  Without them the batch is uploaded once and both batched kernels run on the same packed buffer."""
    if solver_batch is None and lcm_batch is None:
        from . import dispatch
        opt, lcm = dispatch.run_batch(costs, assign=True, lcm=dict(mask_value=100))
    else:
        if solver_batch is None or lcm_batch is None:
            from . import dispatch
            solver_batch = solver_batch or dispatch.solve_batch
            lcm_batch = lcm_batch or (lambda cs: dispatch.LCM_batch(cs, mask_value=100))
        opt, lcm = solver_batch(costs), lcm_batch(costs)
    return [(int(l["total"]), int(o[1])) for l, o in zip(lcm, opt)]


def _stage_runner(dist: np.ndarray, solver_batch: Optional[Callable], lcm_batch: Optional[Callable]):
    """run(instances, assign, lcm=None, transpose=False) -> (col_of_row per instance or None, LCM dict per instance or
    None) for instances given as (cab_to, cust_from) stand index arrays with calculate_cost semantics (positional, padded
    with BIG_COST).  Without injected callables the matrices are built by K1 into packed device buffers and solved by
    the batched kernels (one group per kernel); otherwise they are built on the host and handed to the callables."""
    if solver_batch is None and lcm_batch is None:
        from . import dispatch
        dist_d = dispatch._h2d_i32(dist)
        dist_t = []

        def run_device(insts, assign, lcm=None, transpose=False):
            if transpose and not dist_t:
                dist_t.append(dist_d.t().contiguous())        # the stand table transposed: a layout copy
            ns = [max(len(c), len(d)) for c, d in insts]
            small, mid, large, huge = dispatch.size_groups(ns)
            if huge:
                raise ValueError("the batched experiment holds instances up to %d rows" % dispatch.BATCH_LARGE_MAX_N)
            res_a, res_l = [None] * len(insts), [None] * len(insts)
            for group in (small, mid, large):
                if not group:
                    continue
                packed, sizes, offsets, n_max, gns = dispatch.pack_cost_matrices(
                    dist_t[0] if transpose else dist_d, [insts[b] for b in group], transpose=transpose)
                ra, rl = dispatch.run_packed(packed, sizes, offsets, n_max, gns, assign=assign, lcm=lcm)
                for k, b in enumerate(group):
                    res_a[b] = ra[k][0] if assign else None
                    res_l[b] = rl[k] if lcm is not None else None
            return (res_a if assign else None), (res_l if lcm is not None else None)
        return run_device
    if solver_batch is None or lcm_batch is None:
        from . import dispatch
        solver_batch = solver_batch or dispatch.solve_batch
        lcm_batch = lcm_batch or dispatch.LCM_batch

    def run_host(insts, assign, lcm=None, transpose=False):
        mats = []
        for c, d in insts:
            c, d = np.asarray(c, dtype=np.int64), np.asarray(d, dtype=np.int64)
            m = np.full((max(len(c), len(d)),) * 2, BIG_COST, dtype=np.int32)
            if len(c) and len(d):
                m[: len(c), : len(d)] = dist[c[:, None], d[None, :]]
            mats.append(np.ascontiguousarray(m.T) if transpose else m)
        return ([r[0] for r in solver_batch(mats)] if assign else None), (lcm_batch(mats, **lcm) if lcm is not None else None)
    return run_host


def split_hybrid_vs_optimum(distances, cases: Sequence, threshold: int = 10, solver_batch: Optional[Callable] = None,
                            lcm_batch: Optional[Callable] = None):
    """The paper's split / hybrid experiment (PDF p.5-6; split.py:186-212, greedy_opt.py:129-163) over many cases at once.
    cases is a list of (demand, cabs) (lists of (id, from, to)); the stands are cut into len(distances) / 4 wide ranges
    like split.py's main.  Returns per case (optimum, split total, LCM-split total, hybrid total, n2): the quantities of
    greedy_then_solve (optimum, n2, hybrid), solve_split (split; None without demand or supply, split.py:62-64) and
    split.py:209's LCM on the transposed cost matrix (SURVEY.md section 4 trap 5).
    Three stages, each one batch over all cases: (1) optimum, greedy_opt LCM and split LCM on the full matrices, (2) the
    hybrid rest instances and the four ranges of every case, (3) the split leftovers.  solver_batch(costs) ->
    [(col_of_row, objective)] and lcm_batch(costs, **params) -> [LCM dict] are injectable (tests feed oracles); without
    them the cost matrices are built on the device and never leave it."""
    dist = np.asarray(distances)
    size = len(dist)
    split_size = int(size / 4)
    if split_size <= 0:
        raise ValueError("split needs at least 4 stands")
    run = _stage_runner(dist, solver_batch, lcm_batch)

    def inst(demand, cabs):
        return (np.array([c[2] for c in cabs], dtype=np.int32), np.array([d[1] for d in demand], dtype=np.int32))

    def picked(ins, col):
        """cost[i][col[i]] of every row (count_sum / split.py:89 read these cells)"""
        c, d = ins
        col = np.asarray(col, dtype=np.int64)
        rows = np.arange(len(col))
        out = np.full(len(col), BIG_COST, dtype=np.int64)
        real = (rows < len(c)) & (col < len(d))
        out[real] = dist[c[rows[real]].astype(np.int64), d[col[real]].astype(np.int64)]
        return out

    def real_sum(p):
        return int(p[p < BIG_COST].sum())

    # ---- stage 1: optimum + greedy_opt LCM (greedy_opt.py:141-146), split LCM on the transpose (split.py:209) ----------
    full = [inst(dem, cab) for dem, cab in cases]
    cols, greedy = run(full, True, dict(mask_value=BIG_COST, stop_above=threshold, sum_below=BIG_COST))
    _, lcm_split = run(full, False, dict(mask_value=BIG_COST, sum_below=BIG_COST), transpose=True)
    # ---- stage 2: the hybrid rest (greedy_opt.py:147-150) and the ranges of split.py:66-105 ---------------------------
    stage2, jobs = [], []            # jobs: (case, "rest") or (case, range index, split_demand, split_cabs)
    rest_n2 = []
    ranges = []
    start = 0
    while start < size:
        ranges.append(range(start, start + split_size))
        start += split_size
    for k, (demand, cabs) in enumerate(cases):
        rest_demand = filter_out(demand, greedy[k]["cols"].tolist(), 0)
        rest_cabs = filter_out(cabs, greedy[k]["rows"].tolist(), 0)
        rest_n2.append(max(len(rest_demand), len(rest_cabs)))
        if rest_demand and rest_cabs:
            stage2.append(inst(rest_demand, rest_cabs)); jobs.append((k, "rest"))
        if demand and cabs:
            for r in ranges:
                sd, sc = filter_rows(demand, r, 1), filter_rows(cabs, r, 2)
                if sd and sc:
                    stage2.append(inst(sd, sc)); jobs.append((k, "range", sd, sc))
    cols2, _ = run(stage2, True)
    hyb_rest = [0] * len(cases)
    split_sum = [0] * len(cases)
    rest_cust = [[] for _ in cases]
    rest_cab_ids = [[] for _ in cases]
    for ins, col, job in zip(stage2, cols2, jobs):
        k = job[0]
        p = picked(ins, col)
        if job[1] == "rest":
            hyb_rest[k] = real_sum(p)
            continue
        sd, sc = job[2], job[3]
        split_sum[k] += int(p[p != BIG_COST].sum())
        for taxi in np.nonzero(p == BIG_COST)[0]:                  # split.py:89 -- not served
            if len(sc) > len(sd):
                rest_cab_ids[k].append(sc[taxi][0])
            else:
                rest_cust[k].append(sd[int(col[taxi])][0])
    # ranges with one side only hand all of it to the leftover run (split.py:94-105)
    for k, (demand, cabs) in enumerate(cases):
        if not (demand and cabs):
            continue
        for r in ranges:
            sd, sc = filter_rows(demand, r, 1), filter_rows(cabs, r, 2)
            if sd and not sc:
                rest_cust[k] += [d[0] for d in sd]
            elif sc and not sd:
                rest_cab_ids[k] += [c[0] for c in sc]
    # ---- stage 3: the split leftovers (split.py:109-119) --------------------------------------------------------------
    stage3, owners = [], []
    for k, (demand, cabs) in enumerate(cases):
        rd, rs = filter_rows(demand, rest_cust[k], 0), filter_rows(cabs, rest_cab_ids[k], 0)
        if rd and rs:
            stage3.append(inst(rd, rs)); owners.append(k)
    cols3, _ = run(stage3, True)
    for k, ins, col in zip(owners, stage3, cols3):
        split_sum[k] += real_sum(picked(ins, col))
    out = []
    for k, (demand, cabs) in enumerate(cases):
        opt = real_sum(picked(full[k], cols[k])) if max(len(demand), len(cabs)) else 0
        split = split_sum[k] if (demand and cabs) else None
        out.append((opt, split, int(lcm_split[k]["total"]), hyb_rest[k] + int(greedy[k]["total"]), rest_n2[k]))
    return out


def pool_greedy_vs_optimum(instances: Sequence, dist, accept_all: bool = True, max_loss: float = 1.01,
                           greedy: Optional[Callable] = None, exact: Optional[Callable] = None):
    """pool_opt_min.py: every (frm, to) instance of `instances` is pooled by the Simulator's greedy scan
    (Simulator.java:681-758) and by the optimal pairing (minimum cost among the pairings of maximum cardinality, the
    reference's ILP where it is feasible).  Returns [(greedy_count, greedy_cost, opt_count, opt_cost)] per case;
    opt_count >= greedy_count, and opt_cost <= greedy_cost where the counts are equal.  greedy(frm, to, dist, accept_all,
    max_loss) and exact(instances, dist, accept_all, max_loss) -> row arrays are injectable (tests feed oracles).  Without
    them the whole experiment is one upload, one greedy and one exact batched launch, and one read-back."""
    from . import dispatch
    if greedy is None and exact is None:
        grd, opt = dispatch._find_pairs_batches(instances, dist, accept_all, max_loss, ("greedy", "exact"))
    else:
        opt = (exact or dispatch.find_pool_pairs_exact_batch)(instances, dist, accept_all, max_loss)
        if greedy is None:
            grd = dispatch.find_pool_pairs_batch(instances, dist, accept_all, max_loss)
        else:
            grd = [greedy(f, t, dist, accept_all, max_loss) if len(f) >= 2 else np.zeros((0, 4), np.int32)
                   for f, t in instances]
    out = []
    for g, o in zip(grd, opt):
        g, o = np.asarray(g).reshape(-1, 4), np.asarray(o).reshape(-1, 4)
        out.append((len(g), int(g[:, 3].astype(np.int64).sum()), len(o), int(o[:, 3].astype(np.int64).sum())))
    return out
