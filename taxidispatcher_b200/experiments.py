"""Host-side orchestration of the reference's two composite experiments on top of the dispatch kernels
(SURVEY.md section 8(f)-3):

  solve_split        split.py:61-119   stands cut into size/4-wide ranges, one exact solve per range, then a
                                       last solve over the customers and cabs the ranges left unserved
  greedy_then_solve  greedy_opt.py:131-163   LCM prefix with a distance threshold, exact solve on the rest
  lcm_vs_optimum     heuristic.py:20-40      LCM (mask 100) against the exact optimum on many small instances
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


def pool_greedy_vs_optimum(instances: Sequence, dist, accept_all: bool = True, max_loss: float = 1.01,
                           greedy: Optional[Callable] = None, exact: Optional[Callable] = None):
    """pool_opt_min.py: every (frm, to) instance of `instances` is pooled by the Simulator's greedy scan
    (Simulator.java:681-758) and by the optimal pairing (minimum cost among the pairings of maximum cardinality, the
    reference's ILP where it is feasible).  Returns [(greedy_count, greedy_cost, opt_count, opt_cost)] per case;
    opt_count >= greedy_count, and opt_cost <= greedy_cost where the counts are equal.  greedy(frm, to, dist, accept_all,
    max_loss) and exact(instances, dist, accept_all, max_loss) -> row arrays are injectable (tests feed oracles); without
    them the greedy runs per instance and the exact pool is one batched launch."""
    from . import dispatch
    greedy = greedy or dispatch.find_pool_pairs
    exact = exact or dispatch.find_pool_pairs_exact_batch
    opt = exact(instances, dist, accept_all, max_loss)
    out = []
    for (f, t), o in zip(instances, opt):
        g = greedy(f, t, dist, accept_all, max_loss) if len(f) >= 2 else np.zeros((0, 4), np.int32)
        g, o = np.asarray(g).reshape(-1, 4), np.asarray(o).reshape(-1, 4)
        out.append((len(g), int(g[:, 3].astype(np.int64).sum()), len(o), int(o[:, 3].astype(np.int64).sum())))
    return out
