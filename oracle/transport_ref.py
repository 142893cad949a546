"""CPU model of td_assign_stands_batch: the stand-derived assignment as an S x S transportation problem.

The padded matrix of calculate_cost has identical rows for the cabs of one stand and identical columns for the
customers of one stand, so its optimum is the transportation optimum on the stand counts plus the padding's
(n - min(cabs, customers)) * fill.  Only the counts matter: any n costs one pass over the index arrays.

solve() runs the algorithm the kernel runs -- successive shortest paths from the spare side, dense Dijkstra on int64
reduced costs starting from the column minima, ties broken by (label, side, stand), bottleneck augmentation -- so its
flows, potentials and phase / augmentation counts are the kernel's.  Its optimality is checked independently (tests:
scipy's linear_sum_assignment on the dense matrix, HiGHS on the LP, networkx).  expand() is the documented rule that
turns flows into col_of_row; flows_from_cols() goes back; check_certificate() checks the stand potentials.
"""
from __future__ import annotations

import numpy as np

INF = 1 << 54


def arc_costs(dist, fill: int, cutoff=None) -> np.ndarray:
    """The K1 cell rule on the stand table: dist[a][b], or fill when a cutoff is given and dist >= cutoff."""
    d = np.asarray(dist, dtype=np.int64)
    return np.where(d >= cutoff, np.int64(fill), d) if cutoff is not None and cutoff >= 0 else d.copy()


def stand_counts(idx, S: int) -> np.ndarray:
    idx = np.asarray(idx, dtype=np.int64).reshape(-1)
    if idx.size and (idx.min() < 0 or idx.max() >= S):
        raise IndexError("stand index out of range of the distance table")
    return np.bincount(idx, minlength=S).astype(np.int64)


def solve_counts(C: np.ndarray, s: np.ndarray, d: np.ndarray):
    """Min-cost flow of value min(sum s, sum d) from supplies s (cab stands) to demands d (customer stands) over the
    complete table C.  Returns (flow [S, S] in (cab, customer) orientation, u, v, phases, augmentations)."""
    S = C.shape[0]
    nc, nd = int(s.sum()), int(d.sum())
    tr = nc < nd                                     # sources = the side with more members (cabs when balanced)
    K = C.T.copy() if tr else C.copy()
    cp, cq = (d, s) if tr else (s, d)
    K = np.where(np.outer(cp > 0, cq > 0), K, 0)
    F = np.zeros((S, S), dtype=np.int64)
    al = np.zeros(S, dtype=np.int64)
    colmin = np.where(cp[:, None] > 0, K, np.iinfo(np.int64).max).min(axis=0)
    be = np.where(cq > 0, colmin, 0).astype(np.int64)
    be[(cq > 0) & (cp.sum() == 0)] = 0
    rp, rq = cp.astype(np.int64).copy(), cq.astype(np.int64).copy()
    total = int(cq.sum()) if nc and nd else 0
    flow, phases = 0, 0
    while flow < total:
        lab_p = np.where((cp > 0) & (rp > 0), 0, INF).astype(np.int64)
        lab_q = np.full(S, INF, dtype=np.int64)
        par_p = np.full(S, -1, dtype=np.int64)
        par_q = np.full(S, -1, dtype=np.int64)
        done_p, done_q = cp == 0, cq == 0
        sink, D = -1, 0
        while True:
            mp = np.where(~done_p & (lab_p < INF), lab_p, INF)
            mq = np.where(~done_q & (lab_q < INF), lab_q, INF)
            x, y = int(np.argmin(mp)), int(np.argmin(mq))
            if mp[x] >= INF and mq[y] >= INF:
                break
            if mp[x] <= mq[y]:                           # (label, side, stand): sources first at equal labels
                L = int(mp[x])
                done_p[x] = True
                nl = L + K[x] - al[x] - be
                upd = ~done_q & (nl < lab_q)
                lab_q[upd] = nl[upd]
                par_q[upd] = x
            else:
                L = int(mq[y])
                if rq[y] > 0:
                    sink, D = y, L
                    break
                done_q[y] = True
                nl = L - (K[:, y] - al - be[y])
                upd = ~done_p & (F[:, y] > 0) & (nl < lab_p)
                lab_p[upd] = nl[upd]
                par_p[upd] = y
        if sink < 0:
            break
        al -= np.where(cp > 0, np.minimum(lab_p, D), 0)
        be += np.where(cq > 0, np.minimum(lab_q, D), 0)
        dlt, y = int(rq[sink]), sink
        while True:
            x = int(par_q[y])
            py = int(par_p[x])
            if py < 0:
                dlt = min(dlt, int(rp[x]))
                break
            dlt = min(dlt, int(F[x, py]))
            y = py
        y = sink
        while True:
            x = int(par_q[y])
            F[x, y] += dlt
            py = int(par_p[x])
            if py < 0:
                rp[x] -= dlt
                break
            F[x, py] -= dlt
            y = py
        rq[sink] -= dlt
        flow += dlt
        phases += 1
    if tr:
        return F.T.copy(), be, al, phases, phases
    return F, al, be, phases, phases


def solve(dist, cab_to, cust_from, fill: int, cutoff=None) -> dict:
    """objective (the optimum of the padded calculate_cost matrix), flow, u, v, phases, augmentations."""
    dist = np.asarray(dist)
    S = dist.shape[0]
    s, d = stand_counts(cab_to, S), stand_counts(cust_from, S)
    C = arc_costs(dist, fill, cutoff)
    nc, nd = int(s.sum()), int(d.sum())
    F, u, v, ph, aug = solve_counts(C, s, d)
    obj = int((F * C).sum()) + (max(nc, nd) - min(nc, nd)) * int(fill)
    return {"objective": obj, "flow": F, "u": u, "v": v, "phases": ph, "augmentations": aug}


def expand(flow, cab_to, cust_from, C, fill: int) -> tuple:
    """col_of_row and cost_of_row of the documented rule: the cabs of stand a, in increasing index order, go to the
    customer stands in increasing b, f(a, b) each; the customers of stand b, in increasing index order, are dealt to
    the cab stands in increasing a; spare rows take the unserved customers in index order, spare cabs take the padding
    columns in row order."""
    cab_to = np.asarray(cab_to, dtype=np.int64).reshape(-1)
    cust_from = np.asarray(cust_from, dtype=np.int64).reshape(-1)
    F = np.asarray(flow, dtype=np.int64)
    nc, nd = len(cab_to), len(cust_from)
    n = max(nc, nd)
    col = np.full(n, -1, dtype=np.int64)
    S = F.shape[0]
    cust_lists = [np.flatnonzero(cust_from == b) for b in range(S)]
    taken = np.zeros(S, dtype=np.int64)                 # customers of stand b dealt so far (cab stands in increasing a)
    queue = {}                                          # (a, b) -> customer indices for stand a's cabs
    for a in range(S):
        for b in range(S):
            f = int(F[a, b])
            if f:
                queue[(a, b)] = list(cust_lists[b][taken[b]: taken[b] + f])
                taken[b] += f
    served = np.zeros(nd, dtype=bool)
    spare_col = nd
    for a in range(S):
        rows = np.flatnonzero(cab_to == a)
        k = 0
        for b in range(S):
            for j in queue.get((a, b), []):
                col[rows[k]] = j
                served[j] = True
                k += 1
    for i in range(nc):                                 # spare cabs, in row order
        if col[i] < 0:
            col[i] = spare_col
            spare_col += 1
    r = nc
    for j in range(nd):                                 # spare rows take the unserved customers in index order
        if not served[j]:
            col[r] = j
            r += 1
    return col, padded_costs(col, cab_to, cust_from, C, fill)


def padded_costs(col, cab_to, cust_from, C, fill: int) -> np.ndarray:
    """M[i][col[i]] of the padded matrix."""
    nc, nd = len(cab_to), len(cust_from)
    out = np.full(len(col), fill, dtype=np.int64)
    for i, j in enumerate(col):
        if i < nc and j < nd:
            out[i] = C[cab_to[i], cust_from[j]]
    return out


def flows_from_cols(col, cab_to, cust_from, S: int) -> np.ndarray:
    """Stand flows of a padded col_of_row: f(a, b) = real rows at stand a matched to real columns at stand b."""
    cab_to = np.asarray(cab_to, dtype=np.int64).reshape(-1)
    cust_from = np.asarray(cust_from, dtype=np.int64).reshape(-1)
    col = np.asarray(col, dtype=np.int64)
    nc, nd = len(cab_to), len(cust_from)
    F = np.zeros((S, S), dtype=np.int64)
    rows = np.arange(min(nc, len(col)))
    real = col[rows] < nd
    np.add.at(F, (cab_to[rows[real]], cust_from[col[rows[real]]]), 1)
    return F


def check_certificate(C, s, d, flow, u, v) -> bool:
    """Stand-level complementary slackness: reduced costs >= 0 between stands with members, == 0 where flow runs; the
    spare side's potentials <= 0 and 0 where a member is unmatched; 0 at empty stands; dual = primal."""
    C, s, d, F = (np.asarray(a, dtype=np.int64) for a in (C, s, d, flow))
    u, v = np.asarray(u, dtype=np.int64), np.asarray(v, dtype=np.int64)
    nc, nd = int(s.sum()), int(d.sum())
    if np.any(u[s == 0] != 0) or np.any(v[d == 0] != 0):
        return False
    if nc == 0 or nd == 0:
        return bool(np.all(u == 0) and np.all(v == 0))
    red = C - u[:, None] - v[None, :]
    live = np.outer(s > 0, d > 0)
    if np.any(red[live] < 0) or np.any(red[F > 0] != 0):
        return False
    out, inn = F.sum(axis=1), F.sum(axis=0)
    if nc > nd and (np.any(u > 0) or np.any(u[out < s] != 0)):
        return False
    if nd > nc and (np.any(v > 0) or np.any(v[inn < d] != 0)):
        return False
    return int((s * u).sum() + (d * v).sum()) == int((F * C).sum())
