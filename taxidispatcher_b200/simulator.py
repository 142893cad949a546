"""Replay driver for BASELINE.json config 4: the reference's Simulator (Simulator.java) restated on top of
the dispatch kernels -- per-minute batches of 2-passenger pool -> cost matrix -> LCM (when the model is
larger than MAX_NON_LCM) -> exact solve, over simulations/taxi_demand.txt (SURVEY.md section 3.4, 8(f)-1).

Host logic only (state machine of cabs and customers); every dispatch primitive goes through a backend:
the product default `CudaBackend` calls the CUDA engine; tests inject a CPU backend built from the test-only CPU restatements
to check this host logic against the reference's golden log (simulations/simulog_solv.txt, KAT S1).
No JVM exists here, so this file is a restatement, cited line by line:

  main loop                  Simulator.java:141-218
  checkIfCabAtDestination    :220-254         createTempDemand :329-355     createTempSupply :358-372
  analyzeSolution            :375-421         assignPooledCustomer :424-442 assignToCabAndGo :444-470
  cheatAbit                  :472-477         goToPickupUp :479-494         calculate_cost :497-520
  LCM                        :523-549         analyzePairs :613-674         findPool :681-758
  analyzePool                :760-784         printMetrics :256-277         initSupply :562-574
"""
from __future__ import annotations

import time
from dataclasses import dataclass, field
from typing import List, Optional, Sequence, Tuple

import numpy as np

# constants of Simulator.java:108-115
HOURS = 2
N_STANDS = 50
DROP_TIME = 10
MAX_NON_LCM = 600
N_CABS = 1300
BIG_COST = 250000
MAX_LOSS = 1.01
CLNT_A_ENDS, CLNT_B_ENDS = 0, 1
# cab columns (Simulator.java:91-96)
ID, FROM, TO, CLNT_ASSIGNED, CLNT_ON_BOARD, TIME_STARTED = range(6)


class CudaBackend:
    """The product backend: every primitive runs in libtaxidispatch.so on the GPU.  The cost matrix stays on the
    device between K1 and the LCM / exact solve that consume it (the host copy is only read by the state machine).
    exact_pool=True pools each step's customers by the optimal pairing (find_pool_pairs_exact) instead of the greedy
    scan of Simulator.findPool; the default keeps the reference's greedy."""

    def __init__(self, exact_pool: bool = False):
        import torch
        from . import dispatch
        self.d = dispatch
        self.torch = torch
        self.eng = dispatch.engine()
        self.times = {"pool": 0.0, "cost": 0.0, "lcm": 0.0, "solve": 0.0}
        self._cost_dev = None      # (id of the host array handed out, device tensor)
        self._dist_dev = None      # (host stand table, device copy): the table does not change during a replay
        self._pin = [None, None]   # two pinned read-back buffers, used alternately (a step holds at most two cost matrices)
        self._pin_i = 0
        self.exact_pool = exact_pool

    def _read_back(self, dev):
        """Device int32 tensor -> numpy through a reused pinned buffer (a 1300 x 1300 matrix per step: pageable read-backs
        were most of the replay's host time).  The view stays valid until the second next call."""
        n = dev.numel()
        buf = self._pin[self._pin_i]
        if buf is None or buf.numel() < n:
            buf = self._pin[self._pin_i] = self.torch.empty(max(n, 1 << 21), dtype=dev.dtype).pin_memory()
        self._pin_i ^= 1
        view = buf[:n].view(dev.shape)
        view.copy_(dev)                                   # blocking copy into pinned memory
        return view.numpy()

    def _device_cost(self, cost):
        if self._cost_dev is not None and self._cost_dev[0] is cost:
            return self._cost_dev[1]
        return self.d._h2d_i32(np.asarray(cost))

    def pool_pairs(self, frm, to, dist):
        t0 = time.perf_counter()
        find = self.d.find_pool_pairs_exact if self.exact_pool else self.d.find_pool_pairs
        r = find(frm, to, dist, accept_all=True, max_loss=MAX_LOSS)   # Simulator.java:691
        self.times["pool"] += time.perf_counter() - t0
        return r

    def cost(self, dist, cab_to, cust_from):
        t0 = time.perf_counter()
        n = max(len(cab_to), len(cust_from))
        if n == 0:
            return np.zeros((0, 0), np.int32)
        h2d = self.d._h2d_i32
        empty = self.torch.empty(0, dtype=self.torch.int32, device=self.eng.device)
        if self._dist_dev is None or self._dist_dev[0] is not dist:
            self._dist_dev = (dist, h2d(dist))
        dev = self.eng.cost_matrix(self._dist_dev[1], h2d(cab_to) if len(cab_to) else empty,
                                   h2d(cust_from) if len(cust_from) else empty, BIG_COST, DROP_TIME)
        host = self._read_back(dev)
        self._cost_dev = (host, dev)
        self.times["cost"] += time.perf_counter() - t0
        return host

    def lcm_java(self, cost):
        t0 = time.perf_counter()
        if len(cost) == 0:
            return [], BIG_COST
        r = self.d.Engine.lcm_host_view(*self.eng.lcm(self._device_cost(cost), BIG_COST, stop_at_value=BIG_COST,
                                                      residual_size=MAX_NON_LCM))          # Simulator.java:523-549
        mn = r["last_min"]
        self.times["lcm"] += time.perf_counter() - t0
        return list(zip(r["rows"].tolist(), r["cols"].tolist())), (BIG_COST if mn >= BIG_COST else mn)

    def solve(self, n, cost, n_cabs=None, n_cust=None):
        t0 = time.perf_counter()
        if n == 0:
            return []
        _, _, x, _ = self.eng.assign(self._device_cost(cost), want_x=True, n_real_rows=n_cabs, n_real_cols=n_cust)
        x = x.cpu().numpy()
        self.times["solve"] += time.perf_counter() - t0
        return x


@dataclass(slots=True)
class TempDemand:      # Simulator.java:47-58
    id: int
    frm: int
    to: int
    pool_clnt_id: int = -1
    pool_plan: int = -1
    pool_cost: int = 0


@dataclass
class Metrics:         # Simulator.java:124-136
    total_dropped: int = 0
    total_pickup_time: int = 0
    total_pickup_numb: int = 0
    max_model_size: int = 0
    max_solver_size: int = 0
    total_LCM_used: int = 0
    max_POOL_MEM_size: int = 0
    max_POOL_size: int = 0
    total_second_passengers: int = 0
    step_seconds: List[float] = field(default_factory=list)


def cheat_a_bit(frm: int, cost: int, n_stands: int = N_STANDS) -> int:   # Simulator.java:472-477
    if frm + cost >= n_stands:
        return 0 if frm - cost < 0 else frm - cost
    return frm + cost


class Simulator:
    def __init__(self, demand_rows: Sequence[Tuple[int, int, int, int, int]], backend=None, n_cabs: int = N_CABS,
                 n_stands: int = N_STANDS):
        rows = np.asarray(demand_rows, dtype=np.int64).reshape(-1, 5)
        self.n_stands = n_stands
        self.n_cabs = n_cabs
        self.backend = backend if backend is not None else CudaBackend()
        idx = np.arange(n_stands)
        self.dist = np.abs(idx[:, None] - idx[None, :]).astype(np.int32)          # computeDistances :553-560
        # demand (Simulator.java:60-69, readDemand :280-304)
        self.d_id, self.d_from, self.d_to, self.d_time, self.d_at = (rows[:, k].copy() for k in range(5))
        m = len(rows)
        self.d_cab = np.full(m, -1, np.int64)
        self.d_pickup_t = np.full(m, -1, np.int64)
        self.d_pool_clnt = np.full(m, -1, np.int64)
        self.d_pool_plan = np.full(m, -1, np.int64)
        self.d_pool_cost = np.zeros(m, np.int64)
        self.id_to_row = {int(v): i for i, v in enumerate(self.d_id)}               # ids are row indices in the file
        # cabs (initSupply :562-574)
        self.cabs = np.zeros((n_cabs, 6), np.int64)
        for i in range(n_cabs):
            j = i % n_stands
            self.cabs[i] = (i, j, j, -1, 0, -1)
        self.m = Metrics()
        self.solv_log: List[str] = []

    # ---- Simulator.java:220-254 ----------------------------------------------------------------------
    def check_if_cab_at_destination(self, t: int):
        cabs, dist = self.cabs, self.dist
        # the arrival test for all cabs at once; a cab's update touches only its own row and its own customer, so the
        # arrived cabs can be handled in index order afterwards (same order as the reference's loop)
        arrived = np.nonzero((cabs[:, FROM] != cabs[:, TO]) & (dist[cabs[:, FROM], cabs[:, TO]] == t - cabs[:, TIME_STARTED]))[0]
        for c in arrived.tolist():
            if cabs[c, CLNT_ON_BOARD] == 0:                      # was heading to its customer
                d = self.id_to_row.get(int(cabs[c, CLNT_ASSIGNED]))
                if d is not None:
                    self.d_cab[d] = cabs[c, ID]
                    self.d_pickup_t[d] = t
                    self.m.total_pickup_numb += 1
                    cabs[c, FROM] = self.d_from[d]
                    cabs[c, TO] = self.d_to[d] if self.d_pool_clnt[d] == -1 else cheat_a_bit(int(self.d_from[d]), int(self.d_pool_cost[d]), self.n_stands)
                    cabs[c, CLNT_ASSIGNED] = self.d_id[d]
                    cabs[c, CLNT_ON_BOARD] = 1
                    cabs[c, TIME_STARTED] = t
            else:                                                # a trip has just been completed
                cabs[c, FROM] = cabs[c, TO]
                cabs[c, CLNT_ASSIGNED] = -1
                cabs[c, CLNT_ON_BOARD] = 0
                cabs[c, TIME_STARTED] = -1

    # ---- Simulator.java:329-355 ----------------------------------------------------------------------
    def create_temp_demand(self, t: int) -> List[TempDemand]:
        cand = np.nonzero((self.d_cab == -1) & (t >= self.d_at))[0]
        if len(cand) == 0:
            return []
        late = (t - self.d_at[cand]) >= DROP_TIME
        dropped = cand[late]
        self.d_cab[dropped] = -2
        self.m.total_dropped += len(dropped)
        rest = cand[~late]
        free_to = np.unique(self.cabs[self.cabs[:, CLNT_ASSIGNED] == -1, TO])     # ANY unassigned cab, moving or not
        if len(free_to) == 0:
            return []
        reach = (self.dist[free_to] < DROP_TIME).any(0)                             # per stand
        keep = rest[reach[self.d_from[rest]]]
        return [TempDemand(i, f, t_) for i, f, t_ in zip(self.d_id[keep].tolist(), self.d_from[keep].tolist(), self.d_to[keep].tolist())]

    # ---- Simulator.java:358-372 ----------------------------------------------------------------------
    def create_temp_supply(self) -> List[Tuple[int, int, int]]:
        un_from = np.zeros(self.n_stands, bool)                                     # the WHOLE file, future arrivals too
        un_from[self.d_from[self.d_cab == -1]] = True
        if not un_from.any():
            return []
        reach = (self.dist[:, un_from] < DROP_TIME).any(1)
        c = self.cabs
        sel = np.nonzero((c[:, FROM] == c[:, TO]) & (c[:, CLNT_ASSIGNED] == -1) & reach[c[:, TO]])[0]
        return list(zip(c[sel, ID].tolist(), c[sel, FROM].tolist(), c[sel, TO].tolist()))

    # ---- Simulator.java:681-758 + 760-784 ------------------------------------------------------------
    def find_and_analyze_pool(self, temp_demand: List[TempDemand]) -> List[TempDemand]:
        n = len(temp_demand)
        frm = np.array([d.frm for d in temp_demand], np.int32)
        to = np.array([d.to for d in temp_demand], np.int32)
        pairs = self.backend.pool_pairs(frm, to, self.dist) if n >= 2 else np.zeros((0, 4), np.int32)
        pool_numb = n * (n - 1)                                                     # every ordered pair is accepted (:691)
        self.m.max_POOL_size = max(self.m.max_POOL_size, len(pairs))
        self.m.max_POOL_MEM_size = max(self.m.max_POOL_MEM_size, pool_numb)
        is_b = np.zeros(n, bool)
        pa = np.asarray(pairs).reshape(-1, 4)
        is_b[pa[:, 1]] = True
        a_of = dict(zip(pa[:, 0].tolist(), zip(pa[:, 1].tolist(), pa[:, 2].tolist(), pa[:, 3].tolist())))   # last pair of an `a` wins
        out = []
        for d in np.nonzero(~is_b)[0].tolist():                                     # analyzePool :760-784
            src = temp_demand[d]
            hit = a_of.get(d)
            if hit is None:
                out.append(TempDemand(src.id, src.frm, src.to))
            else:
                out.append(TempDemand(src.id, src.frm, src.to, temp_demand[hit[0]].id, hit[1], hit[2]))
        return out

    # ---- helpers :424-494 ----------------------------------------------------------------------------
    def assign_pooled_customer(self, customer: int, cab: int):
        d = self.id_to_row.get(customer)
        if d is not None:
            self.d_cab[d] = cab
            self.m.total_second_passengers += 1

    def assign_to_cab_and_go(self, t: int, s: int, td: TempDemand):
        c = self.cabs
        c[s, FROM] = td.frm
        c[s, TO] = td.to if td.pool_clnt_id == -1 else cheat_a_bit(td.frm, td.pool_cost, self.n_stands)
        c[s, CLNT_ASSIGNED] = td.id
        c[s, CLNT_ON_BOARD] = 1
        c[s, TIME_STARTED] = t
        self.m.total_pickup_numb += 1

    def go_to_pickup(self, t: int, s: int, td: TempDemand):
        c = self.cabs
        c[s, TO] = td.frm
        c[s, CLNT_ASSIGNED] = td.id
        c[s, CLNT_ON_BOARD] = 0
        c[s, TIME_STARTED] = t
        self.m.total_pickup_time += int(self.dist[c[s, FROM], c[s, TO]])

    def _dispatch_cab(self, t: int, cab_id: int, sup_to: int, td: TempDemand):
        s2 = cab_id                                                                  # cabs[i][ID] == i
        if sup_to == td.frm:
            self.assign_to_cab_and_go(t, s2, td)
        elif self.dist[sup_to, td.frm] < DROP_TIME:
            self.go_to_pickup(t, s2, td)

    # ---- Simulator.java:613-674 ----------------------------------------------------------------------
    def analyze_pairs(self, t: int, pairs, temp_demand: List[TempDemand], temp_supply):
        cab_first = {}
        clnt_first = {}
        for cab, clnt in pairs:                       # "first i with pairs[i].cab == s" / ".clnt == d"
            cab_first.setdefault(int(cab), int(clnt))
            clnt_first.setdefault(int(clnt), int(cab))
        supply2, demand2 = [], []
        for s, (sid, sfrom, sto) in enumerate(temp_supply):
            if s in cab_first:
                self._dispatch_cab(t, sid, sto, temp_demand[cab_first[s]])
            else:
                supply2.append((sid, sfrom, sto))
        for d, td in enumerate(temp_demand):
            if d in clnt_first:
                row = self.id_to_row.get(td.id)
                if row is not None:
                    cab_id = temp_supply[clnt_first[d]][0]
                    self.d_cab[row] = cab_id
                    self.d_pickup_t[row] = t
                    if td.pool_clnt_id > -1:
                        self.assign_pooled_customer(td.pool_clnt_id, cab_id)
                        self.m.total_pickup_numb += 1
            else:
                demand2.append(td)                      # records are not modified after find_and_analyze_pool
        return supply2, demand2

    # ---- Simulator.java:375-421 ----------------------------------------------------------------------
    def analyze_solution(self, x, cost, t: int, temp_demand: List[TempDemand], temp_supply) -> int:
        nn = len(cost)
        total = 0
        if nn == 0:
            return 0
        xm = np.asarray(x).reshape(nn, nn)
        for s, (sid, sfrom, sto) in enumerate(temp_supply):
            if sfrom != sto:
                continue
            hits = np.nonzero((xm[s, : len(temp_demand)] == 1) & (np.asarray(cost[s][: len(temp_demand)]) < BIG_COST))[0]
            if len(hits) == 0:
                continue
            c = int(hits[0])
            td = temp_demand[c]
            total += 1
            row = self.id_to_row.get(td.id)
            if row is not None:
                self.d_cab[row] = sid
                self.d_pickup_t[row] = t
                if td.pool_clnt_id > -1:
                    self.assign_pooled_customer(td.pool_clnt_id, sid)
                    self.d_pool_clnt[row], self.d_pool_plan[row], self.d_pool_cost[row] = td.pool_clnt_id, td.pool_plan, td.pool_cost
                    self.m.total_pickup_numb += 1
            self._dispatch_cab(t, sid, sto, td)
        return total

    def _cost(self, temp_demand, temp_supply):
        return self.backend.cost(self.dist, [s[2] for s in temp_supply], [d.frm for d in temp_demand])

    # ---- Simulator.java:141-218 ----------------------------------------------------------------------
    def step(self, t: int):
        t0 = time.perf_counter()
        self.check_if_cab_at_destination(t)
        temp_demand = self.create_temp_demand(t)
        if not temp_demand:
            return
        temp_supply = self.create_temp_supply()
        line = "t:%d. Initial Count of demand=%d, supply=%d. " % (t, len(temp_demand), len(temp_supply))
        cost = np.zeros((0, 0), np.int32)
        x = []
        if temp_supply:
            temp_demand = self.find_and_analyze_pool(temp_demand)
            cost = self._cost(temp_demand, temp_supply)
            self.m.max_model_size = max(self.m.max_model_size, len(cost))
            if len(cost) > MAX_NON_LCM:
                pairs, lcm_min_val = self.backend.lcm_java(cost)
                self.m.total_LCM_used += 1
                line += "LCM n_pairs=%d" % len(pairs)
                temp_supply, temp_demand = self.analyze_pairs(t, pairs, temp_demand, temp_supply)
                if lcm_min_val == BIG_COST:                       # :188-189 -- nothing left for the solver
                    self.solv_log.append(line)
                    self.m.step_seconds.append(time.perf_counter() - t0)
                    return
                cost = self._cost(temp_demand, temp_supply)
                line += ". Sent to solver: demand=%d, supply=%d. " % (len(temp_demand), len(temp_supply))
            self.m.max_solver_size = max(self.m.max_solver_size, len(cost))
            x = self.backend.solve(len(cost), cost, len(temp_supply), len(temp_demand))
            if len(cost) == 0:
                x = []
        total = self.analyze_solution(x, cost, t, temp_demand, temp_supply)
        line += "; OPT count=%d" % total
        self.solv_log.append(line)
        self.m.step_seconds.append(time.perf_counter() - t0)

    def run(self, steps: int = HOURS * 60):
        t0 = time.perf_counter()
        for t in range(steps):
            self.step(t)
        self.total_simul_time = time.perf_counter() - t0
        return self.solv_log, self.metrics()

    def metrics(self) -> dict:                                     # printMetrics :256-277
        m = self.m
        return {"Total customers": int(len(self.d_id)), "Total dropped customers": m.total_dropped,
                "Total pickedup customers": m.total_pickup_numb,
                "Total customers with assigned cabs": int((self.d_cab > -1).sum()),
                "Total pickup time": m.total_pickup_time, "Max model size": m.max_model_size,
                "Max solver size": m.max_solver_size, "LCM use count": m.total_LCM_used,
                "Max POOL array size": m.max_POOL_MEM_size, "Max POOL size": m.max_POOL_size,
                "Total second customers in POOL": m.total_second_passengers}
