#!/usr/bin/env python
"""bench.py -- the headline benchmark of the dispatch hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--components all|none]
                    [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W

Primary workload (BASELINE.json configs[2], SURVEY.md section 8(d) config 3): the reference's
4-passenger pool search (pool_n.c + findpool.c) over 722 waiting customers -- 8 logical shards by
leading customer, per-shard greedy dedup, merge -- metric "pool plans evaluated / s".  One step =
the whole `findpool` job: 3 042 951 264 leaf plans (pool_n.c:103 count_all), checked against the
reference's known answers every run.  At N > 1 the 8 logical shards are spread over the ranks
(the reference's own fan-out, findpool.c:138-142), survivors are all-gathered over NCCL and merged.

One JSON line on stdout (rank 0).  `value` = device-resident throughput (CUDA events, max over
ranks); `e2e` = the same job through the public host API with host buffers (pinned H2D + D2H
inside the timed region); `roofline` = the dominant kernel (pool_enum_kernel) against the measured
HBM peak using the LOGICAL bytes of SURVEY.md section 8(d) (80 B per evaluated plan + 36 B per
feasible plan); `cpu_baseline` = the reference's own pool_n.c compiled -O3, run on the host cores
on a bounded sample; `components` = the other kernels of the path (K2 20k x 20k time-to-optimal,
K3 LCM/s at 2000 x 2000, K1 cost build GB/s at 20k x 20k), each with its own roofline figure.

`--dump-outputs DIR` writes what the last timed step computed, as float64 .npy files (rank 0):
pool_merged_plans.npy [plans, 9] (pool_n.c record layout: 4 pick-up customers, 4 drop-off
customers, cost) and pool_shard_counters.npy [8, 3] (kept, evaluated, feasible per logical shard).
The inputs are seeded, so two builds can be compared output for output.

`--impl reference` times ONLY the reference CPU implementation (oracle/_ref/pool_n_big64, the
unmodified pool_n.c with its shard count raised so that a step is a bounded 1/8 sample).
"""
from __future__ import annotations

import argparse
import concurrent.futures as cf
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

POOL_N = 722
POOL_K = 4
POOL_STANDS = 50
LOGICAL_B_PER_PLAN = 80      # SURVEY.md 8(d): 4 customers x the 5-int32 demand record (pool_n.c:20)
LOGICAL_B_PER_FEASIBLE = 36  # one pool[] record (pool_n.c:26)


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            d = json.load(open(p))
            return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---------------------------------------------------------------------------------------------------
# clocks sampling during the timed region
# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index=0):
        self.index = index
        self.samples = []
        self._stop = threading.Event()
        self._t = None

    def _run_nvml(self):
        """In-process NVML sampling (about 200 Hz) -- an nvidia-smi subprocess takes longer than a short timed region."""
        import pynvml as nv
        nv.nvmlInit()
        h = nv.nvmlDeviceGetHandleByIndex(self.index)
        mx = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        bits = [getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8), getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)]
        while not self._stop.is_set():
            r = get_reasons(h)
            self.samples.append([str(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)), str(mx)] +
                                ["Active" if (r & b) else "Not Active" for b in bits])
            self._stop.wait(0.005)

    def _run(self):
        try:
            self._run_nvml()
            return
        except Exception:
            pass
        while not self._stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                f = [x.strip() for x in out.strip().split(",")]
                if len(f) >= 6:
                    self.samples.append(f)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        self._t = threading.Thread(target=self._run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(timeout=6)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        mhz = [int(s[0]) for s in self.samples if s[0].isdigit()]
        mx = [int(s[1]) for s in self.samples if s[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names) if any(s[2 + k].lower().startswith("active") for s in self.samples)]
        return {"sm_mhz": statistics.median(mhz) if mhz else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(self.samples)}


# ---------------------------------------------------------------------------------------------------
# the reference CPU arm (also the cpu_baseline of our arm)
# ---------------------------------------------------------------------------------------------------
def _run_ref_slice(args):
    exe, csv_path, n, k, t = args
    with tempfile.TemporaryDirectory() as td:
        res = subprocess.run([exe, str(k), str(t), csv_path, str(n), os.path.join(td, "out.csv")], cwd=td,
                             capture_output=True, text=True)
    m = re.search(r"Count ALL: (\d+)", res.stdout)
    return int(m.group(1)) if m else 0


def reference_sample(n_slices=8, ways=64):
    """One bounded sample of config 3 on the host cores: slices 0..n_slices-1 of a `ways`-way shard rule of the
    UNMODIFIED pool_n.c (oracle/_ref/pool_n_big64 or _big512), one process per slice, all at once (the way
    findpool.c:138-142 fans out).  Returns (plans, seconds, processes)."""
    from oracle import gen_inputs as g
    exe = os.path.join(ROOT, "oracle", "_ref", "pool_n_big%d" % ways)
    if not os.path.exists(exe):
        from oracle import _clib
        _clib.build_ref()
    if not os.path.exists(exe):
        raise FileNotFoundError(exe)
    dem = g.pool_demand(POOL_N)
    with tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False) as f:
        f.write(g.demand_csv(dem))
        csv_path = f.name
    procs = min(n_slices, os.cpu_count() or 1)
    try:
        t0 = time.perf_counter()
        with cf.ThreadPoolExecutor(procs) as ex:
            counts = list(ex.map(_run_ref_slice, [(exe, csv_path, POOL_N, POOL_K, t) for t in range(n_slices)]))
        dt = time.perf_counter() - t0
    finally:
        os.unlink(csv_path)
    return sum(counts), dt, procs


def _host_procs():
    """One pool_n process per host core, at most 16 (the reference fans out 8, findpool.c:138-142; more cores get more)."""
    return max(1, min(os.cpu_count() or 1, 16))


def sample_text_64(n_slices):
    return "leading customers 0..%d of 722 (slices 0-%d of a 64-way pool_n.c shard rule, one process per slice)" % (
        12 * n_slices - 1, n_slices - 1)
SAMPLE_TEXT_512 = "leading customers 0..%d of 722 (%d slices of a 512-way pool_n.c shard rule, one process per slice)"


def reference_whole_job(check=False):
    """ONE step of the reference arm = the whole config-3 job the way findpool.c runs it: the 8 stock shards
    (`pool_n 4 t demand.csv 722 out.csv`, t = 0..7, one OS process each, all at once -- findpool.c:138-142) followed by
    the merge (findpool.c:83-108, restated in oracle/pool_oracle.c; findpool.c itself is Windows process plumbing).
    Returns (leaf plans evaluated, seconds, processes)."""
    from oracle import gen_inputs as g, pool_ref
    exe = os.path.join(ROOT, "oracle", "_ref", "pool_n_big")
    if not os.path.exists(exe):
        from oracle import _clib
        _clib.build_ref()
    if not os.path.exists(exe):
        raise FileNotFoundError(exe)
    dem = g.pool_demand(POOL_N)
    with tempfile.TemporaryDirectory() as td:
        csv_path = os.path.join(td, "demand.csv")
        with open(csv_path, "w") as f:
            f.write(g.demand_csv(dem))
        for t in range(8):
            os.mkdir(os.path.join(td, "s%d" % t))
        t0 = time.perf_counter()
        procs = [subprocess.Popen([exe, str(POOL_K), str(t), csv_path, str(POOL_N), "out.csv"], cwd=os.path.join(td, "s%d" % t),
                                  stdout=subprocess.PIPE, text=True) for t in range(8)]
        outs = [p.communicate()[0] for p in procs]
        shard_plans = [pool_ref.parse_result_csv(open(os.path.join(td, "s%d" % t, "out.csv")).read(), POOL_K) for t in range(8)]
        merged = pool_ref.merge(shard_plans, POOL_N, POOL_K)
        dt = time.perf_counter() - t0
    counts = [int(re.search(r"Count ALL: (\d+)", o).group(1)) for o in outs]
    if check:
        assert counts == g.POOL722_EVALUATED and len(merged) == 110 and int(merged[:, 8].sum()) == 1840, "reference arm result"
    return sum(counts), dt, 8


def run_reference_arm(args, rank):
    if rank != 0:
        return
    try:
        # every step is the WHOLE job (8 stock pool_n processes + merge), the same config our arm times
        for i in range(args.warmup):
            reference_whole_job(check=(i == 0))
        t_tot, plans_tot, procs = 0.0, 0, 8
        for i in range(args.steps):
            plans, dt, procs = reference_whole_job(check=(i == 0 and args.warmup == 0))
            t_tot += dt
            plans_tot += plans
        val = plans_tot / t_tot
        how = "whole job per step: 8 stock pool_n.c -O3 processes (findpool.c:138-142) + merge, %d host cores" % (os.cpu_count() or 0)
        line = {"impl": "reference", "metric": "pool plans evaluated per second", "value": val, "unit": "plans/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_tot / args.steps,
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
                "config": {"workload": "pool_n 4-passenger pool search, 722 customers, 8 logical shards + merge "
                                       "(BASELINE.json configs[2], SURVEY 8(d) config 3)",
                           "pool_size": POOL_K, "customers": POOL_N, "stands": POOL_STANDS, "max_wait": 3, "max_loss_pct": 1,
                           "plans_per_step": plans_tot // args.steps},
                "cpu_baseline": {"value": val, "unit": "plans/s", "cores": procs, "kind": "reference", "sample": how},
                "e2e": {"value": val, "unit": "plans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
    except Exception as e:  # the oracle always exists; report instead of crashing the driver
        line = {"impl": "reference", "unavailable": "%s: %s" % (type(e).__name__, e)}
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--components", default="all", choices=["all", "none"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--pool-large", type=int, default=5000, help="customers of the north-star pool component (0: skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's results to DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the results of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else max(args.warmup, 0)

    rank, world, local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.impl == "reference":
        run_reference_arm(args, rank)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    from oracle import gen_inputs as g       # inputs + known answers (checker only)
    from taxidispatcher_b200 import _lib, dispatch, parallel

    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"   # keep stdout to the single JSON line (NCCL prints its version there)
        import datetime
        # a rank that fails between two collectives must not leave the others waiting for ever
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=240))
    lib = _lib.lib()
    eng = dispatch.Engine()
    dev = eng.device
    hbm_peak, peak_src = measured_peaks()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    flush_buf = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def flush_l2():
        flush_buf.fill_(1)

    # ---- pool job, device resident ---------------------------------------------------------------
    dem_np = g.pool_demand(POOL_N)
    dist_np = g.stand_distances(POOL_STANDS)
    dem_d = torch.from_numpy(dem_np).to(dev)
    dist_d = torch.from_numpy(dist_np).to(dev)
    my_shards = parallel.shards_for_rank(rank, world)     # contiguous block of logical shards
    slots = (8 + world - 1) // world
    cap = POOL_N // 2 + 1
    # headed blocks (td_pool_find_shards_headed): a shard's survivors, their count and its counters travel together, so
    # the multi-GPU step needs ONE collective; padding slots (ranks with fewer shards) keep their zero count for ever
    blocks = torch.zeros((slots, cap + 1, 9), dtype=torch.int32, device=dev)
    all_blocks = torch.zeros((world * slots, cap + 1, 9), dtype=torch.int32, device=dev)
    slot_plans = torch.zeros((slots, cap, 9), dtype=torch.int32, device=dev)
    slot_counts = torch.zeros(slots, dtype=torch.int32, device=dev)
    slot_shard_l, slot_real = [], []
    for r in range(world):
        sh_r = parallel.shards_for_rank(r, world)
        slot_shard_l += sh_r + [0] * (slots - len(sh_r))   # padding slots carry count 0
        slot_real += [True] * len(sh_r) + [False] * (slots - len(sh_r))
    slot_shard = torch.tensor(slot_shard_l, dtype=torch.int32, device=dev)

    def pool_step(want_stats=False):
        if want_stats:                                       # synchronous sizing / checking call (untimed)
            stats = []
            if my_shards:
                _, _, stats = eng.pool_find_shards(dem_d, dist_d, POOL_K, my_shards[0], len(my_shards), 8,
                                                   out=slot_plans[: len(my_shards)], counts_out=slot_counts[: len(my_shards)],
                                                   want_stats=True)
        else:
            stats = []
        if my_shards:                                        # ONE asynchronous device call for all of this rank's shards
            eng.pool_find_shards_headed(dem_d, dist_d, POOL_K, my_shards[0], len(my_shards), 8, out=blocks[: len(my_shards)])
        if world > 1:
            dist.all_gather_into_tensor(all_blocks, blocks)  # the only collective of the step
            src = all_blocks
        else:
            src = blocks
        merged = cnt = None
        if rank == 0:
            merged, cnt = eng.pool_merge_headed(src, slot_shard, POOL_N, POOL_K)
        return merged, cnt, stats

    # correctness gate (also the first warm-up): counts and merged result must equal the known answers
    merged, cnt, stats = pool_step(want_stats=True)
    torch.cuda.synchronize()
    ev_local = sum(int(s.evaluated) for s in stats)
    fe_local = sum(int(s.feasible) for s in stats)
    for st, sh in zip(stats, my_shards):
        assert int(st.evaluated) == g.POOL722_EVALUATED[sh] and int(st.feasible) == g.POOL722_FEASIBLE[sh], \
            "pool counts differ from the reference's known answers (shard %d)" % sh
    tot = torch.tensor([ev_local, fe_local], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(tot)
    plans_per_step, feas_per_step = int(tot[0]), int(tot[1])
    if rank == 0:
        m = merged[: int(cnt.item())].cpu().numpy()
        assert len(m) == 110 and int(m[:, 8].sum()) == 1840, "merged pool result differs from KAT P2"
        golden = json.load(open(os.path.join(ROOT, "tests", "golden", "pool722.json")))["merged"]
        assert m.tolist() == golden, "merged pool result differs from tests/golden/pool722.json"
    for _ in range(args.warmup - 1):
        pool_step()
    barrier()

    lib.td_prof_reset()
    lib.td_prof_enable(1)
    lib.td_launch_count_reset()
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps)]
    with ClockSampler(local_rank) as clocks:
        barrier()
        for i in range(args.steps):
            flush_l2()
            ev0[i].record()
            merged_last = pool_step()[:2]
            ev1[i].record()
        barrier()
    launches = int(lib.td_launch_count())
    lib.td_prof_enable(0)
    # the timed steps ran asynchronously (no host round trip): make sure the last one was a complete, valid job
    assert int(blocks[: max(len(my_shards), 1), 0, 0].min().item()) >= 0, "record list overflowed inside the timed region"
    if rank == 0:
        last = merged_last[0][: int(merged_last[1].item())].cpu().numpy()
        assert last.tolist() == golden, "timed steps produced a different result than the golden merge"
        if args.dump_outputs:
            headers = (all_blocks if world > 1 else blocks)[:, 0, :].cpu().numpy()[slot_real]   # shard order
            kept, evaluated, feasible = dispatch.Engine.headers_host_view(headers)
            os.makedirs(args.dump_outputs, exist_ok=True)
            np.save(os.path.join(args.dump_outputs, "pool_merged_plans.npy"), last.astype(np.float64))
            np.save(os.path.join(args.dump_outputs, "pool_shard_counters.npy"),
                    np.stack([kept, evaluated, feasible], axis=1).astype(np.float64))
    step_ms = [a.elapsed_time(b) for a, b in zip(ev0, ev1)]
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX)
    total_ms = float(total_ms.item())
    value = plans_per_step * args.steps / (total_ms * 1e-3)

    # dominant kernel: pool_enum (per-launch average over the timed region, this rank's shards)
    import ctypes
    pm, pc = ctypes.c_double(), ctypes.c_int64()
    lib.td_prof_read(_lib.PROF_POOL_ENUM, ctypes.byref(pm), ctypes.byref(pc))
    enum_ms, enum_n = pm.value, pc.value
    lib.td_prof_read(_lib.PROF_POOL_SELECT, ctypes.byref(pm), ctypes.byref(pc))
    sel_ms = pm.value
    lib.td_prof_reset()
    bytes_per_launch = float(LOGICAL_B_PER_PLAN * ev_local + LOGICAL_B_PER_FEASIBLE * fe_local)  # one launch = all local shards
    avg_enum_ms = enum_ms / max(enum_n, 1)
    hbm_logical = bytes_per_launch / (avg_enum_ms * 1e-3) / 1e9 if avg_enum_ms > 0 else 0.0
    # The kernel's real bound is warp-instruction ISSUE (INT32 + shared-memory look-ups; DRAM traffic is ~1 % of peak):
    # achieved = warp instructions of the launch / its measured duration, peak = 4 issue slots x SMs x SM clock.
    # The instruction count of a launch is a property of the input (deterministic): it comes from the committed ncu
    # capture of this very launch shape (profiles/traffic.json, smsp__inst_executed.sum), the duration is measured live.
    prof = {}
    try:
        prof = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    except Exception:
        prof = {}
    k4 = prof.get("pool_enum_k4_config3", {})
    inst_per_plan = k4.get("warp_inst_per_plan")
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    clk = clocks.summary()
    sm_hz = 1e6 * float(clk["sm_mhz"] or 1965.0)
    peak_issue = 4.0 * sms * sm_hz / 1e9                     # G warp-instructions / s
    achieved_issue = (inst_per_plan * ev_local / (avg_enum_ms * 1e-3) / 1e9) if (inst_per_plan and avg_enum_ms > 0) else None
    roofline = {"bound": "int32_issue", "kernel": "pool_enum_kernel<4>", "achieved": achieved_issue, "peak": peak_issue,
                "unit": "Gwarp-inst/s", "frac": (achieved_issue / peak_issue) if achieved_issue else None,
                "traffic": k4.get("dram_bytes_per_launch"),
                "peak_source": "4 issue slots x %d SMs x %.0f MHz (median SM clock sampled during the timed region)" % (sms, sm_hz / 1e6),
                "warp_inst_per_plan": inst_per_plan, "warp_inst_source": k4.get("source"),
                "issue_active_pct_ncu": k4.get("issue_active_pct"),
                "hbm_logical": {"achieved": hbm_logical, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_logical / hbm_peak,
                                "peak_source": peak_src,
                                "note": "SURVEY 8(d) LOGICAL bytes (80 B per evaluated plan + 36 B per feasible plan): a label "
                                        "for north_star's HBM fraction, not traffic -- the kernel moves ~0.03 B per plan"},
                "avg_launch_ms": avg_enum_ms, "launches": enum_n, "share_of_step": enum_ms / max(sum(step_ms), 1e-9),
                "pool_select_share_of_step": sel_ms / max(sum(step_ms), 1e-9)}

    # ---- e2e: the public host API with host buffers ----------------------------------------------
    e2e_steps = args.steps

    def e2e_step():
        if world == 1:
            return dispatch.find_pool_all(dem_np, dist_np, POOL_K)
        return parallel.find_pool_sharded(dem_np, dist_np, POOL_K)

    for _ in range(5):     # warm-up: call 1 sizes the record list, 2-3 take the asynchronous path, 4-5 the captured graph
        e2e_step()
    barrier()
    copied0 = dict(dispatch.COPIED)
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        m_e2e, st_e2e = e2e_step()
    barrier()
    e2e_s = time.perf_counter() - t0
    # bytes counted at the copy sites of the public API (dispatch._h2d_i32 / _d2h / pool_read_stats), per step, this rank
    h2d = (dispatch.COPIED["h2d"] - copied0["h2d"]) // e2e_steps
    d2h = (dispatch.COPIED["d2h"] - copied0["d2h"]) // e2e_steps
    e2e_t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX)
    e2e_s = float(e2e_t.item())
    if rank == 0:
        assert len(m_e2e) == 110 and st_e2e["evaluated"] == plans_per_step
        golden_m = json.load(open(os.path.join(ROOT, "tests", "golden", "pool722.json")))["merged"]
        assert np.asarray(m_e2e).tolist() == golden_m, "e2e pool result differs from tests/golden/pool722.json"
    e2e = {"value": plans_per_step * e2e_steps / e2e_s, "unit": "plans/s", "h2d_bytes_per_step": h2d,
           "d2h_bytes_per_step": d2h, "steps": e2e_steps, "ms_per_step": 1e3 * e2e_s / e2e_steps,
           "api": "taxidispatcher_b200.find_pool_all(demand, dist, 4)" if world == 1 else
                  "taxidispatcher_b200.parallel.find_pool_sharded(demand, dist, 4)"}

    # ---- north-star scale: 4-passenger pool over 5000 customers, sharded like the 722 job -----------
    pool_large = None
    if args.components == "all" and args.pool_large > 0:
        try:
            pool_large = run_pool_large(torch, dist, np, g, eng, parallel, args.pool_large, rank, world, hbm_peak)
        except Exception as e:
            pool_large = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---- N > 1: independent dispatch instances, one complete 722-customer job per GPU (weak scaling view) ----
    replicas = None
    if world > 1 and args.components == "all":
        replicas = run_replica_jobs(torch, dist, eng, dem_d, dist_d, world, plans_per_step, steps=min(args.steps, 30))

    # ---- K1 with the cab rows split across the ranks (north_star), 20k x 20k, 4000 stands ----------------------------
    cost_sharded = None
    if args.components == "all":
        try:
            cost_sharded = run_cost_sharded(torch, dist, np, g, eng, parallel, rank, world, hbm_peak, flush_l2)
        except Exception as e:
            cost_sharded = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---- config 5: split.py 4-way regional split of the 20k x 20k instance, ranges spread over the ranks ---
    split_comp = None
    if args.components == "all":
        try:
            split_comp = run_split_component(np, g, world)
        except Exception as e:
            split_comp = {"error": "%s: %s" % (type(e).__name__, e)}

    # ---- CPU baseline + the other kernels (rank 0, N = 1 only) -----------------------------------
    cpu_baseline = None
    components = {}
    if rank == 0 and world == 1:
        if not args.no_cpu_baseline:
            try:
                n_sl = _host_procs()
                plans, dt, procs = reference_sample(n_sl)
                plans2, dt2, _ = reference_sample(n_sl)
                cpu_baseline = {"value": (plans + plans2) / (dt + dt2), "unit": "plans/s", "cores": procs, "kind": "reference",
                                "sample": sample_text_64(n_sl) + ", run twice", "host_cores": os.cpu_count()}
            except Exception as e:
                cpu_baseline = {"value": None, "unit": "plans/s", "cores": 0, "kind": "reference", "sample": "failed: %s" % e}
        if args.components == "all":
            try:
                components = run_components(torch, np, g, eng, lib, _lib, dispatch, hbm_peak, flush_l2)
            except Exception as e:
                components = {"error": "%s: %s" % (type(e).__name__, e)}
            try:
                components["simulator_replay"] = run_simulator_component()
            except Exception as e:
                components["simulator_replay"] = {"error": "%s: %s" % (type(e).__name__, e)}
    if pool_large is not None:
        components["pool_%d" % args.pool_large] = pool_large
    if cost_sharded is not None:
        components["cost_matrix_20k_rows_per_rank"] = cost_sharded
    if split_comp is not None:
        components["split_20k_4way"] = split_comp
    if replicas is not None:
        components["pool_722_one_job_per_gpu"] = replicas

    if world > 1:
        dist.barrier()
    if rank == 0:
        line = {"metric": "pool plans evaluated per second", "value": value, "unit": "plans/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
                "scaling": "strong", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
                "config": {"workload": "pool_n 4-passenger pool search, 722 customers, 8 logical shards + merge "
                                       "(BASELINE.json configs[2], SURVEY 8(d) config 3)",
                           "pool_size": POOL_K, "customers": POOL_N, "stands": POOL_STANDS, "max_wait": 3, "max_loss_pct": 1,
                           "plans_per_step": plans_per_step, "feasible_per_step": feas_per_step,
                           "parallelism": "8 logical shards in contiguous blocks over %d rank(s), all_gather + merge" % world,
                           "l2": "256 MiB write between steps (untimed); inputs are 15 KB"},
                "e2e": e2e, "gpu_launches": launches, "clocks": clocks.summary(), "roofline": roofline,
                "cpu_baseline": cpu_baseline, "components": components}
        print(json.dumps(line), flush=True)
    dispatch.release_pool_graphs()
    if world > 1:
        dist.destroy_process_group()


def run_pool_large(torch, dist, np, g, eng, parallel, n_cust, rank, world, hbm_peak):
    """north_star: 4-passenger pool over >= 5k waiting customers.  The feasible set (~4e10 plans at 5000
    customers) does not fit in memory, so td_pool_find_shards runs its cost-window passes (SURVEY 'hard parts':
    pool result capacity).  Each rank takes its contiguous block of the 8 logical shards; plans/s = all leaf
    plans of the job / max-over-ranks device time.  Checked through size-independent properties."""
    dem_np = g.pool_demand(n_cust, seed=n_cust)
    dist_np = g.stand_distances(POOL_STANDS)
    dev = eng.device
    dem_d, dist_d = torch.from_numpy(dem_np).to(dev), torch.from_numpy(dist_np).to(dev)
    mine = parallel.shards_for_rank(rank, world)
    slots = (8 + world - 1) // world
    cap = n_cust // 2 + 1
    slot_plans = torch.zeros((slots, cap, 9), dtype=torch.int32, device=dev)
    slot_counts = torch.zeros(slots, dtype=torch.int32, device=dev)
    # record list of 1.6e9 plans = 4 x 25.6 GB of the 180 GB HBM: the ~4e10 feasible plans then need 10 cost windows
    # instead of 40 (every window re-enumerates).  Falls back to 2e8 records if the allocation fails.  The workspace is
    # allocated BEFORE the timed region (a 100 GB cudaMalloc takes 0.1-0.3 s and is not part of the path).
    records = int(os.environ.get("TD_BENCH_POOL_RECORDS", "1600000000"))
    if mine:
        try:
            eng._workspace("pool", eng.lib.td_pool_shards_workspace_bytes(n_cust, POOL_STANDS, POOL_K, len(mine), records))
        except torch.OutOfMemoryError:
            eng._ws.pop("pool", None)
            torch.cuda.empty_cache()
            records = 200_000_000
            eng._workspace("pool", eng.lib.td_pool_shards_workspace_bytes(n_cust, POOL_STANDS, POOL_K, len(mine), records))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    st = []
    if mine:
        _, _, st = eng.pool_find_shards(dem_d, dist_d, POOL_K, mine[0], len(mine), 8, max_feasible=records,
                                        out=slot_plans[: len(mine)], counts_out=slot_counts[: len(mine)])
    if world > 1:
        allp = torch.zeros((world * slots, cap, 9), dtype=torch.int32, device=dev)
        allc = torch.zeros(world * slots, dtype=torch.int32, device=dev)
        dist.all_gather_into_tensor(allp, slot_plans)
        dist.all_gather_into_tensor(allc, slot_counts)
    else:
        allp, allc = slot_plans, slot_counts
    sl = []
    for r in range(world):
        sh_r = parallel.shards_for_rank(r, world)
        sl += sh_r + [0] * (slots - len(sh_r))
    merged, mcnt = eng.pool_merge_padded(allp, allc, torch.tensor(sl, dtype=torch.int32, device=dev), n_cust, POOL_K)
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
    tot = torch.tensor([sum(int(s.evaluated) for s in st), sum(int(s.feasible) for s in st)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot)
    sec = float(ms.item()) * 1e-3
    ev, fe = int(tot[0]), int(tot[1])
    # properties (rank 0): merged plans are customer-disjoint, sorted by cost, each one feasible under the
    # reference's wait and detour rules (formulas of SURVEY 8(a)), and every shard's survivors lead in their shard
    m = merged[: int(mcnt.item())].cpu().numpy()
    ok = True
    if rank == 0 and len(m):
        F, T, W, L = (dem_np[:, k].astype(np.int64) for k in (1, 2, 3, 4))
        p, q, cost = m[:, :4], m[:, 4:8], m[:, 8]
        ok = ok and bool((np.diff(cost) >= 0).all()) and len(set(p.ravel().tolist())) == p.size
        legs = dist_np[F[p[:, :-1]], F[p[:, 1:]]]
        cum = np.concatenate([np.zeros((len(p), 1), np.int64), np.cumsum(legs, 1)], 1)
        first = dist_np[F[p[:, -1]], T[q[:, 0]]]
        drops = dist_np[T[q[:, :-1]], T[q[:, 1:]]]
        ok = ok and bool((cum <= W[p]).all()) and bool((legs.sum(1) + first + drops.sum(1) == cost).all())
        dcum = np.concatenate([np.zeros((len(p), 1), np.int64), np.cumsum(drops, 1)], 1) + first[:, None]
        for d in range(4):
            c = q[:, d]
            pos = (p == c[:, None]).argmax(1)
            suffix = np.array([legs[i, pos[i]:].sum() for i in range(len(p))])
            ok = ok and bool((suffix + dcum[:, d] <= dist_np[F[c], T[c]] * (1 + L[c] / 100.0)).all())
    per_gpu = ev / sec / world
    return {"customers": n_cust, "seconds": sec, "plans_evaluated": ev, "feasible": fe, "merged_plans": int(len(m)),
            "plans_per_s": ev / sec, "enumeration_passes": int(st[0].passes) if st else None, "record_capacity": records,
            "properties_ok": bool(ok),
            "roofline": pool_large_roofline(torch, dev, per_gpu, hbm_peak)}


def pool_large_roofline(torch, dev, plans_per_s_per_gpu, hbm_peak):
    """Issue-slot view of the whole 5000-customer call (all enumeration passes, selections and the merge are inside the
    time, so this is a LOWER bound of the enumeration kernel's own fraction).  Instructions per leaf plan come from the
    committed ncu capture of one slice of this input (profiles/traffic.json); the SM clock is the device's maximum."""
    try:
        k = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get("pool_enum_k4_5000", {})
    except Exception:
        k = {}
    ipp = k.get("warp_inst_per_plan")
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    try:
        mhz = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["sm_max_mhz"])
    except Exception:
        mhz = 1965.0
    peak = 4.0 * sms * mhz * 1e6 / 1e9
    ach = ipp * plans_per_s_per_gpu / 1e9 if ipp else None
    return {"bound": "int32_issue", "achieved": ach, "peak": peak, "unit": "Gwarp-inst/s", "frac": (ach / peak) if ach else None,
            "warp_inst_per_plan": ipp, "warp_inst_source": k.get("source"),
            "scope": "per GPU, whole call (every enumeration pass, selection and merge inside the time)",
            "hbm_logical": {"achieved": plans_per_s_per_gpu * LOGICAL_B_PER_PLAN / 1e9, "peak": hbm_peak, "unit": "GB/s",
                            "frac": plans_per_s_per_gpu * LOGICAL_B_PER_PLAN / 1e9 / hbm_peak,
                            "note": "SURVEY 8(d) logical bytes (80 B per evaluated plan): north_star's 'fraction of the HBM "
                                    "roofline' label, not traffic"}}


def run_cost_sharded(torch, dist, np, g, eng, parallel, rank, world, hbm_peak, flush_l2):
    """calculate_cost (split.py:123-136) on config 5-B with the cab rows split across the ranks: every rank builds its
    contiguous block of the 20 000 x 20 000 matrix on its own device, no exchange.  Device-timed (CUDA events), max over
    ranks; bytes = the block written + the index vectors + the stand rows read."""
    n, S = 20000, 4000
    cab_to, cust_from = g.config5b()
    dev = eng.device
    dist_d = torch.from_numpy(g.stand_distances(S)).to(dev)
    cab_d, cust_d = torch.from_numpy(cab_to).to(dev), torch.from_numpy(cust_from).to(dev)
    lo, hi = parallel.rows_for_rank(n, rank, world)
    out = torch.empty((hi - lo, n), dtype=torch.int32, device=dev)
    for _ in range(3):
        eng.cost_matrix(dist_d, cab_d, cust_d, out=out, rows=(lo, hi))
    torch.cuda.synchronize()
    ms = []
    for _ in range(7):
        flush_l2()
        if world > 1:
            dist.barrier()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        eng.cost_matrix(dist_d, cab_d, cust_d, out=out, rows=(lo, hi))
        b.record()
        torch.cuda.synchronize()
        ms.append(a.elapsed_time(b))
    med = torch.tensor([statistics.median(ms)], dtype=torch.float64, device=dev)
    chk = out.sum(dtype=torch.int64).reshape(1)
    if world > 1:
        dist.all_reduce(med, op=dist.ReduceOp.MAX)
        dist.all_reduce(chk)
    ok = int(chk.item()) == int(np.abs(cab_to[:, None].astype(np.int64) - cust_from[None, :]).sum())
    sec = float(med.item()) * 1e-3
    per_gpu_bytes = 4.0 * (hi - lo) * n + 4.0 * (hi - lo + n) + 4.0 * min(hi - lo, S) * S
    total_bytes = 4.0 * n * n + 4.0 * 2 * n * world
    return {"rows_per_rank": hi - lo, "ms": sec * 1e3, "checksum_ok": bool(ok), "ranks": world,
            "gbs_per_gpu": per_gpu_bytes / sec / 1e9, "gbs_aggregate": total_bytes / sec / 1e9,
            "roofline": {"bound": "hbm", "achieved": per_gpu_bytes / sec / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": per_gpu_bytes / sec / 1e9 / hbm_peak,
                         "note": "write-only kernel: the device's measured fill bandwidth is 7.3 TB/s, its copy bandwidth (peak) 6.45 TB/s"},
            "api": "taxidispatcher_b200.parallel.cost_matrix_sharded / Engine.cost_matrix(rows=rows_for_rank(n, rank, world))"}


def run_replica_jobs(torch, dist, eng, dem_d, dist_d, world, plans_per_job, steps):
    """Batches of independent dispatch instances (north_star): every rank runs the WHOLE config-3 job (8 logical shards +
    merge) on its own GPU, no collective on the data path.  Aggregate plans/s = world x plans per job / max-over-ranks
    device time -- the weak-scaling companion of the headline, which splits ONE job over the ranks."""
    dev = eng.device
    cap = POOL_N // 2 + 1
    plans = torch.zeros((8, cap, 9), dtype=torch.int32, device=dev)
    counts = torch.zeros(8, dtype=torch.int32, device=dev)

    def job():
        eng.pool_find_shards(dem_d, dist_d, POOL_K, 0, 8, 8, out=plans, counts_out=counts, want_stats=False)
        return eng.pool_merge_padded(plans, counts, None, POOL_N, POOL_K)

    ok, elapsed = 1, 0.0
    try:
        # the first, synchronous call sizes the record list for 8 shards (asynchronous calls cannot grow it)
        eng.pool_find_shards(dem_d, dist_d, POOL_K, 0, 8, 8, out=plans, counts_out=counts, want_stats=True)
        for _ in range(3):
            job()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            merged, cnt = job()
        e1.record()
        torch.cuda.synchronize()
        ok = 1 if int(cnt.item()) == 110 else 0
        elapsed = e0.elapsed_time(e1)
    except Exception:
        ok = 0
    # every rank reaches the collectives whatever happened above
    ms = torch.tensor([elapsed, float(1 - ok)], dtype=torch.float64, device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    if float(ms[1]) > 0:
        return {"error": "a replica job failed its known-answer check"}
    per_job_ms = float(ms[0]) / steps
    return {"jobs_per_step": world, "ms_per_step": per_job_ms, "plans_per_s": world * plans_per_job / (per_job_ms * 1e-3),
            "scaling": "weak", "steps": steps, "l2": "not flushed between steps (inputs are 15 KB)"}


def run_split_component(np, g, world):
    """split.py:61-119 on config 5-B (20 000 cabs and customers over 4000 stands): four regional instances
    (one per rank when there are ranks to spare) + the dependent leftover solve.  Wall clock around the reference-shaped
    Python call, host lists in, total cost out (every rank returns the same number)."""
    from taxidispatcher_b200 import experiments
    S = 4000
    cab_to, cust_from = g.config5b()
    distances = g.stand_distances(S)
    cabs = [(i, 0, int(t)) for i, t in enumerate(cab_to)]
    demand = [(i, int(f), 0) for i, f in enumerate(cust_from)]
    experiments.solve_split(S, distances, demand[:2000], cabs[:2000], distributed=world > 1)   # warm-up (workspaces)
    t0 = time.perf_counter()
    total = experiments.solve_split(S, distances, demand, cabs, distributed=world > 1)
    dt = time.perf_counter() - t0
    closed = int(np.abs(np.sort(cab_to).astype(np.int64) - np.sort(cust_from).astype(np.int64)).sum())   # |a-b| costs: sorted matching
    return {"seconds": dt, "split_total_cost": int(total), "unsplit_optimum": closed,
            "instances": "4 ranges of 1000 stands + leftover solve", "ranks": world,
            "api": "taxidispatcher_b200.experiments.solve_split(4000, distances, demand, cabs)"}


def run_simulator_component():
    """Config 4: replay of simulations/taxi_demand.txt (120 one-minute dispatch batches, 42 161 customers)."""
    import gzip
    from taxidispatcher_b200 import formats
    from taxidispatcher_b200.simulator import Simulator
    rows = formats.read_taxi_demand(gzip.open(os.path.join(ROOT, "tests", "golden", "taxi_demand.txt.gz"), "rt").read())
    gold = [ln for ln in open(os.path.join(ROOT, "tests", "golden", "simulog_solv.txt")).read().split("\n") if ln.startswith("t:")]
    sim = Simulator(rows)
    t0 = time.perf_counter()
    log, met = sim.run(120)
    sec = time.perf_counter() - t0
    match = 0
    for a, b in zip(log, gold):
        if a != b:
            break
        match += 1
    out = {"seconds_120_steps": sec, "kernel_seconds": {k: round(v, 4) for k, v in sim.backend.times.items()},
           "golden_log_lines_identical": match, "reference_seconds": 2603,
           "metrics": {k: met[k] for k in ("Total dropped customers", "Total pickedup customers", "Max model size",
                                           "Max solver size", "Max POOL size", "Total second customers in POOL")}}
    try:
        from oracle.sim_backend import OracleBackend
        ref = Simulator(rows, backend=OracleBackend())
        t0 = time.perf_counter()
        ref.run(120)
        out["cpu_oracle_seconds"] = time.perf_counter() - t0
        out["cpu_oracle_kernel_seconds"] = {k: round(v, 3) for k, v in ref.backend.times.items()}
    except Exception as e:
        out["cpu_oracle_seconds"] = "failed: %s" % e
    return out


def run_components(torch, np, g, eng, lib, _lib, dispatch, hbm_peak, flush_l2):
    """K1 / K2 / K3 on their BASELINE.json shapes (config 5 and config 2), device timings with CUDA events."""
    import ctypes
    out = {}

    def timed(fn, reps, warm=1):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        ms = []
        for _ in range(reps):
            flush_l2()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            r = fn()
            b.record()
            torch.cuda.synchronize()
            ms.append(a.elapsed_time(b))
        return ms, r

    # K1: 20k x 20k cost build, 4000 stands (config 5-B)
    n = 20000
    cab_to, cust_from = g.config5b()
    dist_d = torch.from_numpy(g.stand_distances(4000)).cuda()
    cab_d, cust_d = torch.from_numpy(cab_to).cuda(), torch.from_numpy(cust_from).cuda()
    cost_b = torch.empty((n, n), dtype=torch.int32, device="cuda")
    ms, _ = timed(lambda: eng.cost_matrix(dist_d, cab_d, cust_d, out=cost_b), reps=5, warm=3)
    k1_bytes = 4 * n * n + 4 * 2 * n + 4 * 4000 * 4000
    best = min(ms)
    out["cost_matrix_20k"] = {"ms": statistics.median(ms), "ms_best": best, "bytes": k1_bytes,
                              "roofline": {"bound": "hbm", "achieved": k1_bytes / (statistics.median(ms) * 1e-3) / 1e9,
                                           "peak": hbm_peak, "unit": "GB/s",
                                           "frac": k1_bytes / (statistics.median(ms) * 1e-3) / 1e9 / hbm_peak}}
    # K2: exact 20k x 20k, config 5-B (stand derived) and 5-A (U[1,39])
    for name, cost in (("assign_20k_5B_stand", cost_b), ("assign_20k_5A_uniform", None)):
        if cost is None:
            cost = torch.from_numpy(g.config5a()).cuda()
        res = {}

        def solve():
            col, obj, _, st = eng.assign(cost, want_stats=True)
            res["st"], res["obj"] = st, int(obj.item())
        ms, _ = timed(solve, reps=2, warm=1)
        st = res["st"]
        sec = statistics.median(ms) * 1e-3
        swept = 4.0 * n * st.rows_scanned
        out[name] = {"time_to_optimal_s": sec, "objective": res["obj"], "phases": st.phases, "levels": st.search_steps,
                     "rows_scanned": st.rows_scanned, "sweeps": st.rows_scanned / n,
                     "roofline": {"bound": "hbm", "achieved": swept / sec / 1e9, "peak": hbm_peak, "unit": "GB/s",
                                  "frac": swept / sec / 1e9 / hbm_peak, "bytes_model": "4n bytes per cost row relaxed"}}
        # e2e: host matrix in pinned memory -> device -> solve -> assignment back on the host
        if name == "assign_20k_5B_stand":
            host = cost.cpu().pin_memory()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            dcost = host.to("cuda", non_blocking=True)
            col, obj, _, _ = eng.assign(dcost)
            col_h = col.cpu()
            obj_h = int(obj.item())
            out[name]["e2e_s"] = time.perf_counter() - t0
            out[name]["e2e_h2d_bytes"] = host.numel() * 4
            assert obj_h == res["obj"]
            del host, dcost
        if name == "assign_20k_5A_uniform":
            del cost
    # K2 on the reference's own sizes: config 1 (python.py: 200 x 200, uniform and stand-derived with 10 dummy rows) and
    # config 2 (2000 x 2000); CPU beside it: scipy linprog (HiGHS) on the reference's 2n x n^2 model (python.py's path;
    # n = 200 only -- the dense model of solver.py:15-19 needs 128 GB at n = 2000) and scipy's LSA, one host core
    from oracle import assign_ref, cost_ref
    d1, cab1, cust1 = g.config1b()
    _, c1b = cost_ref.calculate_cost_np(d1, cab1, cust1)
    for name, Mnp, lp in (("assign_200_1A_uniform", g.config1a(), True), ("assign_200_1B_stand_padded", c1b, True),
                          ("assign_2000_2_uniform", g.config2(), False), ("assign_2000_2_stand", g.config2_stand(), False)):
        Md = torch.from_numpy(np.ascontiguousarray(Mnp, dtype=np.int32)).cuda()
        res = {}

        def solve_small():
            col, obj, _, _ = eng.assign(Md)
            res["obj"] = obj
        ms, _ = timed(solve_small, reps=10, warm=3)
        t0 = time.perf_counter()
        ref_obj, _ = assign_ref.solve_scipy(Mnp)
        lsa_s = time.perf_counter() - t0
        assert int(res["obj"].item()) == ref_obj, name
        out[name] = {"time_to_optimal_s": statistics.median(ms) * 1e-3, "objective": ref_obj, "n": int(Mnp.shape[0]),
                     "cpu_scipy_lsa_s": lsa_s, "cpu_cores": 1}
        if lp:
            t0 = time.perf_counter()
            lp_obj = assign_ref.lp_relaxation(Mnp)[0]
            out[name]["cpu_scipy_linprog_highs_s"] = time.perf_counter() - t0
            out[name]["lp_relaxation_rel_err"] = abs(lp_obj - ref_obj) / max(abs(ref_obj), 1)
        del Md
    # K3: LCM on 2000 x 2000 (config 2), heuristic.py variant
    c2 = torch.from_numpy(g.config2()).cuda()
    ms, r = timed(lambda: eng.lcm(c2, 100), reps=10, warm=3)
    hv = eng.lcm_host_view(*r)
    golden = json.load(open(os.path.join(ROOT, "tests", "golden", "lcm.json")))["config2_heuristic"]
    assert hv["total"] == golden["total"], "LCM total differs from the golden trace"
    med = statistics.median(ms)
    t0 = time.perf_counter()
    from oracle import lcm_ref
    cpu_tot = lcm_ref.lcm_c(g.config2(), 100)["total"]          # literal array algorithm (C twin of heuristic.py:24-33), one core
    lcm_cpu_s = time.perf_counter() - t0
    assert cpu_tot == hv["total"]
    out["lcm_2000"] = {"ms": med, "lcm_per_s": 1e3 / med, "total": hv["total"], "cpu_literal_c_s": lcm_cpu_s, "cpu_cores": 1,
                       "roofline": {"bound": "hbm", "achieved": 4 * 2000 * 2000 / (med * 1e-3) / 1e9, "peak": hbm_peak,
                                    "unit": "GB/s", "frac": 4 * 2000 * 2000 / (med * 1e-3) / 1e9 / hbm_peak,
                                    "bytes_model": "4 n^2 (each cost read once); L2-resident and sync-latency bound"}}
    return out


if __name__ == "__main__":
    main()
