#!/usr/bin/env python
"""Per-kernel device time of the flagship step (find_pool_all on config 3: 722 customers, K = 4, 8 logical shards) from
torch.profiler with CUDA activities, averaged over the profiled steps.  Run on the GPU box, in a process of its own (the
profiler slows the host; bench.py gives the end-to-end time):  python profiles/kernel_times.py [steps]"""
import collections
import os
import sys

import torch
from torch.profiler import ProfilerActivity, profile

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import taxidispatcher_b200 as td  # noqa: E402
from oracle import gen_inputs as g  # noqa: E402

steps = int(sys.argv[1]) if len(sys.argv) > 1 else 20
dem, dist = g.pool_demand(), g.stand_distances(50)
for _ in range(5):
    td.find_pool_all(dem, dist, 4, 8)
torch.cuda.synchronize()
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    for _ in range(steps):
        td.find_pool_all(dem, dist, 4, 8)
    torch.cuda.synchronize()
tot = collections.defaultdict(lambda: [0, 0.0])
for ev in prof.events():
    if ev.device_type == torch.autograd.DeviceType.CUDA:
        t = tot[ev.name.split("(")[0][:60]]
        t[0] += 1
        t[1] += ev.device_time_total if hasattr(ev, "device_time_total") else ev.cuda_time_total
for name, (cnt, us) in sorted(tot.items(), key=lambda kv: -kv[1][1]):
    print("%-62s launches/step %5.2f  us/step %8.1f" % (name, cnt / steps, us / steps))
