#!/usr/bin/env python3
"""Per-year quantiles of w-year means selected on the device (ldsr_posterior_quantile_batch) against the year-by-year
counts of the same replicates (ldsr_posterior_yearly_batch, the same seed and years), alternated in one process.
NPlds theta (u = v = t(NPpc), T = 813 from 1200), the pre-instrumental years 1200-1959; quantiles: windows of 1, 10
and 20 years, levels 0.05, 0.5, 0.95; yearly: windows of 10 and 20 years, run lengths of 5 and 10 years, threshold
mean(Qa).  10^5 and 10^6 replicates of one model.
Device time: ldsr_last_device_ms (CUDA events around the coefficient pass, every sampler pass and the selection
kernels); wall time: the whole call into host (numpy) arrays; medians over the timed runs, after one warm-up run of
each call.  Then, in runs of their own: the kernel times of one quantile call (torch.profiler, CUDA activities: the
range pass, the first histogram pass and the rest), the rise of the device's used memory during one call in a
fresh context (free memory polled from another thread, so a lower bound of the peak), and at 10^5 replicates the host
route it replaces (the trajectory call, then window means and np.quantile(method="inverted_cdf") in numpy).  The
GPU's name and power limit are read in the same run.
    python tools/profile_posterior_quantiles.py [runs] [output file, default profiles/posterior_quantiles.txt]"""
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ldsr_b200 import _lib  # noqa: E402
from tests import data  # noqa: E402

runs = int(sys.argv[1]) if len(sys.argv) > 1 else 7
path = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "profiles", "posterior_quantiles.txt")
lines = ["# python tools/profile_posterior_quantiles.py %d" % runs]
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()[0]
lines.append("GPU: %s" % gpu)
g = data.load("nplds.json")
th = data.theta_of(g["theta"])[None, :]
y, u, mu, inst = data.np_case(1, 1200)
qa = np.array(data.load("np.json")["NPannual"]["Qa"])
ser = [dict(y=y, u=u, v=u)]
windows, levels, lo, hi = (1, 10, 20), (0.05, 0.5, 0.95), 0, 1960 - 1200
ctx = _lib.Ctx(n_devices=1)
common = dict(seed=0, mu=[mu], transform="log", ranges=[(lo, hi)], ctx=ctx)
calls = {"quantile": lambda n: _lib.posterior_quantile_batch(ser, [0], None, [0], th, n, windows=windows,
                                                             levels=levels, **common),
         "yearly": lambda n: _lib.posterior_yearly_batch(ser, [0], None, [0], th, n, windows=(10, 20), lengths=(5, 10),
                                                         threshold=[float(qa.mean())], **common)}
for n_reps in (100_000, 1_000_000):
    t = {k: {"dev": [], "wall": []} for k in calls}
    passes = None
    for k in range(runs + 1):  # the first pass of each warms up
        for name, call in calls.items():
            t0 = time.perf_counter()
            r = call(n_reps)
            t1 = time.perf_counter()
            if name == "quantile":
                passes = r["passes"]
            if k:
                t[name]["dev"].append(r["device_ms"])
                t[name]["wall"].append((t1 - t0) * 1e3)
    lines.append("1 model x %d replicates (T = %d, years 1200-1959), median of %d alternated runs:" % (n_reps, y.size,
                                                                                                     runs))
    for name in calls:
        d, w = t[name]["dev"], t[name]["wall"]
        lines.append("  %-9s call: device %8.2f ms (runs %.2f..%.2f), wall %8.1f ms"
                     % (name, np.median(d), min(d), max(d), np.median(w)))
    lines.append("  sampler passes of the quantile call: %d" % passes)
    lines.append("  ratio quantile / yearly: device %.3f, wall %.3f"
                 % (np.median(t["quantile"]["dev"]) / np.median(t["yearly"]["dev"]),
                    np.median(t["quantile"]["wall"]) / np.median(t["yearly"]["wall"])))
    # kernel times of one call, in a run of its own
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.init()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        calls["quantile"](n_reps)
        torch.cuda.synchronize()
    ev = sorted((e for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA),
                key=lambda e: e.time_range.start)
    samp = [e.device_time / 1e3 for e in ev if "posterior_rep_kernel" in e.name]
    other = sum(e.device_time / 1e3 for e in ev if "quant_" in e.name)
    lines.append("  kernels of one call (torch.profiler): sampler passes %s ms; selection kernels %.2f ms in all"
                 % (", ".join("%.2f" % s for s in samp), other))
    if len(samp) > 1:
        lines.append("  range pass %.2f ms, first histogram pass %.2f ms" % (samp[0], samp[1]))
    # device memory: free memory polled while one call runs
    free0 = torch.cuda.mem_get_info()[0]
    low = [free0]
    stop = threading.Event()

    def poll():
        while not stop.is_set():
            low[0] = min(low[0], torch.cuda.mem_get_info()[0])

    fresh = _lib.Ctx(n_devices=1)  # the timed context's pool already holds blocks from the runs above
    th_poll = threading.Thread(target=poll)
    th_poll.start()
    _lib.posterior_quantile_batch(ser, [0], None, [0], th, n_reps, windows=windows, levels=levels,
                                  **dict(common, ctx=fresh))
    stop.set()
    th_poll.join()
    fresh.close()
    lines.append("  device memory in use during one call (polled, a lower bound of the peak): +%.1f MB"
                 % ((free0 - low[0]) / 2**20))
# the host route at 10^5 replicates: every trajectory to the host, then numpy
n_reps = 100_000
t0 = time.perf_counter()
Q = _lib.posterior_rep_batch(ser, [0], None, [0], th, n_reps, want=("simQ",), seed=0, mu=[mu], transform="log",
                             ctx=ctx)["simQ"][0][:, lo:hi]
t1 = time.perf_counter()
for w in windows:
    c = np.concatenate([np.zeros((n_reps, 1)), np.cumsum(Q, axis=1)], axis=1)
    M = (c[:, w:] - c[:, :-w]) / w
    np.quantile(M, levels, axis=0, method="inverted_cdf")
t2 = time.perf_counter()
lines.append("host route, %d replicates: trajectory call %.0f ms wall, window means and np.quantile %.0f ms, "
             "%.0f ms in all" % (n_reps, (t1 - t0) * 1e3, (t2 - t1) * 1e3, (t2 - t0) * 1e3))
ctx.close()
print("\n".join(lines))
os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
with open(path, "w") as fh:
    fh.write("\n".join(lines) + "\n")
