#!/usr/bin/env python3
"""Year-by-year drought counts reduced across replicates on the device (ldsr_posterior_yearly_batch) against the
per-replicate drought statistics of the same replicates (ldsr_posterior_stats_batch, the same seed, windows,
threshold and years), alternated in one process.  NPlds theta (u = v = t(NPpc), T = 813 from 1200), the
pre-instrumental years 1200-1959, threshold mean(Qa); yearly: windows of 10 and 20 years and run lengths of 5 and 10
years; statistics: windows of 10 and 20 years and the run statistics.  10^5 and 10^6 replicates of one model.
Device time: ldsr_last_device_ms (CUDA events around the coefficient pass and the sampler); wall time: the whole call
into host (numpy) arrays; medians over the timed runs, after one warm-up run of each call.  The GPU's name and power
limit are read in the same run.
    python tools/profile_posterior_yearly.py [runs] [output file, default profiles/posterior_yearly.txt]"""
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from ldsr_b200 import _lib  # noqa: E402
from tests import data  # noqa: E402

runs = int(sys.argv[1]) if len(sys.argv) > 1 else 7
path = sys.argv[2] if len(sys.argv) > 2 else os.path.join(ROOT, "profiles", "posterior_yearly.txt")
lines = ["# python tools/profile_posterior_yearly.py %d" % runs]
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()[0]
lines.append("GPU: %s" % gpu)
g = data.load("nplds.json")
th = data.theta_of(g["theta"])[None, :]
y, u, mu, inst = data.np_case(1, 1200)
qa = np.array(data.load("np.json")["NPannual"]["Qa"])
ser = [dict(y=y, u=u, v=u)]
windows, lengths, lo, hi, thr = (10, 20), (5, 10), 0, 1960 - 1200, float(qa.mean())
ctx = _lib.Ctx(n_devices=1)
common = dict(seed=0, mu=[mu], transform="log", windows=windows, threshold=[thr], ranges=[(lo, hi)], ctx=ctx)
calls = {"yearly": lambda n: _lib.posterior_yearly_batch(ser, [0], None, [0], th, n, lengths=lengths, **common),
         "statistics": lambda n: _lib.posterior_stats_batch(ser, [0], None, [0], th, n, **common)}
for n_reps in (100_000, 1_000_000):
    t = {k: {"dev": [], "wall": []} for k in calls}
    for k in range(runs + 1):  # the first pass of each warms up
        for name, call in calls.items():
            t0 = time.perf_counter()
            r = call(n_reps)
            t1 = time.perf_counter()
            if k:
                t[name]["dev"].append(r["device_ms"])
                t[name]["wall"].append((t1 - t0) * 1e3)
    lines.append("1 model x %d replicates (T = %d, years 1200-1959), median of %d alternated runs:" % (n_reps, y.size,
                                                                                                     runs))
    for name in calls:
        d, w = t[name]["dev"], t[name]["wall"]
        lines.append("  %-11s call: device %8.2f ms (runs %.2f..%.2f), wall %8.1f ms"
                     % (name, np.median(d), min(d), max(d), np.median(w)))
    lines.append("  ratio yearly / statistics: device %.3f, wall %.3f"
                 % (np.median(t["yearly"]["dev"]) / np.median(t["statistics"]["dev"]),
                    np.median(t["yearly"]["wall"]) / np.median(t["statistics"]["wall"])))
ctx.close()
print("\n".join(lines))
os.makedirs(os.path.dirname(os.path.abspath(path)), exist_ok=True)
with open(path, "w") as fh:
    fh.write("\n".join(lines) + "\n")
