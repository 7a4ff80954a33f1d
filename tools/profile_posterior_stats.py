#!/usr/bin/env python3
"""Drought statistics of conditioned replicates reduced on the device (ldsr_posterior_stats_batch) against the
trajectory call (ldsr_posterior_rep_batch, simQ only) and the trajectory call followed by the same statistics in
numpy (tests/posterior_stats_oracle.py), alternated in one process.  NPlds theta (u = v = t(NPpc), T = 813 from
1200), windows of 5, 10, 20 and 30 years, the pre-instrumental years 1200-1959, threshold mean(Qa):
  * 100 000 replicates of one model;
  * 1 000 000 replicates (the statistics call only: simQ alone would take 6.5 GB of host memory);
  * an 8-member ensemble (perturbed copies of the NPlds theta) x 12 500 replicates.
Device time: ldsr_last_device_ms (CUDA events around the coefficient pass and the sampler), median of the runs;
wall time: the whole call into host (numpy) arrays, median.
    python tools/profile_posterior_stats.py [runs]"""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ldsr_b200 import _lib  # noqa: E402
from tests import data  # noqa: E402
from tests import posterior_stats_oracle as PS  # noqa: E402

runs = int(sys.argv[1]) if len(sys.argv) > 1 else 5
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()[0]
print("GPU: %s" % gpu)
g = data.load("nplds.json")
th = data.theta_of(g["theta"])
y, u, mu, inst = data.np_case(1, 1200)
qa = np.array(data.load("np.json")["NPannual"]["Qa"])
T = y.size
ser = [dict(y=y, u=u, v=u)]
windows, lo, hi, thr = (5, 10, 20, 30), 0, 1960 - 1200, float(qa.mean())
rng = np.random.default_rng(1)
ens = np.vstack([th] + [th * (1 + 0.01 * rng.standard_normal(th.size)) for _ in range(7)])
ctx = _lib.Ctx(n_devices=1)


def stats_call(thetas, n_reps, seed):
    nf = thetas.shape[0]
    return _lib.posterior_stats_batch(ser, [0], None, np.zeros(nf, dtype=np.int32), thetas, n_reps, seed=seed,
                                      mu=np.full(nf, mu), transform="log", windows=windows, threshold=np.full(nf, thr),
                                      ranges=np.tile([lo, hi], (nf, 1)), ctx=ctx)


def traj_call(thetas, n_reps, seed):
    nf = thetas.shape[0]
    return _lib.posterior_rep_batch(ser, [0], None, np.zeros(nf, dtype=np.int32), thetas, n_reps, seed=seed,
                                    mu=np.full(nf, mu), transform="log", want=("simQ",), ctx=ctx)


shapes = (("1 model x 100 000 replicates", th[None, :], 100_000, True),
          ("1 model x 1 000 000 replicates", th[None, :], 1_000_000, False),
          ("8-member ensemble x 12 500 replicates", ens, 12_500, True))
for name, thetas, n_reps, with_traj in shapes:
    nf = thetas.shape[0]
    t = {k: [] for k in ("stats_dev", "stats_wall", "traj_dev", "traj_wall", "numpy_wall")}
    for k in range(runs + 1):  # the first pass of each warms up
        t0 = time.perf_counter()
        s = stats_call(thetas, n_reps, k)
        t1 = time.perf_counter()
        if k:
            t["stats_dev"].append(s["device_ms"])
            t["stats_wall"].append((t1 - t0) * 1e3)
        if not with_traj:
            continue
        t0 = time.perf_counter()
        r = traj_call(thetas, n_reps, k)
        t1 = time.perf_counter()
        for f in range(nf):
            PS.stats(r["simQ"][f], windows, thr, lo, hi)
        t2 = time.perf_counter()
        if k:
            t["traj_dev"].append(r["device_ms"])
            t["traj_wall"].append((t1 - t0) * 1e3)
            t["numpy_wall"].append((t2 - t0) * 1e3)
        del r
    md = {k: (np.median(v) if v else float("nan")) for k, v in t.items()}
    rows = nf * n_reps
    print("%s (T = %d; statistics out %.1f MB, simQ %.2f GB), median of %d alternated runs:"
          % (name, T, rows * (24 * len(windows) + 24) / 1e6, rows * T * 8 / 1e9, runs))
    print("  statistics call:           device %8.2f ms (runs %.2f..%.2f), wall %8.1f ms"
          % (md["stats_dev"], min(t["stats_dev"]), max(t["stats_dev"]), md["stats_wall"]))
    if with_traj:
        print("  trajectory call (simQ):    device %8.2f ms (runs %.2f..%.2f), wall %8.1f ms"
              % (md["traj_dev"], min(t["traj_dev"]), max(t["traj_dev"]), md["traj_wall"]))
        print("  trajectory call + numpy:   wall %8.1f ms" % md["numpy_wall"])
        print("  ratio statistics / trajectory: device %.3f, wall %.3f; statistics / (trajectory + numpy) wall %.4f"
              % (md["stats_dev"] / md["traj_dev"], md["stats_wall"] / md["traj_wall"],
                 md["stats_wall"] / md["numpy_wall"]))
ctx.close()
