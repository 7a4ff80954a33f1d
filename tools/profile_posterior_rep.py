#!/usr/bin/env python3
"""Replicates conditioned on the observed record (ldsr_posterior_rep_batch) against LDS_rep's open-loop
replicates (ldsr_rep_batch) on the same output shape, alternated in one process:
  * BASELINE.json config 4's shape: 100 000 replicates of the NPlds model (u = v = t(NPpc), T = 813), simX + simY +
    simQ (1.95 GB to the host);
  * an 8-member ensemble (perturbed copies of the NPlds theta) x 12 500 replicates: the same 100 000 rows.
Device time: CUDA events around the kernels (for the posterior: the coefficient pass and the sampler), median of
the runs; wall time: the whole call into host (numpy) arrays.  Output rate: bytes written / device time.
    python tools/profile_posterior_rep.py [runs]"""
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from ldsr_b200 import _lib  # noqa: E402
from tests import data  # noqa: E402

runs = int(sys.argv[1]) if len(sys.argv) > 1 else 7
try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()[0]
except (OSError, IndexError):
    gpu = "unknown GPU"
print("GPU: %s" % gpu)
g = data.load("nplds.json")
th = data.theta_of(g["theta"])
y, u, mu, inst = data.np_case(1, 1200)
T = y.size
ser = [dict(y=y, u=u, v=u)]
rng = np.random.default_rng(1)
ens = np.vstack([th] + [th * (1 + 0.01 * rng.standard_normal(th.size)) for _ in range(7)])
ctx = _lib.Ctx(n_devices=1)
shapes = (("config 4: 1 model x 100 000 replicates", th[None, :], 100_000),
          ("8-member ensemble x 12 500 replicates", ens, 12_500))
for name, thetas, n_reps in shapes:
    nf = thetas.shape[0]
    post_ms, rep_ms, post_wall, rep_wall = [], [], [], []
    for k in range(runs + 1):  # the first pass of each warms up
        t0 = time.perf_counter()
        r = _lib.posterior_rep_batch(ser, [0], None, np.zeros(nf, dtype=np.int32), thetas, n_reps, seed=k,
                                     mu=np.full(nf, mu), transform="log", ctx=ctx)
        t1 = time.perf_counter()
        q = _lib.rep_batch(th, u, u, T, nf * n_reps, seed=k, mu=mu, ctx=ctx.h)
        t2 = time.perf_counter()
        if k:
            post_ms.append(r["device_ms"])
            rep_ms.append(q["device_ms"])
            post_wall.append(t1 - t0)
            rep_wall.append(t2 - t1)
    nbytes = 3 * 8 * nf * n_reps * T
    pm, rm = np.median(post_ms), np.median(rep_ms)
    print("%s (T = %d, simX + simY + simQ = %.2f GB), median of %d alternated runs:" % (name, T, nbytes / 1e9, runs))
    print("  posterior: device %.2f ms (%.0f GB/s of output; runs %.2f..%.2f), wall %.1f ms"
          % (pm, nbytes / (pm * 1e-3) / 1e9, min(post_ms), max(post_ms), np.median(post_wall) * 1e3))
    print("  LDS_rep:   device %.2f ms (%.0f GB/s of output; runs %.2f..%.2f), wall %.1f ms"
          % (rm, nbytes / (rm * 1e-3) / 1e9, min(rep_ms), max(rep_ms), np.median(rep_wall) * 1e3))
    print("  ratio posterior / LDS_rep: device %.3f, wall %.3f" % (pm / rm, np.median(post_wall) / np.median(rep_wall)))
ctx.close()
