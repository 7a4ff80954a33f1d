"""One batched call over many stations against the loop of single-station calls.

Workload: 48 synthetic stations of positive annual flows (the construction of workloads.synthetic_stations:
u = v ~ N(0, diag(4/i)), p = q = 10, T = 400, an instrumental period of the last 60..85 years, flows
simulated from a random stable LDS), each with its own start year, plus one station with a two-member
ensemble -- cross-validated at the reference vignette's setting (make_Z's 30 folds x 20 restarts) and
reconstructed with 50 restarts.  Each timing is wall clock from the call to its host result (the
functions return numpy arrays, so the device work has finished).  Both forms are warmed up, then timed
alternately `--reps` times on the same seeded draws; the largest differences between their results and
the GPU name and power limit of the run are printed with the times.

    python tools/profile_stations.py [--stations 48] [--reps 3] [--json FILE]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import ldsr_b200 as L  # noqa: E402
from ldsr_b200 import _lib, api, workloads  # noqa: E402


def make_stations(n_stations=48, T=400, p=10, seed=workloads.SEED):
    out = []
    for st in range(n_stations):
        rng = np.random.default_rng(seed + 1 + st)
        u = rng.standard_normal((p, T)) * np.sqrt(4.0 / np.arange(1, p + 1))[:, None]
        A, Cc = rng.uniform(0.3, 0.9), rng.uniform(0.01, 0.1)
        B = rng.uniform(-1, 1, p) / np.sqrt(p) * 0.1
        D = rng.uniform(-1, 1, p) / np.sqrt(p) * 0.1
        x, y = 0.0, np.empty(T)
        for t in range(T):
            y[t] = Cc * x + D @ u[:, t] + rng.standard_normal() * 0.1
            x = A * x + B @ u[:, t] + rng.standard_normal()
        n_inst = int(rng.integers(60, 86))
        start = 1500 + int(rng.integers(0, 100))
        years = np.arange(start + T - n_inst, start + T)
        flows = np.exp(np.log(rng.uniform(50, 500)) + y[T - n_inst:])  # positive flows, log-normal about a level
        out.append(dict(Qa=dict(year=years, Qa=flows), u=u, v=u, start_year=start))
    e = out[-1]
    out.append(dict(e, u=[e["u"], e["u"][:5]], v=[e["v"], e["v"][:5]]))  # the same gauge with a two-model ensemble
    return out


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:  # the timings stand without it; say so
        return "unknown (%s)" % e


def timed(fn):
    t = time.perf_counter()
    out = fn()
    return time.perf_counter() - t, out


def rel_diff(a, b, floor=1e-8):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    ok = ~(np.isnan(a) & np.isnan(b))
    return float(np.max(np.abs(a[ok] - b[ok]) / np.maximum(np.abs(b[ok]), floor))) if ok.any() else 0.0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--stations", type=int, default=48)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--folds", type=int, default=30)
    ap.add_argument("--restarts", type=int, default=20)
    ap.add_argument("--rec-restarts", type=int, default=50)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--json", default=None, help="also write the result as JSON to this file")
    a = ap.parse_args()
    if _lib.device_count() < 1:
        sys.exit("no CUDA device: this measurement needs the GPU")
    st = make_stations(a.stations)
    for s in st:  # the folds are part of the input, drawn once: make_Z(Qa, nRuns = folds)
        s["Z"] = L.make_Z(s["Qa"]["Qa"], a.folds, rng=np.random.default_rng(a.seed))
    n_fits = sum(len(s["Z"]) * (len(s["u"]) if isinstance(s["u"], list) else 1) for s in st) * a.restarts

    def cv_batched():
        return L.cvLDS_stations(st, num_restarts=a.restarts, rng=np.random.default_rng(a.seed))

    def cv_loop():
        rng = np.random.default_rng(a.seed)
        return [L.cvLDS(s["Qa"], s["u"], s["v"], s["start_year"], Z=s["Z"], num_restarts=a.restarts, rng=rng)
                for s in st]

    def rec_batched():
        return L.LDS_reconstruction_stations(st, num_restarts=a.rec_restarts, rng=np.random.default_rng(a.seed))

    def rec_loop():
        rng = np.random.default_rng(a.seed)
        return [L.LDS_reconstruction(s["Qa"], s["u"], s["v"], s["start_year"], num_restarts=a.rec_restarts, rng=rng)
                for s in st]

    res = dict(gpu=gpu_info(), stations=len(st), cv_fits=n_fits, folds=a.folds, restarts=a.restarts,
               rec_restarts=a.rec_restarts, reps=a.reps)
    for name, batched, loop in (("cvLDS", cv_batched, cv_loop), ("LDS_reconstruction", rec_batched, rec_loop)):
        batched(), loop()  # warm-up: module load, context, allocator
        tb, tl = [], []
        for _ in range(a.reps):  # alternate the two forms
            t, ob = timed(batched)
            tb.append(t)
            t, ol = timed(loop)
            tl.append(t)
        if name == "cvLDS":
            diff = dict(lik=max(rel_diff(x["lik"], y["lik"]) for x, y in zip(ob, ol)),
                        Ycv=max(rel_diff(x["Ycv"], y["Ycv"]) for x, y in zip(ob, ol)),
                        metrics=max(rel_diff(x["metrics_dist"][k], y["metrics_dist"][k], 1e-6)
                                    for x, y in zip(ob, ol) for k in _lib.METRIC_NAMES),
                        best_equal=all(np.array_equal(x["best"], y["best"]) for x, y in zip(ob, ol)),
                        iters_equal=all(np.array_equal(x["iters"], y["iters"]) for x, y in zip(ob, ol)))
        else:
            mem = lambda o: [m for x in o for m in x.get("ensemble", [x])]
            diff = dict(lik=max(rel_diff(x["lik"], y["lik"]) for x, y in zip(mem(ob), mem(ol))),
                        theta=max(rel_diff(api.theta_to_vec(x["theta"]), api.theta_to_vec(y["theta"]))
                                  for x, y in zip(mem(ob), mem(ol))),
                        rec_Q=max(rel_diff(x["rec"]["Q"], y["rec"]["Q"]) for x, y in zip(mem(ob), mem(ol))))
        res[name] = dict(batched_s=tb, loop_s=tl, batched_median_s=float(np.median(tb)),
                         loop_median_s=float(np.median(tl)), speedup=float(np.median(tl) / np.median(tb)),
                         max_rel_diff=diff)
        print("%-19s one call %.3f s  loop of %d calls %.3f s  (median of %d; x%.2f)  max rel diff %s"
              % (name, np.median(tb), len(st), np.median(tl), a.reps, np.median(tl) / np.median(tb), diff),
              flush=True)
    print("GPU (name, power limit):", res["gpu"])
    if a.json:
        with open(a.json, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
