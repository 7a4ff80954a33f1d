#!/usr/bin/env python3
"""bench.py -- EM fits/sec of the batched LDS-EM hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path
    python bench.py --impl reference ...                     # the reference's CPU algorithm (oracle)
    python bench.py ... --dump-outputs DIR                   # + the last timed step's results as DIR/*.npy

A "step" is one pass of the hot path over one batch: config[1] of BASELINE.json -- cvLDS on
NPannual/NPpc (T=413, p=q=3), 100 make_Z hold-out folds x 100 restarts = 10 000 independent EM
fits, niter=1000, tol=1e-5, followed by the per-fold restart selection and the winners' smoothed
trajectories.  With N>1 (torchrun, one rank per GPU) every rank owns its own such batch
(different folds / initial values): weak scaling, no data-path collective.

Printed JSON (one line, rank 0): see the task contract; extra keys `roofline`, `cpu_baseline`, `run`
(how the line was measured), `strong` (BASELINE config 3 = 480 000 fits SHARED by the N ranks: groups
dealt by ldsr_shard_groups, slowest rank timed, plus `e2e_sharded`: the one-process host-buffer call
ldsr_em_batch(n_devices=N) on rank 0) and `configs` (the other BASELINE configurations, one record each).
  value   fits/s, inputs resident in HBM (ldsr_plan_em), device time by CUDA events per step
  e2e     fits/s through the public host-buffer call (ldsr_em_batch): packing, H2D of all inputs,
          EM, D2H of all results inside the timed region (wall clock, synchronised)
  roofline  em_chunk_kernel: algorithmic FP64 flops (SURVEY.md 8d) / its CUDA-event time, against
          the DFMA rate measured in this run (MEASURED_PEAKS.json has no FP64 entry)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: the benchmark writes nothing into it

from ldsr_b200 import workloads as W  # noqa: E402

METRIC = "EM fits/sec (T~400, restarts x CV folds)"


def build_workload(name, rank):
    seed = W.SEED + 7919 * rank
    if name == "np_cv":
        return W.np_cv(100, 100, seed)
    if name == "np_restarts":
        return W.np_restarts(100, seed)
    if name == "synthetic":
        return W.synthetic_stations(seed=seed)
    if name == "synthetic_small":
        return W.synthetic_stations(n_stations=4, n_folds=25, n_restarts=100, seed=seed)
    raise SystemExit("unknown workload " + name)


def workload_config(w, args):
    s = w["series"][0]
    return {"workload": w["name"], "n_fits_per_gpu": int(w["fit_group"].size), "n_groups_per_gpu": int(len(w["group_series"])),
            "n_series": len(w["series"]), "T": int(s["y"].size), "p": int(s["p"]), "q": int(s["q"]),
            "niter": args.niter, "tol": args.tol, "chunk_iters": args.chunk or 100}


def total_flops(w, iters):
    """Algorithmic FP64 flops of the EM job (SURVEY.md 8d)."""
    gs, fg = w["group_series"], w["fit_group"]
    it_g = np.bincount(fg, weights=iters, minlength=len(gs))
    n_g = np.bincount(fg, minlength=len(gs))
    tot = 0.0
    for g in range(len(gs)):
        s = w["series"][gs[g]]
        T = s["y"].size
        n_obs = int(np.isfinite(s["y"]).sum()) - len(np.unique(w["held"][g]))
        tot += it_g[g] * W.flops_per_iter(T, s["p"], s["q"], n_obs) + n_g[g] * T * (2 * s["q"] + 1)
    return tot


# ---- clocks sampler (B200_PROFILING.md "clocks DURING the timed region") ----------------------
class ClockSampler:
    FIELDS = ("timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_id):
        self.lines = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(gpu_id), "--query-gpu=" + self.FIELDS,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append((time.time(), ln.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        time.sleep(0.12)
        self.proc.terminate()
        rows = [ln for (ts, ln) in self.lines if t0 - 0.05 <= ts <= t1 + 0.1] or [ln for _, ln in self.lines]
        sm, mx, reasons, pw = [], [], set(), []
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for ln in rows:
            f = [x.strip() for x in ln.split(",")]
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
                pw.append(float(f[3]))
            except Exception:
                continue
            for nm, val in zip(names, f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


def cpu_sample_groups(w, seconds, cores):
    """How many groups of `w` give about `seconds` of oracle work on `cores` threads."""
    s = w["series"][w["group_series"][0]]
    per_fit = 1000 * s["y"].size * (30 + 4 * (s["p"] + s["q"])) * 1e-9  # ~50 ns/(iter*step) at p=q=3
    fits_per_group = w["fit_group"].size / len(w["group_series"])
    g = int(seconds * cores / (per_fit * fits_per_group))
    return max(1, min(g, len(w["group_series"])))


def cpu_sample_seconds(args):
    """Oracle work per step/sample: the same in the cpu_baseline leg and in the reference arm, bounded so
    that `--impl reference --steps K --warmup W` ends within a few minutes."""
    return min(args.cpu_seconds, 150.0 / max(1, args.steps + args.warmup))


def host_cores():
    """Host threads the CPU arm may use: the process's CPU affinity, not OMP_NUM_THREADS (torchrun sets
    that to 1 for every rank; the reference arm runs on rank 0 alone and takes the whole box)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except Exception:
        return max(1, os.cpu_count() or 1)


def matches_oracle(ro, res, ns, g):
    """The parity gates of BASELINE.json on a sample: identical iteration counts and selected restarts,
    log-likelihood to 1e-9, theta to 1e-6 (relative)."""
    th_o, th_g = ro["theta"], res["theta"][:ns, :ro["theta"].shape[1]]
    return bool(np.array_equal(ro["iters"], res["iters"][:ns]) and np.array_equal(ro["best"], res["best"][:g])
                and np.allclose(ro["lik"], res["lik"][:ns], rtol=1e-9, atol=0)
                and np.allclose(th_g, th_o, rtol=1e-6, atol=1e-12))


def run_oracle(sample, args, threads):
    from oracle import oracle as O
    t0 = time.perf_counter()
    r = O.em_batch(sample["series"], sample["group_series"], sample["held"], sample["fit_group"], sample["theta0"],
                   args.niter, args.tol, n_threads=threads)
    return time.perf_counter() - t0, r


def oracle_check(w, res, args, seconds):
    """Oracle (CPU port of src/EM.cpp) on the first groups of `w` against the GPU results `res` of the
    whole job: returns (cpu record, match flag)."""
    cores = host_cores()
    g = cpu_sample_groups(w, seconds, cores)
    sample = W.subset(w, g)
    dt, ro = run_oracle(sample, args, cores)
    ns = int(sample["fit_group"].size)
    return {"value": ns / dt, "unit": "fits/s", "cores": cores, "kind": "port",
            "sample": "first %d of %d groups (%d fits), %.1f s" % (g, len(w["group_series"]), ns, dt)}, \
        matches_oracle(ro, res, ns, g)


DUMP_LIMIT = 64 << 20  # bytes of --dump-outputs, all arrays together


def dump_outputs(dirname, res, fit_group):
    """Writes the arrays of a fetched EM result as DIR/<name>.npy in float64.  A result above DUMP_LIMIT is cut
    to a fixed sample of whole groups (their fits, selections and trajectory rows; traj_ptr renumbered), listed
    in sample_groups.npy.  Groups differ in size, so the sample aims at half the limit."""
    ng = res["best"].size
    total = sum(np.asarray(a).size * 8 for a in res.values())
    if total > DUMP_LIMIT:
        keep = np.sort(np.random.default_rng(0).choice(ng, max(1, ng * DUMP_LIMIT // (2 * total)), replace=False))
        ptr = res["traj_ptr"]
        rows = np.concatenate([np.arange(ptr[g], ptr[g + 1]) for g in keep])
        fits = np.isin(fit_group, keep)
        res = dict({k: res[k][fits] for k in ("theta", "lik", "iters", "status")}, best=res["best"][keep],
                   traj_ptr=np.concatenate([[0], np.cumsum(np.diff(ptr)[keep])]), sample_groups=keep,
                   **{k: res[k][rows] for k in ("X", "Y", "V", "J")})
    os.makedirs(dirname, exist_ok=True)
    for k, a in res.items():
        np.save(os.path.join(dirname, k + ".npy"), np.asarray(a, dtype=np.float64))


def device_steps(plan, args, steps, warmup, torch, flush, stream):
    """`warmup` untimed + `steps` timed passes of plan.em on the current stream: CUDA-event ms per step."""
    for _ in range(warmup):
        plan.em(args.niter, args.tol, chunk_iters=args.chunk, stream=stream)
    torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    stats = []
    for k in range(steps):
        flush.zero_()
        ev[k][0].record()
        stats.append(plan.em(args.niter, args.tol, chunk_iters=args.chunk, stream=stream))
        ev[k][1].record()
    torch.cuda.synchronize()
    return [a.elapsed_time(b) for a, b in ev], stats


def strong_block(args, rank, world, local, dev, torch, dist, flush, fp64_peak, cpu_group):
    """BASELINE config 3 (48 stations x 100 folds x 100 restarts = 480 000 fits, T=400, p=q=10) as ONE job
    shared by the ranks: groups dealt by ldsr_shard_groups (the partition ldsr_em_batch itself uses), no
    data-path collective; the step time is the slowest rank's.  Rank 0 then runs the same job through the
    one-process host-buffer call ldsr_em_batch(n_devices=world) (what an R session calls)."""
    from ldsr_b200 import _lib
    w3 = build_workload(args.strong_workload, 0)  # the same job on every rank
    ng, nf = len(w3["group_series"]), int(w3["fit_group"].size)
    shard = _lib.shard_groups(w3["series"], w3["group_series"], w3["held"], w3["fit_group"], w3["theta0"], world)
    mine = W.take_groups(w3, np.nonzero(shard == rank)[0])
    plan = _lib.Plan(mine["series"], mine["group_series"], mine["held"], mine["fit_group"], mine["theta0"], device=local)
    stream = torch.cuda.current_stream().cuda_stream
    if world > 1:
        dist.barrier()
    step_ms, stats = device_steps(plan, args, args.strong_steps, 3, torch, flush, stream)  # 3 warm-up steps
    res = plan.fetch(want_traj=False)
    my = torch.tensor([sum(step_ms) / len(step_ms), float(res["iters"].sum()), total_flops(mine, res["iters"]),
                       float(np.mean([st["em_kernel_ns"] for st in stats])) * 1e-6], dtype=torch.float64, device=dev)
    allv = [torch.zeros_like(my) for _ in range(world)]
    if world > 1:
        dist.all_gather(allv, my)
    else:
        allv = [my]
    allv = np.array([a.cpu().numpy() for a in allv])
    plan.close()
    del plan
    per_rank_ms = allv[:, 0]
    step = float(per_rank_ms.max())
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
    out = None
    if rank == 0:
        flops = float(allv[:, 2].sum())
        out = {"workload": w3["name"], "scaling": "strong", "n_fits": nf, "n_groups": ng, "n_gpus": world,
               "steps": args.strong_steps, "warmup": 3, "l2": "flushed (256 MiB write) between timed steps",
               "value": nf / (step * 1e-3), "unit": "fits/s", "ms_per_step": step,
               "per_rank_ms": [round(float(x), 3) for x in per_rank_ms],
               "per_rank_em_kernel_ms": [round(float(x), 3) for x in allv[:, 3]],
               "imbalance": float(per_rank_ms.max() / per_rank_ms.mean() - 1.0),
               "mean_iters": float(allv[:, 1].sum() / nf), "kernel": stats[0]["kernel"],
               "roofline": {"bound": "fp64", "achieved": flops / (step * 1e-3) / 1e12, "peak": fp64_peak * world,
                            "unit": "TFLOP/s", "frac": flops / (step * 1e-3) / 1e12 / (fp64_peak * world),
                            "note": "algorithmic flops of all ranks / slowest rank's step time / (N x DFMA peak)"},
               "partition": "ldsr_shard_groups (whole groups, greedy LPT), no collective on the data path"}
        # ---- the one-process path: host buffers in and out, one worker thread + stream per device
        ndev = min(world, _lib.device_count())
        ctx = _lib.Ctx(devices=list(range(ndev)))
        call = lambda: _lib.em_batch(w3["series"], w3["group_series"], w3["held"], w3["fit_group"], w3["theta0"],
                                     args.niter, args.tol, chunk_iters=args.chunk, ctx=ctx, n_devices=ndev)
        r = call()
        t0 = time.perf_counter()
        for _ in range(2):
            r = call()
        dt = (time.perf_counter() - t0) / 2
        out["e2e_sharded"] = {"value": nf / dt, "unit": "fits/s", "ms_per_call": dt * 1e3, "n_devices": ndev,
                              "timing": "wall clock around one-process ldsr_em_batch(n_devices=%d), host buffers" % ndev}
        if not args.no_cpu:
            cpu, same = oracle_check(w3, r, args, args.strong_cpu_seconds)
            out["cpu_baseline"] = dict(cpu, gpu_matches_oracle_on_sample=same,
                                       checked="ldsr_em_batch(n_devices=%d) results vs the oracle" % ndev)
        ctx.close()
    if world > 1:
        # the other ranks wait on the HOST (gloo): a pending NCCL barrier is a kernel spinning on their
        # GPU, and without MPS it would time-slice with rank 0's worker on that device (measured: the
        # second device of ldsr_em_batch(n_devices=2) took 1455 ms instead of 697 ms)
        dist.barrier(group=cpu_group)
    return out


def config1_block(args, local, torch, flush):
    """BASELINE config 1: LDS_reconstruction(NPannual, NPpc, NPpc, start.year=1600, num.restarts=100) -- 100
    restarts of one series (1 group), and a single LDS_EM fit.  Device time per call."""
    from ldsr_b200 import _lib
    stream = torch.cuda.current_stream().cuda_stream
    w = build_workload("np_restarts", 0)
    out = {}
    for name, n in (("restarts_100", 100), ("single_fit", 1)):
        sub = dict(w, fit_group=w["fit_group"][:n], theta0=w["theta0"][:n])
        plan = _lib.Plan(sub["series"], sub["group_series"], sub["held"], sub["fit_group"], sub["theta0"], device=local)
        ms, stats = device_steps(plan, args, 5, 3, torch, flush, stream)
        res = plan.fetch(want_traj=False)
        rec = {"n_fits": n, "ms": float(np.median(ms)), "value": n / (float(np.median(ms)) * 1e-3), "unit": "fits/s",
               "mean_iters": float(res["iters"].mean()), "kernel": stats[0]["kernel"]}
        if not args.no_cpu:
            _, ro = run_oracle(sub, args, host_cores())
            rec["gpu_matches_oracle"] = matches_oracle(ro, res, n, 1)
        out[name] = rec
        plan.close()
    out["workload"] = w["name"]
    return out


def config4_block(args, hbm_peak):
    """BASELINE config 4: LDS_rep, 100 000 stochastic replicates of the fitted NP model (theta = data/theta.rda,
    u = v = t(NPpc), T = 813): 81.3 M (x, y, Q) triples.  Device time of the replicate kernels (CUDA events,
    ldsr_last_device_ms) against the HBM roofline -- 24 B written per (replicate, step) -- and the wall clock
    of the host-buffer call (kernels + PCIe + the copy into the caller's arrays, pipelined)."""
    from ldsr_b200 import _lib
    from tests import data
    d = data.load("np.json")
    th = data.theta_of(d["theta"])
    y, u, mu, inst = data.np_case(1, 1200)
    T, n_reps = y.size, args.rep_replicates
    best = None
    for _ in range(3):
        t0 = time.perf_counter()
        r = _lib.rep_batch(th, u, u, T, n_reps, seed=W.SEED, mu=mu)
        wall = time.perf_counter() - t0
        best = (r["device_ms"], wall) if best is None else (min(best[0], r["device_ms"]), min(best[1], wall))
    nbytes = 24.0 * n_reps * T
    gbs = nbytes / (best[0] * 1e-3) / 1e9
    simq = np.asarray(r["simQ"])
    return {"workload": "LDS_rep %d replicates x T=%d (NP model), simX+simY+simQ" % (n_reps, T),
            "value": n_reps * T / (best[0] * 1e-3), "unit": "(replicate,step)/s", "device_ms": best[0],
            "wall_ms": best[1] * 1e3, "bytes_out": nbytes,
            "roofline": {"bound": "hbm", "achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak,
                         "note": "algorithmic bytes (24 B per replicate and step) / device time of the replicate "
                                 "kernels; the noise is generated in the kernel (two FP64 normals per step), "
                                 "which is what bounds it"},
            "finite": bool(np.isfinite(simq).all()), "median_simQ": float(np.median(simq))}


def config5_block(args):
    """BASELINE config 5: state dimension 4, 20 proxies, T = 100 000, 10 % missing: associative-scan smoother
    against the sequential recursion on the device (beyond the reference, which is scalar-state only)."""
    from ldsr_b200 import _lib
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    rng = np.random.default_rng(W.SEED)
    d, p, q, T = 4, 20, 20, args.scan_T
    M = rng.standard_normal((d, d))
    A = 0.9 * M / np.max(np.abs(np.linalg.eigvals(M)))
    L = 0.4 * rng.standard_normal((d, d))
    th = np.concatenate([A.ravel(), (0.3 * rng.standard_normal((d, p)) / np.sqrt(p)).ravel(), rng.standard_normal(d),
                         0.3 * rng.standard_normal(q) / np.sqrt(q), (L @ L.T + 0.1 * np.eye(d)).ravel(), [0.3],
                         np.zeros(d), np.eye(d).ravel()])
    u, v = rng.standard_normal((p, T)), rng.standard_normal((q, T))
    y = rng.standard_normal(T)
    y[rng.uniform(size=T) < 0.1] = np.nan
    _lib.smoother_d(d, y, u, v, th, method=1, want=())  # warm-up
    seq = _lib.smoother_d(d, y, u, v, th, method=0, want=("X", "V"))
    best = None
    for _ in range(3):
        sc = _lib.smoother_d(d, y, u, v, th, method=1, want=("X", "V"))
        best = sc["kernel_ms"] if best is None else min(best, sc["kernel_ms"])
    return {"workload": "d=%d state, %d proxies, T=%d, 10%% missing, 1 parameter set" % (d, p, T),
            "scan_ms": best, "sequential_ms": seq["kernel_ms"], "speedup": seq["kernel_ms"] / best,
            "value": T / (best * 1e-3), "unit": "steps/s",
            "max_abs_dX": float(np.max(np.abs(sc["X"] - seq["X"]))), "max_abs_dV": float(np.max(np.abs(sc["V"] - seq["V"]))),
            "rel_dlik": float(np.max(np.abs(sc["lik"] - seq["lik"]) / np.abs(seq["lik"]))),
            "parity": "scan vs sequential recursion on the device; both vs the general-d oracle in tests/test_gpu_scan.py"}


def reference_arm(args, rank, world):
    """The reference's CPU algorithm (oracle/ldsr_oracle.c, restating src/EM.cpp) on all host threads.
    The real Rcpp/Armadillo build cannot run here (no R): see DESIGN.md."""
    if rank != 0:
        return
    cores = host_cores()
    w = build_workload(args.workload, 0)
    K, Wm = args.steps, args.warmup
    g = cpu_sample_groups(w, cpu_sample_seconds(args), cores)
    sample = W.subset(w, g)
    nf = int(sample["fit_group"].size)
    for _ in range(Wm):
        run_oracle(sample, args, cores)
    times = []
    esteps = 0
    for _ in range(K):
        dt, r = run_oracle(sample, args, cores)
        times.append(dt)
        esteps = int(r["iters"].sum())
    tot = sum(times)
    value = nf * K / tot
    desc = "first %d of %d groups (%d fits) per step" % (g, len(w["group_series"]), nf)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "fits/s", "n_gpus": args.gpus, "steps": K,
        "warmup": Wm, "ms_per_step": 1e3 * tot / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "bundled NP series + synthetic initial values/folds (seeded)",
        "config": workload_config(w, args),
        "cpu_baseline": {"value": value, "unit": "fits/s", "cores": cores, "kind": "port", "sample": desc},
        "e2e": {"value": value, "unit": "fits/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "iter_steps_per_s": esteps * w["series"][0]["y"].size / (tot / K),
    }))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="np_cv")
    ap.add_argument("--niter", type=int, default=1000)
    ap.add_argument("--tol", type=float, default=1e-5)
    ap.add_argument("--chunk", type=int, default=0)
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="oracle work per cpu_baseline sample")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--strong-workload", default="synthetic", help="job shared by the ranks in the `strong` block")
    ap.add_argument("--strong-steps", type=int, default=3)
    ap.add_argument("--strong-cpu-seconds", type=float, default=3.0)
    ap.add_argument("--no-strong", action="store_true", help="skip the `strong` block (config 3)")
    ap.add_argument("--no-configs", action="store_true", help="skip the `configs` block (configs 1, 4, 5)")
    ap.add_argument("--rep-replicates", type=int, default=100000, help="config 4: LDS_rep replicates")
    ap.add_argument("--scan-T", type=int, default=100000, help="config 5: series length")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the results of the last timed step (rank 0) as DIR/<name>.npy, float64, <= 64 MB")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from ldsr_b200 import _lib

    if not torch.cuda.is_available() or _lib.device_count() < 1:
        raise SystemExit("bench.py: no CUDA device; this path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    cpu_group = None
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
        cpu_group = dist.new_group(backend="gloo")  # host-side waits that must not occupy a GPU

    w = build_workload(args.workload, rank)
    nf = int(w["fit_group"].size)
    K, Wm = args.steps, args.warmup
    fp64_peak = _lib.measure_fp64_peak(local)

    # ---------------- device-resident path (value) ----------------
    plan = _lib.Plan(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], device=local)
    stream = torch.cuda.current_stream().cuda_stream
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    for _ in range(Wm):
        plan.em(args.niter, args.tol, chunk_iters=args.chunk, stream=stream)
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    uuid = str(torch.cuda.get_device_properties(local).uuid)
    sampler = ClockSampler(uuid if uuid.startswith("GPU-") else "GPU-" + uuid) if rank == 0 else None
    time.sleep(0.6 if rank == 0 else 0.0)  # let nvidia-smi start sampling
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t_wall0 = time.time()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    stats = []
    for k in range(K):
        flush.zero_()  # L2 flush between timed iterations (not inside the event pair)
        ev[k][0].record()
        stats.append(plan.em(args.niter, args.tol, chunk_iters=args.chunk, stream=stream))
        ev[k][1].record()
    torch.cuda.synchronize()
    t_wall1 = time.time()
    if world > 1:
        dist.barrier()
    step_ms = [a.elapsed_time(b) for a, b in ev]
    tot_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tot_ms, op=dist.ReduceOp.MAX)
    tot_ms = float(tot_ms.item())
    clocks = sampler.stop(t_wall0, t_wall1) if sampler else None
    res = plan.fetch(want_traj=bool(args.dump_outputs))
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, res, w["fit_group"])
    iters = res["iters"].astype(np.float64)
    value = world * nf * K / (tot_ms * 1e-3)

    # ---------------- end-to-end through the public host-buffer API ----------------
    ctx = _lib.Ctx(devices=[local])
    call = lambda: _lib.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], args.niter,
                                 args.tol, chunk_iters=args.chunk, ctx=ctx)
    for _ in range(2):
        r_e2e = call()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(K):
        r_e2e = call()
    torch.cuda.synchronize()
    e2e_s = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_s, op=dist.ReduceOp.MAX)
    e2e_value = world * nf * K / float(e2e_s.item())
    h2d = sum(s["y"].nbytes + (0 if s["u"] is None else s["u"].nbytes) + (0 if s["v"] is None else s["v"].nbytes)
              for s in w["series"]) + w["theta0"].nbytes + w["fit_group"].nbytes + w["group_series"].nbytes + \
        sum(h.nbytes for h in w["held"])
    d2h = sum(r_e2e[k].nbytes for k in ("theta", "lik", "iters", "status", "best", "X", "Y", "V", "J"))
    assert np.array_equal(r_e2e["iters"], res["iters"]) and np.array_equal(r_e2e["best"], res["best"])

    # ---------------- BASELINE config 3 shared by the ranks (strong scaling) ----------------
    del plan
    ctx.close()
    strong = None
    if not args.no_strong and args.workload == "np_cv":
        strong = strong_block(args, rank, world, local, dev, torch, dist, flush, fp64_peak, cpu_group)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- roofline of the dominant kernel (the EM kernel) ----------------
    flops = total_flops(w, iters)  # per step
    em_ns = float(np.mean([s["em_kernel_ns"] for s in stats]))
    chunks = float(np.mean([s["chunks"] for s in stats]))
    achieved = flops / (em_ns * 1e-9) / 1e12
    # DRAM bytes per launch and FP64-pipe activity of the EM kernel: counters of the committed
    # `ncu --set full` capture of this command (a profiler run is never timed; profiles/README.md)
    traffic, pipe_pct, ncu_src = None, None, None
    try:
        with open(os.path.join(ROOT, "profiles", "em_split_traffic.json")) as f:
            tj = json.load(f)
        if tj.get("kernel") == stats[0].get("kernel") and args.workload == "np_cv":
            traffic = int(tj["dram_bytes_read"]) + int(tj["dram_bytes_write"])
            pipe_pct, ncu_src = tj.get("sm__pipe_fp64_cycles_active_pct"), tj.get("source")
    except Exception:
        traffic = None
    roofline = {"bound": "fp64", "kernel": stats[0].get("kernel", "em_chunk_kernel"), "achieved": achieved, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": achieved / fp64_peak, "traffic": traffic,
                "ncu": {"sm__pipe_fp64_cycles_active_pct": pipe_pct, "source": ncu_src},
                "peak_source": "DFMA microbenchmark in this run (ldsr_measure_fp64_peak); MEASURED_PEAKS.json has no FP64 entry",
                "flops_per_launch": flops / chunks, "launch_ms": em_ns * 1e-6 / chunks, "launches_per_step": chunks,
                "kernel_share_of_step": em_ns * 1e-6 / (tot_ms / K)}
    # the same launch against the HBM roofline, to show which bound is the live one: the DRAM traffic of
    # the committed ncu capture over the launch time, against the driver's measured copy bandwidth
    if traffic is not None:
        hbm_peak, hbm_src = 6650.0, "of fallback (B200_PROFILING.md)"
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                hbm_peak, hbm_src = float(json.load(f)["hbm_gbs"]), "of measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
        hbm_ach = traffic / (em_ns * 1e-9 / chunks) / 1e9
        roofline["hbm"] = {"achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_ach / hbm_peak,
                           "peak_source": hbm_src, "note": "not the bound: the working set stays in shared memory"}

    # ---------------- CPU baseline (oracle port of src/EM.cpp), bounded sample ----------------
    cpu = None
    if not args.no_cpu and world == 1:
        cpu, same = oracle_check(w, res, args, cpu_sample_seconds(args))
        cpu["gpu_matches_oracle_on_sample"] = same
        cpu["checked"] = "iters and best identical, lik rel 1e-9, theta rel 1e-6"

    configs = None
    if not args.no_configs and args.workload == "np_cv" and world == 1:
        hbm_peak = 6650.0  # fallback of B200_PROFILING.md
        try:
            with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
                hbm_peak = float(json.load(f)["hbm_gbs"])
        except Exception:
            pass
        configs = {"config1": config1_block(args, local, torch, flush), "config4": config4_block(args, hbm_peak),
                   "config5": config5_block(args)}
        if strong is not None:
            configs["config3"] = {k: strong[k] for k in ("workload", "value", "unit", "ms_per_step", "mean_iters")}
            configs["config3"]["frac"] = strong["roofline"]["frac"]
            configs["config3"]["gpu_matches_oracle_on_sample"] = (strong.get("cpu_baseline") or {}).get(
                "gpu_matches_oracle_on_sample")

    out = {
        "metric": METRIC, "value": value, "unit": "fits/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": tot_ms / K, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "bundled NP series (tests/golden/np.json) + synthetic initial values/folds (seeded)",
        "config": workload_config(w, args),
        "run": {"l2": "flushed (256 MiB write) between timed steps", "mean_iters": float(iters.mean()),
                "parallelism": "one batch per rank (weak), %d GPU(s), no collective; the shared job is in `strong`" % world},
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "fits/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                "timing": "wall clock around ldsr_em_batch (host packing + pageable H2D + EM + D2H)"},
        "gpu_launches": int(sum(s["launches"] for s in stats)),
        "roofline": roofline, "cpu_baseline": cpu,
        "iter_steps_per_s": world * float(iters.sum()) * w["series"][0]["y"].size / (tot_ms / K * 1e-3),
        "step_ms": [round(x, 3) for x in step_ms],
        "strong": strong, "configs": configs,
    }
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
