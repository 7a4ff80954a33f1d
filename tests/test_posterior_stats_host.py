"""Drought statistics of conditioned replicates (ldsr_posterior_stats_batch), without a GPU:
  * the reference (tests/posterior_stats_oracle.py) on hand-written series with known answers: ties, runs clipped
    by the range, runs touching the first and last step, windows as long as the range and longer, no run, and
    non-finite flows inside and outside the range;
  * the statistics mode of posterior_rep_kernel, run from source by the CPU emulator at widths 3 and 16 with caller
    noise, equals the reference applied to the emulated trajectory mode's simQ for the same noise, and is
    bit-identical under four thread schedules;
  * ldsr_posterior_stats_batch checks its arguments before it looks for a device."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

from ldsr_b200 import _lib
from tests import posterior_stats_oracle as PS
from tests import test_gpu_step_kernels as SK
from tests import test_posterior_rep_host as PH

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_simt")
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ldsr_b200", "csrc")
_hostsim = None


def hostsim_lib():
    """tests/host_simt/sim_posterior_stats.cpp built for the CPU, into the temporary directory under a name keyed by
    its sources (as test_posterior_rep_host.py builds sim_posterior.cpp)."""
    global _hostsim
    if _hostsim is None:
        srcs = [os.path.join(HERE, f) for f in ("sim_posterior_stats.cpp", "sim_posterior.cpp", "sim_em.cpp",
                                                "host_simt.h")]
        srcs += sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh"))
        key = hashlib.sha256(b"".join(open(f, "rb").read() for f in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "ldsr_hostsim_stats_%s_%d.so" % (key, os.getuid()))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-DLDSR_HOST_SIM", "-Wno-unknown-pragmas", "-mfma",
                            "-ffp-contract=off", "-shared", "-fPIC", "-DLDSR_HAVE_WIDE", "-DLDSR_HAVE_SCAN",
                            srcs[0], "-o", tmp], check=True)
            os.replace(tmp, so)
        _hostsim = C.CDLL(so)
    return _hostsim


_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int)


# ---- the reference on hand-written series ---------------------------------------------------------------------
def _one(Q, windows=(), thr=None, lo=0, hi=None):
    Q = np.asarray(Q, dtype=float)
    r = PS.stats(Q[None, :], windows, thr, lo, Q.size if hi is None else hi)
    return {k: (v[:, 0].tolist() if k.startswith("w") else v[0].item()) for k, v in r.items() if k != "sums"}


def test_reference_ties_take_the_smallest_start_and_the_earliest_run():
    r = _one([1, 2, 1, 2, 1], windows=(1, 2), thr=1.5)
    assert r["wmin"] == [1.0, 1.5] and r["wmin_at"] == [0, 0]  # every 2-step window has the mean 1.5
    assert r["wmax"] == [2.0, 1.5] and r["wmax_at"] == [1, 0]
    # runs at 0, 2 and 4 (the first and the last step), each of length 1 and deficit 0.5
    assert (r["run_len"], r["run_at"], r["deficit"], r["deficit_at"], r["n_runs"]) == (1, 0, 0.5, 0, 3)
    # the longest run and the largest deficit are different runs
    r = _one([0.9, 0.9, 0.9, 5, 0, 5], thr=1.0)
    assert (r["run_len"], r["run_at"], r["deficit"], r["deficit_at"], r["n_runs"]) == (3, 0, 1.0, 4, 2)


def test_reference_clips_runs_to_the_range():
    Q = [0, 0, 0, 5, 0, 5, 0, 0, 0]
    whole = _one(Q, thr=1.0)
    assert (whole["run_len"], whole["run_at"], whole["deficit"], whole["deficit_at"], whole["n_runs"]) == (3, 0, 3.0,
                                                                                                          0, 3)
    # [2, 7): the runs 0..2 and 6..8 are cut to one step each; three runs of one step, the earliest wins
    r = _one(Q, thr=1.0, lo=2, hi=7)
    assert (r["run_len"], r["run_at"], r["deficit"], r["deficit_at"], r["n_runs"]) == (1, 2, 1.0, 2, 3)
    # a run cut at lo is still the longest
    r = _one([0, 0, 0, 0, 5, 0, 5], thr=1.0, lo=1, hi=7)
    assert (r["run_len"], r["run_at"], r["n_runs"]) == (3, 1, 2)


def test_reference_windows_as_long_as_the_range_and_longer():
    Q = [9, 9, 1, 2, 3, 4, 5, 9, 9]
    r = _one(Q, windows=(5, 6, 1), lo=2, hi=7)
    assert r["wmin"][0] == r["wmax"][0] == 3.0 and r["wmin_at"][0] == r["wmax_at"][0] == 2  # one candidate
    assert np.isnan(r["wmin"][1]) and np.isnan(r["wmax"][1]) and r["wmin_at"][1] == r["wmax_at"][1] == -1
    assert (r["wmin"][2], r["wmin_at"][2], r["wmax"][2], r["wmax_at"][2]) == (1.0, 2, 5.0, 6)


def test_reference_without_a_run():
    r = _one([3, 4, 5], windows=(2,), thr=1.0)
    assert (r["run_len"], r["run_at"], r["deficit"], r["deficit_at"], r["n_runs"]) == (0, -1, 0.0, -1, 0)


def test_reference_non_finite_flows_inside_and_outside_the_range():
    Q = [1.0, 0.5, np.nan, 0.2, 3.0]
    r = _one(Q, windows=(1, 2), thr=1.0)
    assert all(np.isnan(v) for v in r["wmin"] + r["wmax"]) and np.isnan(r["deficit"])
    assert r["wmin_at"] == r["wmax_at"] == [-1, -1]
    assert (r["run_len"], r["run_at"], r["deficit_at"], r["n_runs"]) == (-1, -1, -1, -1)
    r = _one(Q, windows=(1, 2), thr=1.0, lo=3, hi=5)  # the NaN is outside [3, 5)
    assert r["wmin"] == [0.2, 1.6] and r["wmin_at"] == [3, 3] and r["wmax"] == [3.0, 1.6]
    assert (r["run_len"], r["run_at"], r["deficit"], r["deficit_at"], r["n_runs"]) == (1, 3, 0.8, 3, 1)


# ---- the emulated kernel against the reference on the emulated trajectories --------------------------------------
def sim_stats(s, held, fit_group, theta, n_reps, z, mu, tr, lams, windows, thr, ranges, order=0):
    L = hostsim_lib()
    y = np.ascontiguousarray(s["y"], dtype=np.float64)
    uf = None if s["u"] is None else np.ascontiguousarray(np.asarray(s["u"], dtype=np.float64).T)
    vf = None if s["v"] is None else np.ascontiguousarray(np.asarray(s["v"], dtype=np.float64).T)
    hp = np.zeros(len(held) + 1, dtype=np.int32)
    hp[1:] = np.cumsum([len(h) for h in held])
    hi = np.ascontiguousarray(np.concatenate([np.asarray(h, dtype=np.int32) for h in held] + [np.zeros(1, np.int32)]))
    fg = np.ascontiguousarray(fit_group, dtype=np.int32)
    nf, nw = fg.size, len(windows)
    win = np.ascontiguousarray(windows, dtype=np.int32)
    th_a = None if thr is None else np.ascontiguousarray(thr, dtype=np.float64)
    rg = np.ascontiguousarray(ranges, dtype=np.int32)
    outs = {k: np.full((nw, nf, n_reps), 7, dtype=np.int32 if k.endswith("_at") else np.float64)
            for k in _lib.WINDOW_STATS}
    if thr is not None:
        outs.update({k: np.full((nf, n_reps), 7, dtype=np.float64 if k == "deficit" else np.int32)
                     for k in _lib.RUN_STATS})
    d = lambda a: None if a is None else a.ctypes.data_as(_dp)
    i = lambda a: None if a is None else a.ctypes.data_as(_ip)
    o = lambda k: None if k not in outs else (d if outs[k].dtype == np.float64 else i)(outs[k])
    rc = L.hostsim_posterior_stats(s["y"].size, s["p"], s["q"], d(y), d(uf), d(vf), len(held), i(hp), i(hi), nf,
                                   i(fg), d(np.ascontiguousarray(theta, dtype=np.float64)), n_reps,
                                   d(np.ascontiguousarray(z)), d(np.ascontiguousarray(mu, dtype=np.float64)),
                                   _lib.TRANSFORMS[tr], d(np.ascontiguousarray(lams, dtype=np.float64)), nw, i(win),
                                   d(th_a), i(rg), order, *(o(k) for k in _lib.WINDOW_STATS + _lib.RUN_STATS))
    assert rc == 0, rc
    return outs


def _ranges(rng, T):
    """Whole series, a range inside one 16-step tile, and one across tiles (where T allows)."""
    out = [(0, T)]
    if T >= 3:
        t0 = (T - 1) // 16 * 16
        a = min(t0 + 1, T - 2) if T - t0 >= 3 else max(0, T - 3)
        out.append((a, min(a + 2 + rng.integers(0, 3), T)))
    if T > 20:
        a = int(rng.integers(1, 14))
        out.append((a, T - int(rng.integers(1, 14))))
    return out


# (transform, lambda, mu offset): Box-Cox with mu far below 0 makes (y + mu) lambda + 1 < 0 at some steps (NaN flows)
TRANSFORM_CASES = (("log", 0.0, 0.0), ("none", 0.0, 0.0), ("boxcox", 0.35, 3.0), ("boxcox", 0.0, 0.0),
                   ("boxcox", 0.35, -3.6))
TS = (2, 15, 16, 17, 63, 64, 65, 129, 213)
WINDOW_SETS = ((1, 15, 16, 17), (64,), (16, 1), (17, 64, 15))


@pytest.mark.parametrize("width", [(3, 3, "vu"), (16, 16, "sep")], ids=SK.case_id)
def test_emulated_statistics_equal_the_reference_on_the_emulated_trajectories(width):
    p, q, form = width
    rng = np.random.default_rng(p * 7 + q)
    n_nan = 0
    for ti, T in enumerate(TS):
        tr, lam, dmu = TRANSFORM_CASES[ti % len(TRANSFORM_CASES)]
        s = SK.make_series(rng, p, q, form, T)
        held = [SK.holdout(rng, s["y"], k) for k in ("none", "scattered")]
        fit_group = np.array([0, 1, 1])
        nf = fit_group.size
        theta = np.stack([SK.rand_theta(rng, p, q) for _ in range(nf)])
        mu = rng.uniform(0.5, 1.5, nf) + dmu
        lams = np.full(nf, lam)
        n_reps = (33, 5, 40)[ti % 3]
        z = rng.standard_normal((nf, n_reps, 2 * T))
        traj = PH.sim_posterior(s, held, fit_group, theta, n_reps, z, mu, tr, lams, want=("simQ",))["simQ"]
        for ri, rg in enumerate(_ranges(rng, T)):
            ranges = np.array([rg] * nf)
            windows = WINDOW_SETS[(ti + ri) % len(WINDOW_SETS)]
            Qin = traj[:, :, rg[0]:rg[1]]
            thr = np.array([np.nanmedian(Qin[f]) if np.isfinite(Qin[f]).any() else 1.0 for f in range(nf)])
            thr_arg = None if (ti + ri) % 4 == 3 else thr
            got = sim_stats(s, held, fit_group, theta, n_reps, z, mu, tr, lams, windows, thr_arg, ranges)
            for f in range(nf):
                g = {k: v[:, f] if v.ndim == 3 else v[f] for k, v in got.items()}
                PS.assert_match(g, traj[f], windows, None if thr_arg is None else thr[f], rg[0], rg[1],
                                where=(T, rg, f, tr, windows))
            n_nan += int((~np.isfinite(Qin).all(axis=2)).sum())
            # every thread schedule gives the same bits
            for order in (1, 2, 3):
                again = sim_stats(s, held, fit_group, theta, n_reps, z, mu, tr, lams, windows, thr_arg, ranges,
                                  order=order)
                for k in got:
                    assert np.array_equal(again[k], got[k], equal_nan=True), (T, rg, order, k)
    assert n_nan > 0  # some replicates have non-finite flows in their range (Box-Cox)


# ---- argument errors come before the device ---------------------------------------------------------------------
def _batch():
    y = np.array([0.1, np.nan, -0.2, 0.3])
    return dict(series=[dict(y=y, u=np.ones((1, 4)), v=None, p=1, q=1)], group_series=[0], held=None, fit_group=[0],
                theta=np.array([[0.5, 0.1, 0.8, 0.0, 1.0, 0.5, 0.0, 1.0]]))


def _code(**kw):
    b = _batch()
    args = dict(n_reps=4, windows=(2,), threshold=None, ranges=None)
    args.update(kw)
    n_reps = args.pop("n_reps")
    try:
        _lib.posterior_stats_batch(b["series"], b["group_series"], b["held"], b["fit_group"], args.pop("theta", b["theta"]),
                                   n_reps, **args)
    except _lib.LdsrError as e:
        return e.code
    return _lib.OK


BAD_SPECS = {
    "five_windows": dict(windows=(1, 2, 3, 4, 5)),
    "window_of_zero": dict(windows=(0,)),
    "window_of_65": dict(windows=(10, 65)),
    "no_window_and_no_threshold": dict(windows=()),
    "range_below_zero": dict(ranges=[(-1, 3)]),
    "empty_range": dict(ranges=[(2, 2)]),
    "range_past_the_end": dict(ranges=[(0, 5)]),
    "nan_threshold": dict(threshold=[np.nan]),
    "infinite_threshold": dict(threshold=[np.inf]),
    "run_outputs_without_threshold": dict(want=("wmin", "n_runs")),
    "no_replicates": dict(n_reps=0),
    "unknown_transform": dict(transform=3),
    "box_cox_without_lambda": dict(transform="boxcox"),
    "negative_R": dict(theta=np.array([[0.5, 0.1, 0.8, 0.0, 1.0, -0.5, 0.0, 1.0]])),
}


@pytest.mark.parametrize("case", sorted(BAD_SPECS))
def test_bad_arguments_are_reported_before_the_device(case):
    assert _code(**BAD_SPECS[case]) == _lib.ERR_ARG


def test_valid_call_without_a_device_is_a_cuda_error():
    if _lib.device_count() > 0:
        pytest.skip("a CUDA device is present")
    assert _code(windows=(1, 4), threshold=[1.0], ranges=[(1, 4)]) == _lib.ERR_CUDA
    assert _code(windows=(), threshold=[1.0], transform="boxcox", lams=[0.3]) == _lib.ERR_CUDA


def test_ctypes_structs_match_the_header():
    import re
    src = open(os.path.join(os.path.dirname(HERE), "..", "include", "ldsr_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    for name, cls in (("ldsr_stats_spec", _lib.StatsSpec), ("ldsr_stats_out", _lib.StatsOut)):
        end = src.index("} %s;" % name)
        body = src[src.rindex("typedef struct {", 0, end) + len("typedef struct {"):end]
        fields = [re.findall(r"[A-Za-z_][A-Za-z0-9_]*", d)[-1] for d in body.split(";") if d.strip()]
        assert fields == [f[0] for f in cls._fields_], name
