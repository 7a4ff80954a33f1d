"""Year-by-year drought counts of conditioned replicates (ldsr_posterior_yearly_batch), without a GPU:
  * the reference (tests/posterior_yearly_oracle.py) on hand-written series with known answers: runs of L - 1, L and
    L + 1 steps, runs touching lo and hi, a run longer than 64 and a range all below, ranges shorter than the
    longest length, windows as long as the range and longer, L = 1 and L = 64, and non-finite flows inside a run,
    inside a window and outside the range;
  * the yearly mode of posterior_rep_kernel, run from source by the CPU emulator at widths 3 and 16 with caller
    noise, equals the reference applied to the emulated trajectory mode's simQ for the same noise, and is
    bit-identical under four thread schedules;
  * ldsr_posterior_yearly_batch checks its arguments before it looks for a device."""
import ctypes as C
import hashlib
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from ldsr_b200 import _lib
from tests import posterior_yearly_oracle as PY
from tests import test_gpu_step_kernels as SK
from tests import test_posterior_rep_host as PH

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_simt")
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ldsr_b200", "csrc")
_hostsim = None


def hostsim_lib():
    """tests/host_simt/sim_posterior_yearly.cpp built for the CPU, into the temporary directory under a name keyed by
    its sources (as test_posterior_stats_host.py builds sim_posterior_stats.cpp)."""
    global _hostsim
    if _hostsim is None:
        srcs = [os.path.join(HERE, f) for f in ("sim_posterior_yearly.cpp", "sim_posterior.cpp", "sim_em.cpp",
                                                "host_simt.h")]
        srcs += sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh"))
        key = hashlib.sha256(b"".join(open(f, "rb").read() for f in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "ldsr_hostsim_yearly_%s_%d.so" % (key, os.getuid()))
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
def _one(Q, thr=1.0, windows=(), lengths=(), lo=0, hi=None):
    Q = np.asarray(Q, dtype=float)
    return PY.counts(Q[None, :], thr, windows, lengths, lo, Q.size if hi is None else hi)


def test_reference_runs_of_l_minus_one_l_and_l_plus_one():
    # runs of 2, 3 and 4 steps below 1, separated by one step above
    Q = [0, 0, 5, 0, 0, 0, 5, 0, 0, 0, 0]
    r = _one(Q, lengths=(1, 2, 3, 4, 5))
    assert r["below"].tolist() == [1, 1, 0, 1, 1, 1, 0, 1, 1, 1, 1]
    assert r["in_run"][0].tolist() == r["below"].tolist()
    assert r["in_run"][1].tolist() == [1, 1, 0, 1, 1, 1, 0, 1, 1, 1, 1]
    assert r["in_run"][2].tolist() == [0, 0, 0, 1, 1, 1, 0, 1, 1, 1, 1]
    assert r["in_run"][3].tolist() == [0, 0, 0, 0, 0, 0, 0, 1, 1, 1, 1]
    assert r["in_run"][4].tolist() == [0] * 11
    assert r["nonfinite"].tolist() == [0] * 11


def test_reference_clips_runs_at_lo_and_hi():
    Q = [0, 0, 0, 0, 5, 0, 0, 0, 0]
    whole = _one(Q, lengths=(3, 4))
    assert whole["in_run"][1].tolist() == [1, 1, 1, 1, 0, 1, 1, 1, 1]
    # [2, 7): the run 0..3 is cut to 2..3 and the run 5..8 to 5..6
    r = _one(Q, lengths=(2, 3), lo=2, hi=7)
    assert r["in_run"][0].tolist() == [-1, -1, 1, 1, 0, 1, 1, -1, -1]
    assert r["in_run"][1].tolist() == [-1, -1, 0, 0, 0, 0, 0, -1, -1]
    assert r["below"].tolist() == [-1, -1, 1, 1, 0, 1, 1, -1, -1]


def test_reference_run_longer_than_64_and_a_range_all_below():
    Q = np.zeros(150)
    Q[[10, 100]] = 5.0  # runs 0..9, 11..99 (89 steps) and 101..149 (49 steps)
    r = _one(Q, lengths=(1, 50, 64))
    assert (r["in_run"][1][11:100] == 1).all() and (r["in_run"][1][101:] == 0).all()
    assert (r["in_run"][2][11:100] == 1).all() and (r["in_run"][2][:10] == 0).all()
    allb = _one(np.zeros(70), lengths=(64, 1))
    assert (allb["in_run"] == 1).all()
    assert (_one(np.zeros(63), lengths=(64,))["in_run"] == 0).all()  # a whole range of 63 steps is too short


def test_reference_ranges_shorter_than_the_longest_length_and_not_on_tiles():
    Q = np.zeros(40)
    Q[20] = 5.0
    r = _one(Q, lengths=(3, 17), lo=17, hi=23)  # runs 17..19 and 21..22 inside [17, 23)
    assert r["in_run"][0].tolist()[17:23] == [1, 1, 1, 0, 0, 0]
    assert r["in_run"][1].tolist()[17:23] == [0] * 6
    assert (r["in_run"][:, :17] == -1).all() and (r["in_run"][:, 23:] == -1).all()


def test_reference_windows_as_long_as_the_range_and_longer():
    Q = [9, 9, 1, 2, 3, 4, 5, 9, 9]
    r = _one(Q, thr=3.5, windows=(5, 6, 1, 2), lo=2, hi=7)
    assert r["wbelow"][0].tolist() == [-1, -1, 1, -1, -1, -1, -1, -1, -1]  # one start, mean 3 < 3.5
    assert (r["wbelow"][1] == -1).all()  # no start at all
    assert r["wbelow"][2].tolist() == r["below"].tolist() == [-1, -1, 1, 1, 1, 0, 0, -1, -1]
    assert r["wbelow"][3].tolist() == [-1, -1, 1, 1, 0, 0, -1, -1, -1]  # means 1.5, 2.5, 3.5 (not below), 4.5


def test_reference_non_finite_flows_inside_a_run_a_window_and_outside_the_range():
    Q = [0.0, 0.5, np.nan, 0.2, 0.1, 3.0, np.inf, 0.3]
    r = _one(Q, windows=(2, 1), lengths=(2, 1))
    assert r["below"].tolist() == [1, 1, 0, 1, 1, 0, 0, 1]  # NaN and Inf are not below
    assert r["nonfinite"].tolist() == [0, 0, 1, 0, 0, 0, 1, 0]
    assert r["in_run"][0].tolist() == [1, 1, 0, 1, 1, 0, 0, 0]  # the NaN splits the run
    assert r["wbelow"][0].tolist() == [1, 0, 0, 1, 0, 0, 0, -1]  # windows holding NaN or Inf count nowhere
    assert r["wbelow"][1].tolist() == r["below"].tolist()
    r = _one(Q, windows=(2,), lengths=(2,), lo=3, hi=6)  # both non-finite flows lie outside [3, 6)
    assert r["below"].tolist()[3:6] == [1, 1, 0] and r["nonfinite"].tolist()[3:6] == [0, 0, 0]
    assert r["in_run"][0].tolist()[3:6] == [1, 1, 0] and r["wbelow"][0].tolist()[3:6] == [1, 0, -1]


def test_reference_identities_on_random_flows():
    rng = np.random.default_rng(3)
    Q = rng.standard_normal((50, 300)).cumsum(axis=1) * 0.1
    Q[rng.random(Q.shape) < 0.01] = np.nan
    r = PY.counts(Q, 0.0, (1, 7, 64), (1, 2, 5, 64), 13, 290)
    assert np.array_equal(r["in_run"][0], r["below"]) and np.array_equal(r["wbelow"][0], r["below"])
    d = np.diff(r["in_run"][:, 13:290], axis=0)
    assert (d <= 0).all()


# ---- the emulated kernel against the reference on the emulated trajectories --------------------------------------
def sim_yearly(s, held, fit_group, theta, n_reps, z, mu, tr, lams, windows, lengths, thr, ranges, order=0):
    L = hostsim_lib()
    y = np.ascontiguousarray(s["y"], dtype=np.float64)
    uf = None if s["u"] is None else np.ascontiguousarray(np.asarray(s["u"], dtype=np.float64).T)
    vf = None if s["v"] is None else np.ascontiguousarray(np.asarray(s["v"], dtype=np.float64).T)
    hp = np.zeros(len(held) + 1, dtype=np.int32)
    hp[1:] = np.cumsum([len(h) for h in held])
    hi = np.ascontiguousarray(np.concatenate([np.asarray(h, dtype=np.int32) for h in held] + [np.zeros(1, np.int32)]))
    fg = np.ascontiguousarray(fit_group, dtype=np.int32)
    nf, T = fg.size, s["y"].size
    win = np.ascontiguousarray(windows, dtype=np.int32)
    lens = np.ascontiguousarray(lengths, dtype=np.int32)
    rg = np.ascontiguousarray(ranges, dtype=np.int32)
    outs = {k: np.full((n, nf * T), 7, dtype=np.int32)
            for k, n in (("below", 1), ("in_run", lens.size), ("wbelow", win.size), ("nonfinite", 1))}
    d = lambda a: None if a is None else a.ctypes.data_as(_dp)
    i = lambda a: None if a is None or a.size == 0 else a.ctypes.data_as(_ip)
    rc = L.hostsim_posterior_yearly(T, s["p"], s["q"], d(y), d(uf), d(vf), len(held), i(hp), i(hi), nf, i(fg),
                                    d(np.ascontiguousarray(theta, dtype=np.float64)), n_reps,
                                    d(np.ascontiguousarray(z)), d(np.ascontiguousarray(mu, dtype=np.float64)),
                                    _lib.TRANSFORMS[tr], d(np.ascontiguousarray(lams, dtype=np.float64)), win.size,
                                    i(win), lens.size, i(lens), d(np.ascontiguousarray(thr, dtype=np.float64)),
                                    i(rg), order, *(i(outs[k]) for k in _lib.YEARLY_COUNTS))
    assert rc == 0, rc
    return {k: v.reshape(v.shape[0], nf, T).transpose(1, 0, 2) for k, v in outs.items()}  # [nf, n, T]


def _ranges(rng, T):
    """Whole series, a short range inside or across 16-step tiles (shorter than most lengths), and a long one that
    starts and ends off the tiles (where T allows)."""
    out = [(0, T)]
    if T >= 3:
        a = int(rng.integers(0, T - 2))
        out.append((a, min(T, a + 2 + int(rng.integers(0, 12)))))
    if T > 40:
        out.append((int(rng.integers(1, 14)), T - int(rng.integers(1, 14))))
    return out


# (transform, lambda, mu offset): Box-Cox with mu far below 0 makes (y + mu) lambda + 1 < 0 at some steps (NaN flows)
TRANSFORM_CASES = (("log", 0.0, 0.0), ("none", 0.0, 0.0), ("boxcox", 0.35, 3.0), ("boxcox", 0.0, 0.0),
                   ("boxcox", 0.35, -3.6))
TS = (2, 15, 17, 64, 65, 130, 213, 300)
SPECS = (((1, 16), (1, 3, 17)), ((64,), (64, 2)), ((17, 2, 5), (5,)), ((3,), ()), ((), (1, 16, 33, 64)),
         ((15, 64, 1, 33), (10, 4, 1, 2)))


@pytest.mark.parametrize("width", [(3, 3, "vu"), (16, 16, "sep")], ids=SK.case_id)
def test_emulated_counts_equal_the_reference_on_the_emulated_trajectories(width):
    p, q, form = width
    rng = np.random.default_rng(p * 11 + q)
    n_nan = n_near = 0
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
            windows, lengths = SPECS[(ti + ri) % len(SPECS)]
            Qin = traj[:, :, rg[0]:rg[1]]
            thr = np.array([np.nanmedian(Qin[f]) if np.isfinite(Qin[f]).any() else 1.0 for f in range(nf)])
            got = sim_yearly(s, held, fit_group, theta, n_reps, z, mu, tr, lams, windows, lengths, thr, ranges)
            for f in range(nf):
                g = {k: got[k][f] for k in ("in_run", "wbelow")}
                g.update(below=got["below"][f, 0], nonfinite=got["nonfinite"][f, 0])
                n_near += PY.assert_match(g, traj[f], thr[f], windows, lengths, rg[0], rg[1],
                                          where=(T, rg, f, tr, windows, lengths))
            n_nan += int((~np.isfinite(Qin)).sum())
            # every thread schedule gives the same counts
            for order in (1, 2, 3):
                again = sim_yearly(s, held, fit_group, theta, n_reps, z, mu, tr, lams, windows, lengths, thr, ranges,
                                   order=order)
                for k in got:
                    assert np.array_equal(again[k], got[k]), (T, rg, order, k)
    assert n_nan > 0  # some replicates have non-finite flows in their range (Box-Cox)
    print("\n[emulator] %d window starts near the threshold" % n_near)


# ---- argument errors come before the device ---------------------------------------------------------------------
def _batch():
    y = np.array([0.1, np.nan, -0.2, 0.3])
    return dict(series=[dict(y=y, u=np.ones((1, 4)), v=None, p=1, q=1)], group_series=[0], held=None, fit_group=[0],
                theta=np.array([[0.5, 0.1, 0.8, 0.0, 1.0, 0.5, 0.0, 1.0]]))


def _code(**kw):
    b = _batch()
    args = dict(n_reps=4, windows=(2,), lengths=(2,), threshold=[1.0], ranges=None)
    args.update(kw)
    n_reps = args.pop("n_reps")
    try:
        _lib.posterior_yearly_batch(b["series"], b["group_series"], b["held"], b["fit_group"],
                                    args.pop("theta", b["theta"]), n_reps, **args)
    except _lib.LdsrError as e:
        return e.code
    return _lib.OK


BAD_SPECS = {
    "no_threshold": dict(threshold=None),
    "nan_threshold": dict(threshold=[np.nan]),
    "infinite_threshold": dict(threshold=[-np.inf]),
    "five_windows": dict(windows=(1, 2, 3, 4, 5)),
    "five_lengths": dict(lengths=(1, 2, 3, 4, 5)),
    "window_of_zero": dict(windows=(0,)),
    "window_of_65": dict(windows=(10, 65)),
    "length_of_zero": dict(lengths=(3, 0)),
    "length_of_65": dict(lengths=(65,)),
    "range_below_zero": dict(ranges=[(-1, 3)]),
    "empty_range": dict(ranges=[(2, 2)]),
    "range_past_the_end": dict(ranges=[(0, 5)]),
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
    assert _code(windows=(1, 4), lengths=(1, 64), ranges=[(1, 4)]) == _lib.ERR_CUDA
    assert _code(windows=(), lengths=(), transform="boxcox", lams=[0.3]) == _lib.ERR_CUDA


def test_ctypes_structs_match_the_header():
    src = open(os.path.join(os.path.dirname(HERE), "..", "include", "ldsr_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    for name, cls in (("ldsr_yearly_spec", _lib.YearlySpec), ("ldsr_yearly_out", _lib.YearlyOut)):
        end = src.index("} %s;" % name)
        body = src[src.rindex("typedef struct {", 0, end) + len("typedef struct {"):end]
        fields = [re.findall(r"[A-Za-z_][A-Za-z0-9_]*", d)[-1] for d in body.split(";") if d.strip()]
        assert fields == [f[0] for f in cls._fields_], name
