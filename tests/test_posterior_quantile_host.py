"""Per-step quantiles of w-step mean flows over conditioned replicates (ldsr_posterior_quantile_batch), without a GPU:
  * the reference (tests/posterior_quantile_oracle.py) on hand-written series with known answers: ranks at the level
    boundaries, levels 0 and 1, windows as long as the range and longer, non-finite flows;
  * the whole selection (range pass, histogram passes, single-key brackets, collecting pass and sort) run from
    source by the CPU emulator at widths 3 and 16 with caller noise, with 4 bins and a collect cap of 3 so that every
    path runs, equals the reference applied to the emulated trajectory mode's simQ for the same noise, bit for bit,
    and is bit-identical under four thread schedules and with the default bins and cap;
  * ldsr_posterior_quantile_batch checks its arguments before it looks for a device."""
import ctypes as C
import hashlib
import os
import re
import subprocess
import tempfile

import numpy as np
import pytest

from ldsr_b200 import _lib
from tests import posterior_quantile_oracle as PQO
from tests import test_gpu_step_kernels as SK
from tests import test_posterior_rep_host as PH

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_simt")
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ldsr_b200", "csrc")
_hostsim = None


def hostsim_lib():
    """tests/host_simt/sim_posterior_quantile.cpp built for the CPU, into the temporary directory under a name keyed by
    its sources (as test_posterior_yearly_host.py builds sim_posterior_yearly.cpp)."""
    global _hostsim
    if _hostsim is None:
        srcs = [os.path.join(HERE, f) for f in ("sim_posterior_quantile.cpp", "sim_posterior.cpp", "sim_em.cpp",
                                                "host_simt.h")]
        srcs += sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh"))
        key = hashlib.sha256(b"".join(open(f, "rb").read() for f in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "ldsr_hostsim_quant_%s_%d.so" % (key, os.getuid()))
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
def test_reference_ranks_at_the_level_boundaries():
    Q = np.arange(1.0, 11.0)[:, None]  # ten replicates, one step: values 1 .. 10
    r = PQO.quantiles(Q, (1,), (0.0, 0.1, 0.15, 0.5, 0.51, 0.9, 0.95, 1.0), 0, 1)
    # ranks max(1, ceil(p n)): 1, 1, 2, 5, 6, 9, 10, 10
    assert r["q"][0, :, 0].tolist() == [1, 1, 2, 5, 6, 9, 10, 10]
    assert r["nonfinite"][0].tolist() == [0]
    # numpy's inverted_cdf is the same estimator
    for p in (0.0, 0.1, 0.15, 0.5, 0.51, 0.9, 0.95, 1.0):
        assert np.quantile(Q[:, 0], p, method="inverted_cdf") == PQO.quantiles(Q, (1,), (p,), 0, 1)["q"][0, 0, 0]


def test_reference_windows_as_long_as_the_range_and_longer():
    Q = np.array([[9, 9, 1, 2, 3, 4, 5, 9, 9], [9, 9, 2, 2, 2, 2, 2, 9, 9]], dtype=float)
    r = PQO.quantiles(Q, (5, 6, 2), (0.0, 1.0), 2, 7)
    assert r["q"][0, :, 2].tolist() == [2.0, 3.0]  # one start: means 3 and 2
    assert np.isnan(r["q"][0, :, 3:]).all() and np.isnan(r["q"][0, :, :2]).all()
    assert np.isnan(r["q"][1]).all() and (r["nonfinite"][1] == -1).all()  # no start at all
    assert r["q"][2, 0, 2:6].tolist() == [1.5, 2.0, 2.0, 2.0]
    assert r["q"][2, 1, 2:6].tolist() == [2.0, 2.5, 3.5, 4.5]
    assert r["nonfinite"][2].tolist() == [-1, -1, 0, 0, 0, 0, -1, -1, -1]


def test_reference_non_finite_flows_leave_their_windows():
    Q = np.array([[1.0, np.nan, 3.0, 4.0], [2.0, 2.0, np.inf, 1.0], [3.0, 1.0, 1.0, 1.0]])
    r = PQO.quantiles(Q, (1, 2), (0.0, 0.5, 1.0), 0, 4)
    assert r["nonfinite"].tolist() == [[0, 1, 1, 0], [1, 2, 1, -1]]
    assert r["q"][0, :, 1].tolist() == [1.0, 1.0, 2.0]  # two values: ranks 1, 1, 2
    assert r["q"][1, :, 1].tolist() == [1.0, 1.0, 1.0]  # one window without a non-finite flow
    r = PQO.quantiles(np.array([[np.nan], [np.inf]]), (1,), (0.5,), 0, 1)
    assert np.isnan(r["q"][0, 0, 0]) and r["nonfinite"][0, 0] == 2


def test_reference_running_sum_is_the_kernels():
    # the downward running sum differs from a fresh sum in the last bits; the reference keeps the running one
    rng = np.random.default_rng(5)
    Q = np.exp(rng.standard_normal((3, 200)))
    M, ok = PQO.window_means(Q, 17, 5, 190)
    fresh = np.lib.stride_tricks.sliding_window_view(Q[:, 5:190], 17, axis=1).sum(axis=2) / 17.0
    assert ok.all() and np.allclose(M, fresh, rtol=1e-13, atol=0)
    S = 0.0
    for t in range(189, 5 - 1, -1):  # one replicate by hand
        S = S + Q[1, t]
        if 190 - t > 17:
            S = S - Q[1, t + 17]
        if 190 - t >= 17:
            assert M[1, t - 5] == S / 17.0


# ---- the emulated selection against the reference on the emulated trajectories ---------------------------------
def sim_quantile(s, held, fit_group, theta, n_reps, z, mu, tr, lams, windows, levels, ranges, nb_log2=2, cap=3,
                 order=0):
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
    lev = np.ascontiguousarray(levels, dtype=np.float64)
    rg = np.ascontiguousarray(ranges, dtype=np.int32)
    q = np.full((win.size, lev.size, nf * T), 7.0)
    nonfinite = np.full((win.size, nf * T), 7, dtype=np.int32)
    stats = np.zeros(3, dtype=np.int64)
    d = lambda a: None if a is None else a.ctypes.data_as(_dp)
    i = lambda a: None if a is None or a.size == 0 else a.ctypes.data_as(_ip)
    rc = L.hostsim_posterior_quantile(T, s["p"], s["q"], d(y), d(uf), d(vf), len(held), i(hp), i(hi), nf, i(fg),
                                      d(np.ascontiguousarray(theta, dtype=np.float64)), n_reps,
                                      d(np.ascontiguousarray(z)), d(np.ascontiguousarray(mu, dtype=np.float64)),
                                      _lib.TRANSFORMS[tr], d(np.ascontiguousarray(lams, dtype=np.float64)), win.size,
                                      i(win), lev.size, d(lev), i(rg), nb_log2, cap, order, d(q), i(nonfinite),
                                      stats.ctypes.data_as(C.POINTER(C.c_longlong)))
    assert rc == 0, rc
    return dict(q=q.reshape(win.size, lev.size, nf, T).transpose(2, 0, 1, 3),
                nonfinite=nonfinite.reshape(win.size, nf, T).transpose(1, 0, 2), passes=int(stats[0]),
                hist=int(stats[1]), collected=int(stats[2]))


def _ranges(rng, T):
    """Whole series, a short range inside or across 16-step tiles, and a long one that starts and ends off the tiles
    (where T allows)."""
    out = [(0, T)]
    if T >= 3:
        a = int(rng.integers(0, T - 2))
        out.append((a, min(T, a + 2 + int(rng.integers(0, 12)))))
    if T > 40:
        out.append((int(rng.integers(1, 14)), T - int(rng.integers(1, 14))))
    return out


# (transform, lambda, mu offset): Box-Cox with mu far below 0 makes (y + mu) lambda + 1 < 0 at some steps (NaN flows)
TRANSFORM_CASES = (("log", 0.0, 0.0), ("none", 0.0, 0.0), ("boxcox", 0.35, 3.0), ("boxcox", 0.35, -3.6))
TS = (2, 17, 64, 130, 213)
SPECS = (((1, 16), (0.0, 0.05, 0.5, 0.95, 1.0)), ((64,), (0.5,)), ((17, 1, 15), (0.0, 0.3, 0.31, 1.0)),
         ((15, 64, 1, 16), (0.1, 0.2, 0.25, 0.4, 0.5, 0.6, 0.75, 0.9)))


@pytest.mark.parametrize("width", [(3, 3, "vu"), (16, 16, "sep")], ids=SK.case_id)
def test_emulated_quantiles_equal_the_reference_on_the_emulated_trajectories(width):
    p, q, form = width
    rng = np.random.default_rng(p * 13 + q)
    n_nan = hist = collected = 0
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
            windows, levels = SPECS[(ti + ri) % len(SPECS)]
            got = sim_quantile(s, held, fit_group, theta, n_reps, z, mu, tr, lams, windows, levels, ranges)
            for f in range(nf):
                PQO.assert_match({k: got[k][f] for k in ("q", "nonfinite")}, traj[f], windows, levels, rg[0], rg[1],
                                 where=(T, rg, f, tr, windows, levels))
            n_nan += int((~np.isfinite(traj[:, :, rg[0]:rg[1]])).sum())
            hist += got["hist"]
            collected += got["collected"]
            # every thread schedule, and the default bins and cap, give the same bits
            for order, nb_log2, cap in ((1, 2, 3), (2, 2, 3), (3, 2, 3), (0, 11, 2048)):
                again = sim_quantile(s, held, fit_group, theta, n_reps, z, mu, tr, lams, windows, levels, ranges,
                                     nb_log2=nb_log2, cap=cap, order=order)
                assert np.array_equal(again["q"], got["q"], equal_nan=True), (T, rg, order, nb_log2)
                assert np.array_equal(again["nonfinite"], got["nonfinite"]), (T, rg, order, nb_log2)
                if nb_log2 == 2:
                    assert again["passes"] == got["passes"]
    assert n_nan > 0  # some replicates have non-finite flows in their range (Box-Cox)
    assert hist > 0 and collected > 0  # both kinds of bracket ran
    print("\n[emulator] %d histogram and %d collected brackets" % (hist, collected))


def test_emulated_selection_takes_several_histogram_passes():
    """40 replicates, 4 bins and a cap of 3: the brackets narrow over several passes (values spread over many keys
    need more than one histogram), and w = 1 at observed steps gives the observed flow at every level."""
    rng = np.random.default_rng(11)
    T = 48
    s = SK.make_series(rng, 3, 3, "vu", T)
    held = [SK.holdout(rng, s["y"], "none")]
    theta = SK.rand_theta(rng, 3, 3)[None, :]
    z = rng.standard_normal((1, 40, 2 * T))
    args = (s, held, np.array([0]), theta, 40, z, np.array([1.0]), "log", np.zeros(1), (1, 5), (0.0, 0.3, 0.5, 1.0),
            np.array([(0, T)]))
    got = sim_quantile(*args)
    assert got["passes"] >= 4, got["passes"]
    traj = PH.sim_posterior(s, held, np.array([0]), theta, 40, z, np.array([1.0]), "log", np.zeros(1),
                            want=("simQ",))["simQ"][0]
    ref = PQO.assert_match({k: got[k][0] for k in ("q", "nonfinite")}, traj, (1, 5), (0.0, 0.3, 0.5, 1.0), 0, T)
    obs = np.isfinite(s["y"])
    assert obs.any()
    for l in range(4):  # every replicate's flow is the observation there; the running sum (S + Q_t) - Q_{t+1}
        # gives it back to rounding, not bit for bit
        assert np.allclose(got["q"][0, 0, l, obs], traj[0, obs], rtol=1e-12, atol=0)
    d = np.diff(ref["q"], axis=1)  # quantiles do not decrease with the level
    assert (d[np.isfinite(d)] >= 0).all()


# ---- argument errors come before the device ---------------------------------------------------------------------
def _batch():
    y = np.array([0.1, np.nan, -0.2, 0.3])
    return dict(series=[dict(y=y, u=np.ones((1, 4)), v=None, p=1, q=1)], group_series=[0], held=None, fit_group=[0],
                theta=np.array([[0.5, 0.1, 0.8, 0.0, 1.0, 0.5, 0.0, 1.0]]))


def _code(**kw):
    b = _batch()
    args = dict(n_reps=4, windows=(2,), levels=(0.1, 0.9), ranges=None)
    args.update(kw)
    n_reps = args.pop("n_reps")
    try:
        _lib.posterior_quantile_batch(b["series"], b["group_series"], b["held"], b["fit_group"],
                                      args.pop("theta", b["theta"]), n_reps, **args)
    except _lib.LdsrError as e:
        return e.code
    return _lib.OK


BAD_SPECS = {
    "level_below_zero": dict(levels=(-0.1, 0.5)),
    "level_above_one": dict(levels=(0.5, 1.5)),
    "nan_level": dict(levels=(np.nan,)),
    "levels_not_increasing": dict(levels=(0.5, 0.5)),
    "levels_decreasing": dict(levels=(0.9, 0.1)),
    "no_level": dict(levels=()),
    "nine_levels": dict(levels=tuple(np.linspace(0.1, 0.9, 9))),
    "no_window": dict(windows=()),
    "five_windows": dict(windows=(1, 2, 3, 4, 5)),
    "window_of_zero": dict(windows=(0,)),
    "window_of_65": dict(windows=(10, 65)),
    "range_below_zero": dict(ranges=[(-1, 3)]),
    "empty_range": dict(ranges=[(2, 2)]),
    "range_past_the_end": dict(ranges=[(0, 5)]),
    "no_replicates": dict(n_reps=0),
    "unknown_transform": dict(transform=3),
    "box_cox_without_lambda": dict(transform="boxcox"),
    "negative_R": dict(theta=np.array([[0.5, 0.1, 0.8, 0.0, 1.0, -0.5, 0.0, 1.0]])),
}


def _code_raw(want_passes=True, **kw):
    """As _code, but through the C entry point itself with every output NULL unless asked for."""
    b = _batch()
    pb = _lib.PackedBatch(b["series"], b["group_series"], b["held"], b["fit_group"], b["theta"])
    win = np.array([2], dtype=np.int32)
    lev = np.array([0.5])
    passes = np.zeros(1, dtype=np.int32)
    spec = _lib.QuantSpec(1, win.ctypes.data_as(_ip), 1, lev.ctypes.data_as(_dp), None)
    out = _lib.QuantOut(None, None, passes.ctypes.data_as(_ip) if want_passes else None)
    err = C.create_string_buffer(512)
    return _lib.lib().ldsr_posterior_quantile_batch(None, C.byref(pb.c), 4, None, C.c_ulonglong(0), None, 1, None,
                                                    C.byref(spec), C.byref(out), err, 512)


@pytest.mark.parametrize("case", sorted(BAD_SPECS))
def test_bad_arguments_are_reported_before_the_device(case):
    assert _code(**BAD_SPECS[case]) == _lib.ERR_ARG


def test_every_output_null_is_an_argument_error():
    assert _code_raw(want_passes=False) == _lib.ERR_ARG


def test_valid_call_without_a_device_is_a_cuda_error():
    if _lib.device_count() > 0:
        pytest.skip("a CUDA device is present")
    assert _code(windows=(1, 4), levels=(0.0, 1.0), ranges=[(1, 4)]) == _lib.ERR_CUDA
    assert _code(windows=(64,), levels=tuple(np.linspace(0, 1, 8)), transform="boxcox", lams=[0.3]) == _lib.ERR_CUDA
    assert _code_raw(want_passes=True) == _lib.ERR_CUDA  # the pass count alone is an output


def test_ctypes_structs_match_the_header():
    src = open(os.path.join(os.path.dirname(HERE), "..", "include", "ldsr_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    for name, cls in (("ldsr_quant_spec", _lib.QuantSpec), ("ldsr_quant_out", _lib.QuantOut)):
        end = src.index("} %s;" % name)
        body = src[src.rindex("typedef struct {", 0, end) + len("typedef struct {"):end]
        fields = [re.findall(r"[A-Za-z_][A-Za-z0-9_]*", d)[-1] for d in body.split(";") if d.strip()]
        assert fields == [f[0] for f in cls._fields_], name
