"""Drought statistics of conditioned replicates (ldsr_posterior_stats_batch, api.LDS_rep_posterior_stats) on the GPU:
  * the same seed gives the statistics of ldsr_posterior_rep_batch's simQ (the CPU reference,
    tests/posterior_stats_oracle.py, applied to it) at four input widths, over fits of T = 2 .. 213 in one launch
    with the six hold-out kinds, per-fit ranges and thresholds, and Box-Cox flows that are not finite;
  * caller noise gives the statistics of the CPU reference replicates (tests/posterior_oracle.py) for that noise;
  * NPlds at 100 000 replicates, 1 000 000 replicates of one fit, determinism, and the Python API.
Run with -s to see the largest deviations and the NPlds drought share."""
import numpy as np
import pytest

import ldsr_b200 as L
from ldsr_b200 import _lib, api
from tests import data
from tests import posterior_oracle as PO
from tests import posterior_stats_oracle as PS
from tests import test_gpu_posterior_rep as PR
from tests import test_gpu_step_kernels as SK

pytestmark = pytest.mark.gpu

WINDOWS = ((1, 16, 17, 64), (15, 2), (64,), (3, 5, 10, 30))
CASES = [(3, 3, "vu"), (10, 10, "sep"), (1, 3, "unone"), (24, 24, "vu")]
TRANSFORMS = (("log", 0.0, 0.0), ("none", 0.0, 0.0), ("boxcox", 0.3, 4.0), ("boxcox", 0.3, -3.5))


def _spec(rng, Ts):
    """Per fit: the whole series, or a range starting and ending inside tiles."""
    ranges = []
    for T in Ts:
        lo = 0 if T < 4 or rng.random() < 0.4 else int(rng.integers(0, T // 2))
        hi = T if rng.random() < 0.5 else int(rng.integers(lo + 1, T + 1))
        ranges.append((lo, hi))
    return np.array(ranges, dtype=np.int32)


def _per_fit(r, f):
    return {k: (v[:, f] if v.ndim == 3 else v[f]) for k, v in r.items() if k != "device_ms"}


def _thresholds(Q, ranges):
    """The mean of each fit's finite flows in its range: not one of the flows (a median can be), so that the last bit
    of a reference flow cannot move it across the threshold."""
    out = []
    for q, (lo, hi) in zip(Q, ranges):
        fin = q[:, lo:hi][np.isfinite(q[:, lo:hi])]
        out.append(np.mean(fin) if fin.size else 1.0)
    return np.array(out)


@pytest.mark.parametrize("width", CASES, ids=SK.case_id)
def test_same_seed_gives_the_statistics_of_the_trajectory_call(width):
    i = CASES.index(width)
    c = PR.make_case(*width, seed=900 + i)
    nf = c["fit_group"].size
    Ts = PR.fit_T(c)
    rng = np.random.default_rng(i)
    tr, lam, dmu = TRANSFORMS[i]
    mu = rng.uniform(0.5, 1.5, nf) + dmu
    lams = np.full(nf, lam)
    n_reps = (45, 70, 33, 100)[i]
    windows = WINDOWS[i]
    kw = dict(seed=55 + i, mu=mu, transform=tr, lams=lams)
    Q = PR.call(c, n_reps, want=("simQ",), **kw)["simQ"]
    ranges = _spec(rng, Ts)
    thr = _thresholds(Q, ranges)
    g = _lib.posterior_stats_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], n_reps,
                                   windows=windows, threshold=thr, ranges=ranges, **kw)
    dev, n_bad = 0.0, 0
    for f in range(nf):
        dev = max(dev, PS.assert_match(_per_fit(g, f), Q[f], windows, thr[f], *ranges[f], where=(f, Ts[f])))
        n_bad += int((~np.isfinite(Q[f][:, ranges[f][0]:ranges[f][1]]).all(axis=1)).sum())
    if tr == "boxcox" and dmu < 0:
        assert n_bad > 0  # the case meant to produce non-finite flows did
    print("\n[max deviation] posterior_stats %s: %.1e, %d replicates with non-finite flows" % (SK.case_id(width), dev,
                                                                                              n_bad))


def test_caller_noise_gives_the_statistics_of_the_reference_replicates():
    c = PR.make_case(3, 3, "vu", seed=31)
    nf = c["fit_group"].size
    Ts = PR.fit_T(c)
    rng = np.random.default_rng(4)
    n_reps = 37
    mu = rng.uniform(0.5, 1.5, nf)
    z = rng.standard_normal(2 * n_reps * Ts.sum())
    off = 2 * n_reps * np.concatenate([[0], np.cumsum(Ts)])
    Q = []
    for f in range(nf):
        s, y = SK.group_y(c, c["fit_group"][f])
        zf = z[off[f]:off[f + 1]].reshape(n_reps, 2 * Ts[f])
        Q.append(PO.posterior_rep(c["theta"][f], y, s["u"], s["v"], zf, mu=mu[f], transform="log", p=3, q=3)["simQ"])
    ranges = _spec(rng, Ts)
    thr = _thresholds(Q, ranges)
    windows = (1, 4, 16, 33)
    g = _lib.posterior_stats_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], n_reps, z=z,
                                   mu=mu, transform="log", windows=windows, threshold=thr, ranges=ranges)
    for f in range(nf):
        PS.assert_match(_per_fit(g, f), Q[f], windows, thr[f], *ranges[f], where=f)


def test_nplds_at_scale():
    """NPlds theta, 100 000 replicates of T = 813 from 1200, windows of 5, 10, 20 and 30 years, the pre-instrumental
    years 1200-1959 and the mean of the observed flows as threshold; compared in blocks of 10 000 replicates."""
    g, y, u, mu, th = PR._nplds()
    qa = np.array(data.load("np.json")["NPannual"]["Qa"])
    N, windows, lo, hi = 100000, (5, 10, 20, 30), 0, 1960 - 1200
    thr = float(qa.mean())
    kw = dict(seed=2025, mu=[mu], transform="log")
    st = _lib.posterior_stats_batch([dict(y=y, u=u, v=u)], [0], None, [0], th[None, :], N, windows=windows,
                                    threshold=[thr], ranges=[(lo, hi)], **kw)
    Q = _lib.posterior_rep_batch([dict(y=y, u=u, v=u)], [0], None, [0], th[None, :], N, want=("simQ",), **kw)["simQ"][0]
    dev = 0.0
    for b0 in range(0, N, 10000):
        blk = {k: (v[:, 0, b0:b0 + 10000] if v.ndim == 3 else v[0, b0:b0 + 10000])
               for k, v in st.items() if k != "device_ms"}
        dev = max(dev, PS.assert_match(blk, Q[b0:b0 + 10000], windows, thr, lo, hi, where=b0))
    inst10 = np.convolve(qa, np.ones(10) / 10, mode="valid").min()
    share = float(np.mean(st["wmin"][1, 0] < inst10))
    print("\n[nplds] max deviation %.1e; %.4f of the replicates have a pre-instrumental 10-year mean below the "
          "instrumental minimum (%.1f); device %.2f ms" % (dev, share, inst10, st["device_ms"]))


def test_determinism_and_independence_of_the_batch():
    c = PR.make_case(3, 3, "vu", 5)
    nf = c["fit_group"].size
    kw = dict(seed=123, mu=0.4, transform="log", windows=(2, 10), threshold=np.full(nf, np.exp(0.4)))
    call = lambda cc, n, **k: _lib.posterior_stats_batch(cc["series"], cc["group_series"], cc["held"],
                                                         cc["fit_group"], cc["theta"], n, **dict(kw, **k))
    keys = _lib.WINDOW_STATS + _lib.RUN_STATS
    a, b, big = call(c, 40), call(c, 40), call(c, 1000)
    for k in keys:
        assert np.array_equal(a[k], b[k], equal_nan=True), k
        assert np.array_equal(big[k][..., :40], a[k], equal_nan=True), k
    # a fit added after the others leaves their rows alone
    c2 = dict(c, fit_group=np.append(c["fit_group"], c["fit_group"][-1]), theta=np.vstack([c["theta"], c["theta"][0]]))
    e = call(c2, 40, threshold=np.full(nf + 1, np.exp(0.4)))
    for k in keys:
        assert np.array_equal(e[k][..., :nf, :], a[k], equal_nan=True), k
    ctx = _lib.Ctx(n_devices=1)
    try:
        for seed in (1, 2):
            r1, r2 = call(c, 50, seed=seed, ctx=ctx), call(c, 50, seed=seed)
            for k in keys:
                assert np.array_equal(r1[k], r2[k], equal_nan=True), (seed, k)
    finally:
        ctx.close()


def test_a_million_replicates_of_one_fit():
    g, y, u, mu, th = PR._nplds()
    N = 1000000
    r = _lib.posterior_stats_batch([dict(y=y, u=u, v=u)], [0], None, [0], th[None, :], N, seed=7, mu=[mu],
                                   windows=(5, 10, 20, 30, ), threshold=[float(np.exp(mu))])
    for k in ("wmin", "wmax", "deficit"):
        assert np.isfinite(r[k]).all(), k
    for k in ("wmin_at", "wmax_at"):
        assert (r[k] >= 0).all() and (r[k] <= y.size - 5).all(), k
    assert (r["n_runs"] >= 1).all() and (r["run_len"] >= 1).all()
    print("\n[1e6 replicates] device %.2f ms" % r["device_ms"])


def test_api_ensemble_equals_the_library_call_and_reports_years():
    st = PR._ensemble_station()
    P, B = api.reconstruction_batch([st], "boxcox", 1, np.random.default_rng(0))
    S = P[0]
    rng = np.random.default_rng(8)
    thetas = [api.vec_to_theta(SK.rand_theta(rng, s["p"], s["q"]), s["p"], s["q"]) for s in S["series"]]
    for t in thetas:
        t["R"] = 0.05
    n_reps, windows, period = 50, (3, 10), (1850, 1990)
    out = L.LDS_rep_posterior_stats(thetas, st["Qa"], st["u"], st["v"], st["start_year"], transform="boxcox",
                                    num_reps=n_reps, seed=31, windows=windows, period=period)
    assert isinstance(out, list) and len(out) == 2
    stride = max(s["p"] + s["q"] + 6 for s in S["series"])
    rows = np.stack([np.pad(api.theta_to_vec(t), (0, stride - api.theta_to_vec(t).size)) for t in thetas])
    y0 = int(S["years"][0])
    thr = float(np.mean(st["Qa"]["Qa"]))
    ref = _lib.posterior_stats_batch(B["series"], [0, 1], None, [0, 1], rows, n_reps, seed=31, mu=[S["mu"]] * 2,
                                     transform="boxcox", lams=[S["lam"]] * 2, windows=windows, threshold=[thr] * 2,
                                     ranges=[(period[0] - y0, period[1] - y0 + 1)] * 2)
    year = lambda a: np.where(a >= 0, a + y0, -1)
    for k in range(2):
        o = out[k]
        assert o["threshold"] == thr and o["period"] == period and o["windows"] == windows
        for name, key in (("wmin", "wmin"), ("wmax", "wmax")):
            assert np.array_equal(o[name], ref[key][:, k], equal_nan=True)
            assert np.array_equal(o[name + "_year"], year(ref[key + "_at"][:, k]))
        assert np.array_equal(o["deficit"], ref["deficit"][k], equal_nan=True)
        assert np.array_equal(o["run_year"], year(ref["run_at"][k]))
        assert np.array_equal(o["deficit_year"], year(ref["deficit_at"][k]))
        assert np.array_equal(o["run_len"], ref["run_len"][k]) and np.array_equal(o["n_runs"], ref["n_runs"][k])
        ok = o["wmin_year"] >= 0
        assert (o["wmin_year"][ok] >= period[0]).all() and (o["wmin_year"][ok] <= period[1] - 2).all()
    # the same draws as LDS_rep_posterior: its simQ gives these statistics
    reps = L.LDS_rep_posterior(thetas, st["Qa"], st["u"], st["v"], st["start_year"], transform="boxcox",
                               num_reps=n_reps, seed=31)
    for k in range(2):
        Q = reps[k]["simQ"].reshape(n_reps, S["years"].size)
        got = {kk: ref[kk][:, k] if ref[kk].ndim == 3 else ref[kk][k] for kk in _lib.WINDOW_STATS + _lib.RUN_STATS}
        PS.assert_match(got, Q, windows, thr, period[0] - y0, period[1] - y0 + 1, where=k)
