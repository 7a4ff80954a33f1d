"""Year-by-year drought counts of conditioned replicates (ldsr_posterior_yearly_batch, api.LDS_rep_posterior_yearly)
on the GPU:
  * the same seed gives the counts of ldsr_posterior_rep_batch's simQ (the CPU reference,
    tests/posterior_yearly_oracle.py, applied to it) at four input widths, over fits of T = 2 .. 213 in one launch
    with the six hold-out kinds, per-fit ranges and thresholds, and Box-Cox flows that are not finite; also with
    caller noise, and on a long synthetic series (T = 20 000);
  * the identities in_run(L = 1) = wbelow(w = 1) = below and in_run non-increasing in L, exactly;
  * determinism, independence of the other fits and of the outputs asked for;
  * NPlds at 10^6 replicates: the share below the threshold at every unobserved year is the smoother's marginal
    probability within 5 binomial sigma;
  * the Python API.
Run with -s to see the number of window starts near the threshold and the device times."""
import math

import numpy as np
import pytest

import ldsr_b200 as L
from ldsr_b200 import _lib, api
from tests import data
from tests import posterior_yearly_oracle as PY
from tests import test_gpu_posterior_rep as PR
from tests import test_gpu_step_kernels as SK

pytestmark = pytest.mark.gpu

CASES = [(3, 3, "vu"), (10, 10, "sep"), (1, 3, "unone"), (24, 24, "vu")]
TRANSFORMS = (("log", 0.0, 0.0), ("none", 0.0, 0.0), ("boxcox", 0.3, 4.0), ("boxcox", 0.3, -3.5))
SPECS = (((1, 16, 17, 64), (1, 5, 17, 64)), ((15, 2), (3, 2)), ((64,), (64,)), ((3, 5, 10, 30), (1, 10, 30, 40)))


def _spec(rng, Ts):
    """Per fit: the whole series, or a range starting and ending inside tiles."""
    ranges = []
    for T in Ts:
        lo = 0 if T < 4 or rng.random() < 0.4 else int(rng.integers(0, T // 2))
        hi = T if rng.random() < 0.5 else int(rng.integers(lo + 1, T + 1))
        ranges.append((lo, hi))
    return np.array(ranges, dtype=np.int32)


def _thresholds(Q, ranges):
    """The mean of each fit's finite flows in its range (not one of the flows, so that the last bit of a flow cannot
    move it across the threshold)."""
    out = []
    for q, (lo, hi) in zip(Q, ranges):
        fin = q[:, lo:hi][np.isfinite(q[:, lo:hi])]
        out.append(np.mean(fin) if fin.size else 1.0)
    return np.array(out)


def _per_fit(r, f):
    return {k: r[k][f] for k in _lib.YEARLY_COUNTS if k in r}


def _check_identities(r, f, windows, lengths):
    b = r["below"][f]
    for k, Lk in enumerate(lengths):
        if Lk == 1:
            assert np.array_equal(r["in_run"][f][k], b)
    for k, w in enumerate(windows):
        if w == 1:
            assert np.array_equal(r["wbelow"][f][k], b)
    order = np.argsort(lengths, kind="stable")
    ir = r["in_run"][f][order]
    ok = b >= 0
    assert (np.diff(ir[:, ok], axis=0) <= 0).all()


@pytest.mark.parametrize("width", CASES, ids=SK.case_id)
def test_same_seed_gives_the_counts_of_the_trajectory_call(width):
    i = CASES.index(width)
    c = PR.make_case(*width, seed=950 + i)
    nf = c["fit_group"].size
    Ts = PR.fit_T(c)
    rng = np.random.default_rng(i)
    tr, lam, dmu = TRANSFORMS[i]
    mu = rng.uniform(0.5, 1.5, nf) + dmu
    lams = np.full(nf, lam)
    n_reps = (45, 70, 33, 100)[i]
    windows, lengths = SPECS[i]
    kw = dict(seed=65 + i, mu=mu, transform=tr, lams=lams)
    Q = PR.call(c, n_reps, want=("simQ",), **kw)["simQ"]
    ranges = _spec(rng, Ts)
    thr = _thresholds(Q, ranges)
    g = _lib.posterior_yearly_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], n_reps,
                                    windows=windows, lengths=lengths, threshold=thr, ranges=ranges, **kw)
    n_near, n_bad = 0, 0
    for f in range(nf):
        n_near += PY.assert_match(_per_fit(g, f), Q[f], thr[f], windows, lengths, *ranges[f], where=(f, Ts[f]))
        _check_identities(g, f, windows, lengths)
        n_bad += int(g["nonfinite"][f][g["nonfinite"][f] > 0].sum())
    if tr == "boxcox" and dmu < 0:
        assert n_bad > 0  # the case meant to produce non-finite flows did
    print("\n[yearly] %s: %d window starts near the threshold, %d non-finite flows" % (SK.case_id(width), n_near,
                                                                                       n_bad))


def test_caller_noise_gives_the_counts_of_the_trajectory_call():
    c = PR.make_case(3, 3, "vu", seed=41)
    nf = c["fit_group"].size
    Ts = PR.fit_T(c)
    rng = np.random.default_rng(5)
    n_reps = 37
    mu = rng.uniform(0.5, 1.5, nf)
    z = rng.standard_normal(2 * n_reps * Ts.sum())
    Q = PR.call(c, n_reps, z=z, mu=mu, transform="log", want=("simQ",))["simQ"]
    ranges = _spec(rng, Ts)
    thr = _thresholds(Q, ranges)
    windows, lengths = (1, 4, 16, 33), (2, 7, 1)
    g = _lib.posterior_yearly_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], n_reps, z=z,
                                    mu=mu, transform="log", windows=windows, lengths=lengths, threshold=thr,
                                    ranges=ranges)
    for f in range(nf):
        PY.assert_match(_per_fit(g, f), Q[f], thr[f], windows, lengths, *ranges[f], where=f)
        _check_identities(g, f, windows, lengths)


def test_a_long_series():
    """One synthetic series of 20 000 steps, three fits (whole series, a range off the tiles, a short range), 300
    replicates: 625 warps' counts added per step, every tile and the flush of every delay."""
    rng = np.random.default_rng(12)
    T = 20000
    s = SK.make_series(rng, 3, 3, "vu", T)
    theta = np.stack([SK.rand_theta(rng, 3, 3) for _ in range(3)])
    n_reps = 300
    kw = dict(seed=99, mu=[0.7, 0.9, 1.1], transform="log")
    Q = _lib.posterior_rep_batch([s], [0], None, [0, 0, 0], theta, n_reps, want=("simQ",), **kw)["simQ"]
    ranges = np.array([(0, T), (7, T - 9), (19990, 19997)], dtype=np.int32)
    thr = _thresholds(Q, ranges)
    windows, lengths = (64, 10, 1), (64, 5, 1, 20)
    g = _lib.posterior_yearly_batch([s], [0], None, [0, 0, 0], theta, n_reps, windows=windows, lengths=lengths,
                                    threshold=thr, ranges=ranges, **kw)
    for f in range(3):
        PY.assert_match(_per_fit(g, f), Q[f], thr[f], windows, lengths, *ranges[f], where=f)
        _check_identities(g, f, windows, lengths)
    assert (g["in_run"][0][1] > 0).any()  # runs of 5 steps and more occur


def test_determinism_and_independence_of_the_batch_and_of_the_outputs():
    c = PR.make_case(3, 3, "vu", 5)
    nf = c["fit_group"].size
    kw = dict(seed=123, mu=0.4, transform="log", windows=(2, 10), lengths=(3, 1), threshold=np.full(nf, np.exp(0.4)))
    call = lambda cc, n, **k: _lib.posterior_yearly_batch(cc["series"], cc["group_series"], cc["held"],
                                                          cc["fit_group"], cc["theta"], n, **dict(kw, **k))
    a, b = call(c, 1000), call(c, 1000)
    for k in _lib.YEARLY_COUNTS:
        for f in range(nf):
            assert np.array_equal(a[k][f], b[k][f]), k
    # a fit added after the others leaves their counts alone
    c2 = dict(c, fit_group=np.append(c["fit_group"], c["fit_group"][-1]), theta=np.vstack([c["theta"], c["theta"][0]]))
    e = call(c2, 1000, threshold=np.full(nf + 1, np.exp(0.4)))
    for k in _lib.YEARLY_COUNTS:
        for f in range(nf):
            assert np.array_equal(e[k][f], a[k][f]), k
    # each output alone is the same as with the others
    for k in _lib.YEARLY_COUNTS:
        one = call(c, 1000, want=(k,))
        assert set(one) == {k, "device_ms"}
        for f in range(nf):
            assert np.array_equal(one[k][f], a[k][f]), k


def test_nplds_million_replicates_match_the_smoothers_marginals():
    """NPlds theta, 10^6 replicates of T = 813: at each of the 767 unobserved years, the share of replicates below
    the threshold (the mean of the observed flows) is Phi((log thr - mu - Y_t) / sqrt(C^2 V_t + R)) within 5
    binomial sigma, Y_t and V_t from smoother_batch."""
    g, y, u, mu, th = PR._nplds()
    qa = np.array(data.load("np.json")["NPannual"]["Qa"])
    N, thr = 1000000, float(qa.mean())
    r = _lib.posterior_yearly_batch([dict(y=y, u=u, v=u)], [0], None, [0], th[None, :], N, seed=2026, mu=[mu],
                                    transform="log", windows=(10, 1), lengths=(5, 1), threshold=[thr])
    sm = _lib.smoother_batch([dict(y=y, u=u, v=u)], [0], None, [0], th[None, :])
    p, q = 3, 3
    C, R = th[1 + p], th[3 + p + q]
    Y, V = np.asarray(sm["Y"][0]), np.asarray(sm["V"][0])
    un = np.isnan(y)
    assert un.sum() == 767
    erf = np.vectorize(math.erf)
    P = 0.5 * (1 + erf((np.log(thr) - mu - Y) / np.sqrt(C * C * V + R) / math.sqrt(2)))
    share = r["below"][0] / N
    sig = np.sqrt(P * (1 - P) / N)
    z = np.abs(share - P)[un] / np.maximum(sig[un], 1e-12)
    assert z.max() <= 5, float(z.max())
    # the observed years are above or below for every replicate alike
    assert set(np.unique(r["below"][0][~un])) <= {0, N}
    _check_identities(r, 0, (10, 1), (5, 1))
    p_run = r["in_run"][0][0] / N
    print("\n[nplds 1e6] max |z| %.2f; device %.2f ms; mean P(below) %.3f, mean P(in a run >= 5) %.3f"
          % (z.max(), r["device_ms"], share[un].mean(), p_run[un].mean()))


def test_api_ensemble_equals_the_library_call_and_reports_years():
    st = PR._ensemble_station()
    P, B = api.reconstruction_batch([st], "boxcox", 1, np.random.default_rng(0))
    S = P[0]
    rng = np.random.default_rng(8)
    thetas = [api.vec_to_theta(SK.rand_theta(rng, s["p"], s["q"]), s["p"], s["q"]) for s in S["series"]]
    for t in thetas:
        t["R"] = 0.05
    n_reps, windows, lengths, period = 500, (3, 10), (2, 5), (1850, 1990)
    out = L.LDS_rep_posterior_yearly(thetas, st["Qa"], st["u"], st["v"], st["start_year"], transform="boxcox",
                                     num_reps=n_reps, seed=31, windows=windows, lengths=lengths, period=period)
    assert isinstance(out, list) and len(out) == 2
    stride = max(s["p"] + s["q"] + 6 for s in S["series"])
    rows = np.stack([np.pad(api.theta_to_vec(t), (0, stride - api.theta_to_vec(t).size)) for t in thetas])
    y0 = int(S["years"][0])
    lo, hi = period[0] - y0, period[1] - y0 + 1
    thr = float(np.mean(st["Qa"]["Qa"]))
    ref = _lib.posterior_yearly_batch(B["series"], [0, 1], None, [0, 1], rows, n_reps, seed=31, mu=[S["mu"]] * 2,
                                      transform="boxcox", lams=[S["lam"]] * 2, windows=windows, lengths=lengths,
                                      threshold=[thr] * 2, ranges=[(lo, hi)] * 2)
    for k in range(2):
        o = out[k]
        assert o["threshold"] == thr and o["period"] == period and o["windows"] == windows
        assert o["lengths"] == lengths
        assert np.array_equal(o["year"], np.arange(period[0], period[1] + 1))
        assert np.array_equal(o["below"], ref["below"][k][lo:hi])
        assert np.array_equal(o["in_run"], ref["in_run"][k][:, lo:hi])
        assert np.array_equal(o["wbelow"], ref["wbelow"][k][:, lo:hi])
        assert np.array_equal(o["n_nonfinite"], ref["nonfinite"][k][lo:hi])
        assert np.array_equal(o["p_below"], ref["below"][k][lo:hi] / n_reps)
        assert o["p_run"].shape == (2, hi - lo) and o["p_window"].shape == (2, hi - lo)
        assert np.isnan(o["p_window"][1][-9:]).all() and np.isfinite(o["p_window"][1][:-9]).all()
    # the same draws as LDS_rep_posterior: its simQ gives these counts
    reps = L.LDS_rep_posterior(thetas, st["Qa"], st["u"], st["v"], st["start_year"], transform="boxcox",
                               num_reps=n_reps, seed=31)
    for k in range(2):
        Q = reps[k]["simQ"].reshape(n_reps, S["years"].size)
        PY.assert_match(_per_fit(ref, k), Q, thr, windows, lengths, lo, hi, where=k)
