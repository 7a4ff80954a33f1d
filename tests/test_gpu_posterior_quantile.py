"""Per-step quantiles of w-step mean flows over conditioned replicates (ldsr_posterior_quantile_batch,
api.LDS_rep_posterior_quantiles) on the GPU:
  * the same seed gives, bit for bit, the quantiles of ldsr_posterior_rep_batch's simQ (the CPU reference,
    tests/posterior_quantile_oracle.py, applied to it) at four input widths, over fits of T = 2 .. 213 in one launch
    with the six hold-out kinds, per-fit ranges, every transform and Box-Cox flows that are not finite; also with
    caller noise, with a few thousand replicates (a histogram pass of the default bins), and on a long synthetic
    series (T = 20 000);
  * identities: quantiles do not decrease with the level, levels 0 and 1 are the minimum and maximum, w = 1 at observed
    steps is the observed flow;
  * LDSR_QUANT_TINY=1 (4 bins, collect cap 3) in a child process gives the same bits in more passes;
  * determinism, independence of the other fits and of the outputs asked for;
  * NPlds at 10^6 replicates: at every unobserved year the w = 1 quantile at level p is the smoother's marginal
    quantile within 5 binomial sigma;
  * the Python API.
Run with -s to see the passes and device times."""
import json
import math
import os
import subprocess
import sys

import numpy as np
import pytest

import ldsr_b200 as L
from ldsr_b200 import _lib, api
from tests import posterior_quantile_oracle as PQO
from tests import test_gpu_posterior_rep as PR
from tests import test_gpu_step_kernels as SK

pytestmark = pytest.mark.gpu

CASES = [(3, 3, "vu"), (10, 10, "sep"), (1, 3, "unone"), (24, 24, "vu")]
TRANSFORMS = (("log", 0.0, 0.0), ("none", 0.0, 0.0), ("boxcox", 0.3, 4.0), ("boxcox", 0.3, -3.5))
SPECS = (((1, 16, 17, 64), (0.0, 0.05, 0.5, 0.95, 1.0)), ((15, 2), (0.25, 0.75)), ((64,), (0.0, 1.0)),
         ((1, 5, 10, 30), (0.01, 0.1, 0.2, 0.3, 0.5, 0.7, 0.9, 0.99)))
REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ranges(rng, Ts):
    """Per fit: the whole series, or a range starting and ending inside tiles."""
    ranges = []
    for T in Ts:
        lo = 0 if T < 4 or rng.random() < 0.4 else int(rng.integers(0, T // 2))
        hi = T if rng.random() < 0.5 else int(rng.integers(lo + 1, T + 1))
        ranges.append((lo, hi))
    return np.array(ranges, dtype=np.int32)


def _per_fit(r, f):
    return {k: r[k][f] for k in _lib.QUANT_OUTPUTS if k in r}


def _check_identities(r, f, levels, ref):
    q = r["q"][f]
    d = np.diff(q, axis=1)
    assert (d[np.isfinite(d)] >= 0).all()
    for l, p in enumerate(levels):
        if p == 0.0:
            assert np.array_equal(q[:, l], ref["q"][:, l], equal_nan=True)
        if p == 1.0:
            assert np.array_equal(q[:, l], ref["q"][:, l], equal_nan=True)


def _check_case(c, n_reps, windows, levels, ranges, **kw):
    nf = c["fit_group"].size
    Q = PR.call(c, n_reps, want=("simQ",), **kw)["simQ"]
    g = _lib.posterior_quantile_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], n_reps,
                                      windows=windows, levels=levels, ranges=ranges, **kw)
    for f in range(nf):
        ref = PQO.assert_match(_per_fit(g, f), Q[f], windows, levels, *ranges[f], where=f)
        _check_identities(g, f, levels, ref)
    return g, Q


@pytest.mark.parametrize("width", CASES, ids=SK.case_id)
def test_same_seed_gives_the_quantiles_of_the_trajectory_call(width):
    i = CASES.index(width)
    c = PR.make_case(*width, seed=970 + i)
    nf = c["fit_group"].size
    rng = np.random.default_rng(i)
    tr, lam, dmu = TRANSFORMS[i]
    kw = dict(seed=75 + i, mu=rng.uniform(0.5, 1.5, nf) + dmu, transform=tr, lams=np.full(nf, lam))
    n_reps = (45, 70, 33, 100)[i]
    windows, levels = SPECS[i]
    g, Q = _check_case(c, n_reps, windows, levels, _ranges(rng, PR.fit_T(c)), **kw)
    n_bad = sum(int(x[x > 0].sum()) for x in g["nonfinite"])
    if tr == "boxcox" and dmu < 0:
        assert n_bad > 0  # the case meant to produce non-finite flows did
    print("\n[quantile] %s: %d passes, %d windows without a value, %.2f ms" % (SK.case_id(width), g["passes"], n_bad,
                                                                               g["device_ms"]))


def test_thousands_of_replicates_take_a_histogram_pass():
    c = PR.make_case(3, 3, "vu", seed=977)
    nf = c["fit_group"].size
    rng = np.random.default_rng(17)
    kw = dict(seed=5, mu=rng.uniform(0.5, 1.5, nf), transform="log")
    g, _ = _check_case(c, 5000, (1, 7, 64), (0.0, 0.05, 0.5, 0.95, 1.0), _ranges(rng, PR.fit_T(c)), **kw)
    assert g["passes"] >= 3, g["passes"]  # range, at least one histogram, collect


def test_caller_noise_gives_the_quantiles_of_the_trajectory_call():
    c = PR.make_case(3, 3, "vu", seed=43)
    nf = c["fit_group"].size
    Ts = PR.fit_T(c)
    rng = np.random.default_rng(6)
    n_reps = 37
    z = rng.standard_normal(2 * n_reps * Ts.sum())
    _check_case(c, n_reps, (1, 4, 16, 33), (0.1, 0.5, 0.9), _ranges(rng, Ts), z=z, mu=rng.uniform(0.5, 1.5, nf),
                transform="log")


def test_a_long_series():
    """One synthetic series of 20 000 steps, three fits (whole series, a range off the tiles, a short range), 300
    replicates."""
    rng = np.random.default_rng(13)
    T = 20000
    s = SK.make_series(rng, 3, 3, "vu", T)
    theta = np.stack([SK.rand_theta(rng, 3, 3) for _ in range(3)])
    n_reps = 300
    kw = dict(seed=98, mu=[0.7, 0.9, 1.1], transform="log")
    Q = _lib.posterior_rep_batch([s], [0], None, [0, 0, 0], theta, n_reps, want=("simQ",), **kw)["simQ"]
    ranges = np.array([(0, T), (7, T - 9), (19990, 19997)], dtype=np.int32)
    windows, levels = (64, 10, 1), (0.0, 0.05, 0.5, 0.95, 1.0)
    g = _lib.posterior_quantile_batch([s], [0], None, [0, 0, 0], theta, n_reps, windows=windows, levels=levels,
                                      ranges=ranges, **kw)
    for f in range(3):
        ref = PQO.assert_match(_per_fit(g, f), Q[f], windows, levels, *ranges[f], where=f)
        _check_identities(g, f, levels, ref)


def test_observed_steps_give_the_observed_flow():
    c = PR.make_case(10, 10, "sep", seed=971)
    nf = c["fit_group"].size
    kw = dict(seed=3, mu=np.full(nf, 0.8), transform="log")
    Q = PR.call(c, 200, want=("simQ",), **kw)["simQ"]
    g = _lib.posterior_quantile_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], 200,
                                      windows=(1,), levels=(0.0, 0.5, 1.0), **kw)
    n_obs = 0
    for f in range(nf):
        obs = (Q[f] == Q[f][0]).all(axis=0)  # every replicate takes the observation there
        n_obs += int(obs.sum())
        for l in range(3):  # the running sum (S + Q_t) - Q_{t+1} gives it back to rounding
            assert np.allclose(g["q"][f][0, l, obs], Q[f][0, obs], rtol=1e-12, atol=0)
    assert n_obs > 0


def test_forced_passes_give_the_same_bits():
    """LDSR_QUANT_TINY=1 (4 bins, collect cap 3) is read once per process: run in a child."""
    c = PR.make_case(3, 3, "vu", seed=978)
    nf = c["fit_group"].size
    args = dict(seed=11, mu=[0.6] * nf, transform="log", windows=(1, 10), levels=(0.0, 0.05, 0.5, 0.95, 1.0))
    a = _lib.posterior_quantile_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], 300,
                                      **args)
    code = ("import json, sys, numpy as np\n"
            "from ldsr_b200 import _lib\n"
            "from tests import test_gpu_posterior_rep as PR\n"
            "c = PR.make_case(3, 3, 'vu', seed=978)\n"
            "args = json.loads(sys.argv[1])\n"
            "r = _lib.posterior_quantile_batch(c['series'], c['group_series'], c['held'], c['fit_group'], c['theta'],"
            " 300, **args)\n"
            "np.savez(sys.argv[2], passes=r['passes'], **{'q%d' % f: r['q'][f] for f in range(len(r['q']))},"
            " **{'n%d' % f: r['nonfinite'][f] for f in range(len(r['q']))})\n")
    out = os.path.join(os.environ.get("TMPDIR", "/tmp"), "ldsr_quant_tiny_%d.npz" % os.getpid())
    env = dict(os.environ, LDSR_QUANT_TINY="1")
    subprocess.run([sys.executable, "-c", code, json.dumps(args), out], check=True, cwd=REPO, env=env)
    b = np.load(out)
    os.remove(out)
    for f in range(nf):
        assert np.array_equal(b["q%d" % f], a["q"][f], equal_nan=True), f
        assert np.array_equal(b["n%d" % f], a["nonfinite"][f]), f
    assert int(b["passes"]) > a["passes"], (int(b["passes"]), a["passes"])
    print("\n[quantile] passes: %d default, %d with 4 bins and cap 3" % (a["passes"], int(b["passes"])))


def test_determinism_and_independence_of_the_batch_and_of_the_outputs():
    c = PR.make_case(3, 3, "vu", 5)
    nf = c["fit_group"].size
    kw = dict(seed=123, mu=0.4, transform="log", windows=(2, 10), levels=(0.05, 0.5, 0.95))
    call = lambda cc, n, **k: _lib.posterior_quantile_batch(cc["series"], cc["group_series"], cc["held"],
                                                            cc["fit_group"], cc["theta"], n, **dict(kw, **k))
    a, b = call(c, 3000), call(c, 3000)
    for k in _lib.QUANT_OUTPUTS:
        for f in range(nf):
            assert np.array_equal(a[k][f], b[k][f], equal_nan=True), k
    # a fit added after the others leaves their quantiles alone
    c2 = dict(c, fit_group=np.append(c["fit_group"], c["fit_group"][-1]), theta=np.vstack([c["theta"], c["theta"][0]]))
    e = call(c2, 3000)
    for k in _lib.QUANT_OUTPUTS:
        for f in range(nf):
            assert np.array_equal(e[k][f], a[k][f], equal_nan=True), k
    # each output alone is the same as with the other
    for k in _lib.QUANT_OUTPUTS:
        one = call(c, 3000, want=(k,))
        assert set(one) == {k, "passes", "device_ms"}
        for f in range(nf):
            assert np.array_equal(one[k][f], a[k][f], equal_nan=True), k


def test_nplds_million_replicates_match_the_smoothers_marginals():
    """NPlds theta, 10^6 replicates of T = 813, w = 1, log transform: at each of the 767 unobserved years and level p,
    Phi((log q_p - mu - Y_t) / sqrt(C^2 V_t + R)) is p within 5 binomial sigma, Y_t and V_t from smoother_batch."""
    g, y, u, mu, th = PR._nplds()
    N, levels = 1000000, (0.05, 0.25, 0.5, 0.75, 0.95)
    r = _lib.posterior_quantile_batch([dict(y=y, u=u, v=u)], [0], None, [0], th[None, :], N, seed=2027, mu=[mu],
                                      transform="log", windows=(1, 10), levels=levels)
    sm = _lib.smoother_batch([dict(y=y, u=u, v=u)], [0], None, [0], th[None, :])
    p, q = 3, 3
    C, R = th[1 + p], th[3 + p + q]
    Y, V = np.asarray(sm["Y"][0]), np.asarray(sm["V"][0])
    un = np.isnan(y)
    assert un.sum() == 767
    erf = np.vectorize(math.erf)
    zmax = 0.0
    for l, pl in enumerate(levels):
        P = 0.5 * (1 + erf((np.log(r["q"][0][0, l]) - mu - Y) / np.sqrt(C * C * V + R) / math.sqrt(2)))
        sig = math.sqrt(pl * (1 - pl) / N)
        zl = np.abs(P - pl)[un] / sig
        zmax = max(zmax, float(zl.max()))
    assert zmax <= 5, zmax
    assert (r["nonfinite"][0][0] == 0).all()
    d = np.diff(r["q"][0], axis=1)
    assert (d[np.isfinite(d)] >= 0).all()
    print("\n[nplds 1e6] max |z| %.2f; %d passes; device %.2f ms" % (zmax, r["passes"], r["device_ms"]))


def test_api_ensemble_equals_the_library_call_and_reports_years():
    st = PR._ensemble_station()
    P, B = api.reconstruction_batch([st], "boxcox", 1, np.random.default_rng(0))
    S = P[0]
    rng = np.random.default_rng(9)
    thetas = [api.vec_to_theta(SK.rand_theta(rng, s["p"], s["q"]), s["p"], s["q"]) for s in S["series"]]
    for t in thetas:
        t["R"] = 0.05
    n_reps, windows, levels, period = 500, (1, 10), (0.05, 0.5, 0.95), (1850, 1990)
    out = L.LDS_rep_posterior_quantiles(thetas, st["Qa"], st["u"], st["v"], st["start_year"], transform="boxcox",
                                        num_reps=n_reps, seed=31, windows=windows, levels=levels, period=period)
    assert isinstance(out, list) and len(out) == 2
    stride = max(s["p"] + s["q"] + 6 for s in S["series"])
    rows = np.stack([np.pad(api.theta_to_vec(t), (0, stride - api.theta_to_vec(t).size)) for t in thetas])
    y0 = int(S["years"][0])
    lo, hi = period[0] - y0, period[1] - y0 + 1
    ref = _lib.posterior_quantile_batch(B["series"], [0, 1], None, [0, 1], rows, n_reps, seed=31, mu=[S["mu"]] * 2,
                                        transform="boxcox", lams=[S["lam"]] * 2, windows=windows, levels=levels,
                                        ranges=[(lo, hi)] * 2)
    for k in range(2):
        o = out[k]
        assert o["period"] == period and o["windows"] == windows and o["levels"] == levels
        assert np.array_equal(o["year"], np.arange(period[0], period[1] + 1))
        assert o["q"].shape == (2, 3, hi - lo)
        assert np.array_equal(o["q"], ref["q"][k][..., lo:hi], equal_nan=True)
        assert np.array_equal(o["n_nonfinite"], ref["nonfinite"][k][:, lo:hi])
        assert np.isnan(o["q"][1][:, -9:]).all() and (o["n_nonfinite"][1][-9:] == -1).all()
    # the same draws as LDS_rep_posterior: its simQ gives these quantiles
    reps = L.LDS_rep_posterior(thetas, st["Qa"], st["u"], st["v"], st["start_year"], transform="boxcox",
                               num_reps=n_reps, seed=31)
    for k in range(2):
        Q = reps[k]["simQ"].reshape(n_reps, S["years"].size)
        PQO.assert_match(_per_fit(ref, k), Q, windows, levels, lo, hi, where=k)
