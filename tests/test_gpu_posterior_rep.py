"""Replicates conditioned on the observed record (ldsr_posterior_rep_batch, api.LDS_rep_posterior) on the GPU:
  * caller noise: the CPU reference (tests/posterior_oracle.py), replicate by replicate, at every compiled input
    width (the 18 (p, q) cases of test_gpu_step_kernels.py), with the row bars of one E-step;
  * zero noise: simX is smoother_batch's X and simY its Y at unobserved steps;
  * the device generator: the stored NPlds reconstruction's bands and mean, and the smoother's second moments;
  * determinism (replicates keyed by (seed, fit, replicate)), the chunked output pipeline, and the Python API.
Run with -s to see the largest deviation from the reference per width."""
import os
import subprocess
import sys

import numpy as np
import pytest

import ldsr_b200 as L
from ldsr_b200 import _lib, api
from oracle import oracle as O
from tests import data
from tests import posterior_oracle as PO
from tests import test_gpu_step_kernels as SK

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRANSFORMS = (("log", 0.0), ("none", 0.0), ("boxcox", 0.3))
WANTS = (("simX", "simY", "simQ"), ("simQ",), ("simX", "simY"), ("simY", "simQ"))
N_REPS = (1, 33, 5, 70, 32, 17)


def make_case(p, q, form, seed):
    """Series of 2, 3, 15, 16, 17, 31, 32, 33, 65 and 213 steps (about the 16-step tile and the 32-step mask word),
    groups out of series order with the six hold-out kinds, two or three fits per group."""
    rng = np.random.default_rng(seed)
    Ts = (2, 3, 15, 16, 17, 31, 32, 33, 65, 213)
    series = [SK.make_series(rng, p, q, form, T) for T in Ts]
    pairs = []
    for s, T in enumerate(Ts):
        kinds = SK.HOLD_KINDS if T >= 65 else [SK.HOLD_KINDS[(s + k) % len(SK.HOLD_KINDS)] for k in range(2)]
        pairs += [(s, k) for k in kinds]
    rng.shuffle(pairs)
    group_series = np.array([s for s, _ in pairs], dtype=np.int32)
    held = [SK.holdout(rng, series[s]["y"], k) for s, k in pairs]
    fit_group = np.repeat(np.arange(len(pairs)), [2 + g % 2 for g in range(len(pairs))])
    theta = np.stack([SK.rand_theta(rng, p, q) for _ in fit_group])
    return dict(series=series, group_series=group_series, held=held, fit_group=fit_group, theta=theta)


def call(c, n_reps, **kw):
    return _lib.posterior_rep_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], n_reps, **kw)


def fit_T(c):
    return np.array([c["series"][c["group_series"][g]]["y"].size for g in c["fit_group"]])


@pytest.mark.parametrize("width", SK.WIDTHS, ids=SK.case_id)
def test_caller_noise_matches_the_oracle_at_every_width(width):
    p, q, form = width
    i = SK.WIDTHS.index(width)
    c = make_case(p, q, form, 700 + i)
    nf = c["fit_group"].size
    n_reps = N_REPS[i % len(N_REPS)]
    tr, lam = TRANSFORMS[i % len(TRANSFORMS)]
    want = WANTS[i % len(WANTS)]
    rng = np.random.default_rng(i)
    mu = rng.uniform(0.5, 1.5, nf) + (4.0 if tr == "boxcox" else 0.0)  # Box-Cox: (y + mu) lam + 1 > 0
    lams = np.full(nf, lam)
    Ts = fit_T(c)
    z = rng.standard_normal(2 * n_reps * Ts.sum())
    g = call(c, n_reps, z=z, mu=mu, transform=tr, lams=lams, want=want)
    off = 2 * n_reps * np.concatenate([[0], np.cumsum(Ts)])
    dev = dict.fromkeys(want, 0.0)
    for f in range(nf):
        s, y = SK.group_y(c, c["fit_group"][f])
        T = Ts[f]
        obs = np.isfinite(y)
        zf = z[off[f]:off[f + 1]].reshape(n_reps, 2 * T)
        o = PO.posterior_rep(c["theta"][f], y, s["u"], s["v"], zf, mu=mu[f], transform=tr, lam=lam, p=p, q=q)
        for r in range(n_reps):
            for k in want:
                d = SK.row_dev(g[k][f][r], o[k][r]) if k != "simQ" else SK.rel_dev(g[k][f][r], o[k][r])
                dev[k] = max(dev[k], d)
                assert d < SK.ROW_RTOL, (f, r, k, d)
            if "simY" in want:
                assert np.array_equal(g["simY"][f][r][obs], y[obs]), (f, r)
    SK.report("posterior_rep", width, dev)


@pytest.mark.parametrize("width", [(3, 3, "vu"), (10, 10, "sep"), (1, 3, "unone"), (24, 24, "vu")], ids=SK.case_id)
def test_zero_noise_is_the_smoother(width):
    c = make_case(*width, seed=71)
    Ts = fit_T(c)
    n_reps = 2
    g = call(c, n_reps, z=np.zeros(2 * n_reps * Ts.sum()), transform="none", want=("simX", "simY"))
    sm = _lib.smoother_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"])
    for f in range(Ts.size):
        _, y = SK.group_y(c, c["fit_group"][f])
        un = np.isnan(y)
        for r in range(n_reps):
            assert SK.row_dev(g["simX"][f][r], sm["X"][f]) < SK.ROW_RTOL, f
            if un.any():
                assert SK.row_dev(g["simY"][f][r][un], sm["Y"][f][un]) < SK.ROW_RTOL, f


def _nplds():
    g = data.load("nplds.json")
    y, u, mu, inst = data.np_case(1, 1200)
    return g, y, u, mu, data.theta_of(g["theta"])


def test_replicates_reproduce_the_stored_reconstruction():
    """NPlds theta, 32 768 replicates of T = 813 from the device generator: at each of the 767 unobserved years the
    share of replicates below the stored Ql (above Qu) is 0.05 within 5 sigma of a binomial proportion, the mean of
    simX is within 5 sqrt(V_t / N) of the stored X, and the 46 observed years reproduce Qa."""
    g, y, u, mu, th = _nplds()
    N = 32768
    r = _lib.posterior_rep_batch([dict(y=y, u=u, v=u)], [0], None, [0], th[None, :], N, seed=2024, mu=[mu],
                                 transform="log")
    simQ, simX = r["simQ"][0], r["simX"][0]
    un = np.isnan(y)
    assert un.sum() == 767
    Ql, Qu, X = (np.array(g["rec"][k]) for k in ("Ql", "Qu", "X"))
    lo, hi = 0.05 - 5 * np.sqrt(0.05 * 0.95 / N), 0.05 + 5 * np.sqrt(0.05 * 0.95 / N)
    below = np.mean(simQ < Ql, axis=0)[un]
    above = np.mean(simQ > Qu, axis=0)[un]
    assert lo <= below.min() and below.max() <= hi, (below.min(), below.max())
    assert lo <= above.min() and above.max() <= hi, (above.min(), above.max())
    V = O.kalman_smoother(y, u, u, th)["V"]
    assert np.all(np.abs(simX.mean(axis=0) - X) <= 5 * np.sqrt(V / N))
    qa = np.array(data.load("np.json")["NPannual"]["Qa"])
    assert np.max(np.abs(simQ[:, ~un] - qa) / qa) < 1e-12
    print("\n[bands] share below Ql %.4f..%.4f, above Qu %.4f..%.4f" % (below.min(), below.max(), above.min(),
                                                                        above.max()))


@pytest.mark.parametrize("width", [(3, 3, "vu"), (10, 10, "sep")], ids=SK.case_id)
def test_second_moments_are_the_smoothers(width):
    """Per step, the replicates' variance is V_t within 5 sqrt(2 / N) relative and their lag-1 covariance is the
    smoother's cross-covariance J_t V_{t+1} within 5 standard errors."""
    p, q, form = width
    rng = np.random.default_rng(p)
    s = SK.make_series(rng, p, q, form, 213)
    held = SK.holdout(rng, s["y"], "scattered")
    th = SK.rand_theta(rng, p, q)
    N = 32768
    x = _lib.posterior_rep_batch([s], [0], [held], [0], th[None, :], N, seed=9, want=("simX",))["simX"][0]
    y = np.array(s["y"])
    y[held] = np.nan
    sm = O.kalman_smoother(y, s["u"], s["v"], th, p=p, q=q)
    V, J = sm["V"], sm["J"]
    xc = x - x.mean(axis=0)
    var = np.mean(xc * xc, axis=0)
    assert np.all(np.abs(var / V - 1) <= 5 * np.sqrt(2.0 / N))
    cov = np.mean(xc[:, :-1] * xc[:, 1:], axis=0)
    c0 = J[:-1] * V[1:]
    se = np.sqrt((V[:-1] * V[1:] + c0 * c0) / N)
    assert np.all(np.abs(cov - c0) <= 5 * se)


def test_determinism_and_independence_of_the_batch():
    c = make_case(3, 3, "vu", 5)
    kw = dict(seed=123, mu=0.4, transform="log")
    a = call(c, 40, **kw)
    b = call(c, 40, **kw)
    big = call(c, 1000, **kw)
    for k in ("simX", "simY", "simQ"):
        for f in range(len(a[k])):
            assert np.array_equal(a[k][f], b[k][f]), k
            assert np.array_equal(big[k][f][:40], a[k][f]), k
    # a fit added after the others leaves their rows alone
    c2 = dict(c, fit_group=np.append(c["fit_group"], c["fit_group"][-1]),
              theta=np.vstack([c["theta"], c["theta"][0]]))
    e = call(c2, 40, **kw)
    for f in range(c["fit_group"].size):
        assert np.array_equal(e["simQ"][f], a["simQ"][f])
    # one persistent context, two seeds: each equal to the same call on a fresh context
    ctx = _lib.Ctx(n_devices=1)
    try:
        for seed in (1, 2):
            r1 = call(c, 50, seed=seed, ctx=ctx)
            r2 = call(c, 50, seed=seed)
            assert all(np.array_equal(r1["simX"][f], r2["simX"][f]) for f in range(len(r1["simX"])))
        g, y, u, mu, th = _nplds()
        for r_seed in (3, 4):
            r1 = _lib.rep_batch(th, u, u, y.size, 300, mu=mu, r_seed=r_seed, ctx=ctx.h)
            r2 = _lib.rep_batch(th, u, u, y.size, 300, mu=mu, r_seed=r_seed)
            assert np.array_equal(r1["simQ"], r2["simQ"]), r_seed
    finally:
        ctx.close()


def test_chunked_pipeline_equals_the_single_kernel_path(tmp_path):
    """Three fits of T = 813 (one with a held-out decade) and 4000 replicates: about 9.8 M values per output, so
    the chunked path (forced through LDSR_REP_CHUNKED in a child process) cuts them into two launches of whole
    (fit, 32 replicates) blocks.  Device generator and caller noise."""
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from ldsr_b200 import _lib; from tests import data\n"
            "g = data.load('nplds.json'); th = data.theta_of(g['theta']); y, u, mu, inst = data.np_case(1, 1200)\n"
            "ser = [dict(y=y, u=u, v=u)]; thetas = np.stack([th, th * 0.98, th]); n = 4000\n"
            "kw = dict(seed=77)\n"
            "if sys.argv[2] == 'z': kw = dict(z=np.random.default_rng(3).standard_normal(2 * n * 3 * y.size))\n"
            "r = _lib.posterior_rep_batch(ser, [0, 0], [[], inst[10:20]], [0, 0, 1], thetas, n, mu=[mu] * 3, **kw)\n"
            "np.save(sys.argv[1], np.stack([np.stack(r[k]) for k in ('simX', 'simY', 'simQ')]))\n") % ROOT
    for case in ("seed", "z"):
        outs = []
        for k, env in enumerate(({}, {"LDSR_REP_CHUNKED": "1"})):
            f = str(tmp_path / ("post_%s%d.npy" % (case, k)))
            subprocess.run([sys.executable, "-c", code, f, case], check=True, env=dict(os.environ, **env), timeout=300)
            outs.append(np.load(f))
        assert np.isfinite(outs[0]).all() and np.array_equal(outs[0], outs[1]), case


def _ensemble_station():
    d = data.load("np.json")
    years, qa = np.array(d["NPannual"]["year"]), np.array(d["NPannual"]["Qa"])
    pc = np.array([d["NPpc"][k] for k in ("PC1", "PC9", "PC13")])
    return dict(Qa=dict(year=years, Qa=qa), u=[pc[:, 600:], None], v=[pc[:, 600:], pc[:2, 600:]], start_year=1800)


def test_api_ensemble_equals_the_library_call_and_conditions_on_the_fitted_y():
    st = _ensemble_station()
    P, B = api.reconstruction_batch([st], "boxcox", 1, np.random.default_rng(0))
    S = P[0]
    rng = np.random.default_rng(8)
    thetas = [api.vec_to_theta(SK.rand_theta(rng, s["p"], s["q"]), s["p"], s["q"]) for s in S["series"]]
    for t in thetas:
        t["R"] = 0.05
    n_reps = 7
    out = L.LDS_rep_posterior(thetas, st["Qa"], st["u"], st["v"], st["start_year"], transform="boxcox",
                              num_reps=n_reps, seed=31)
    assert isinstance(out, list) and len(out) == 2
    stride = max(s["p"] + s["q"] + 6 for s in S["series"])
    rows = np.stack([np.pad(api.theta_to_vec(t), (0, stride - api.theta_to_vec(t).size)) for t in thetas])
    ref = _lib.posterior_rep_batch(B["series"], [0, 1], None, [0, 1], rows, n_reps, seed=31, mu=[S["mu"]] * 2,
                                   transform="boxcox", lams=[S["lam"]] * 2)
    N = S["years"].size
    for k in range(2):
        o = out[k]
        assert np.array_equal(o["year"], np.tile(S["years"], n_reps))
        assert np.array_equal(o["rep"], np.repeat(np.arange(1, n_reps + 1), N))
        for name in ("simX", "simY", "simQ"):
            assert np.array_equal(o[name], ref[name][k].ravel(), equal_nan=True), name
        # the y LDS_reconstruction fits on, bit for bit at its observed years; simQ there is its Qa
        y = B["series"][k]["y"]
        obs = np.isfinite(y)
        simY = o["simY"].reshape(n_reps, N)
        assert np.array_equal(simY[:, obs], np.broadcast_to(y[obs], (n_reps, obs.sum())))
        qa = np.asarray(st["Qa"]["Qa"], dtype=float)
        assert np.allclose(o["simQ"].reshape(n_reps, N)[:, obs], qa, rtol=1e-10, atol=0)
    single = L.LDS_rep_posterior(thetas[0], st["Qa"], st["u"][0], st["v"][0], st["start_year"], num_reps=3)
    assert single["simQ"].size == 3 * N and np.isfinite(single["simQ"]).all()
