"""GPU parity tests: the CUDA path (through the C ABI, via ldsr_b200.api / _lib) against the CPU
oracle and the reference's golden values.  Tolerances are BASELINE.json's: log-likelihood
relative 1e-9, theta and reconstructed flow relative 1e-6 at the same iteration count, identical
selected restart."""
import os

import numpy as np
import pytest

import ldsr_b200 as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
from ldsr_b200 import _lib
from oracle import oracle as O
from tests import data

pytestmark = pytest.mark.gpu

LIK_RTOL = 1e-9
THETA_RTOL = 1e-6


def rel(a, b):
    return abs(a - b) / abs(b)


def rand_theta0(rng, p, q, n):
    return np.stack([np.concatenate([[rng.uniform()], rng.uniform(-1, 1, p), [rng.uniform()],
                                     rng.uniform(-1, 1, q), [1, 1, 0, 1]]) for _ in range(n)])


def assert_theta_close(a, b, rtol=THETA_RTOL, floor=1e-8):
    a, b = np.asarray(a), np.asarray(b)
    assert np.array_equal(np.isnan(a), np.isnan(b))  # unused tail of a padded theta row stays NaN
    ok = ~np.isnan(b)
    scale = np.maximum(np.abs(b[ok]), floor)
    assert np.max(np.abs(a[ok] - b[ok]) / scale) < rtol, np.max(np.abs(a[ok] - b[ok]) / scale)


# ---- the reference's own known-answer tests, run on the GPU (tests/testthat/test-LDS-EM.R:21-41)
def test_kat_first_two_iterations_p1():
    y, u, th0, kat = data.p1_case()
    tol = kat["tolerance"]
    theta0 = L.vec_to_theta(th0, 7, 7)
    s1 = L.Kalman_smoother(y, u, u, theta0)
    th1 = L.Mstep(y, u, u, s1)
    s2 = L.Kalman_smoother(y, u, u, th1)
    th2 = L.Mstep(y, u, u, s2)
    assert rel(s1["lik"], kat["smooth1_lik"]) < tol
    assert rel(s1["X"][0], kat["smooth1_X_1_85"][0]) < tol
    assert rel(s1["X"][84], kat["smooth1_X_1_85"][1]) < tol
    for th, g in ((th1, kat["theta1"]), (th2, kat["theta2"])):
        assert rel(th["A"], g["A"]) < tol
        assert abs(th["C"] - g["C"]) < 1e-6
        assert rel(th["Q"], g["Q"]) < tol
    assert rel(s2["lik"], kat["smooth2_lik"]) < 5e-6
    # and against the oracle to full precision
    o1 = O.kalman_smoother(y, u, u, th0)
    assert rel(s1["lik"], o1["lik"]) < 1e-12
    for k in "XYVJ":
        assert np.allclose(s1[k], o1[k], rtol=1e-11, atol=1e-13), k
    assert_theta_close(L.theta_to_vec(th1), O.mstep(y, u, u, o1), 1e-10)


def test_kat_convergence_p1():
    y, u, th0, kat = data.p1_case()
    fit = L.LDS_EM(y, u, u, L.vec_to_theta(th0, 7, 7), kat["em"]["niter"], kat["em"]["tol"])
    assert len(fit["liks"]) == 68
    assert abs(fit["lik"] - kat["em"]["lik"]) < 1e-6
    o = O.em(y, u, u, th0, 100, 1e-5)
    assert np.allclose(fit["liks"], o["liks"], rtol=LIK_RTOL, atol=0)
    assert_theta_close(L.theta_to_vec(fit["theta"]), o["theta"])
    for k in "XYVJ":
        assert np.allclose(fit["fit"][k], o["fit"][k], rtol=1e-6, atol=1e-9), k


def test_nplds_fixture_estep():
    g = data.load("nplds.json")
    y, u, mu, inst = data.np_case(1, 1200)
    th = data.theta_of(g["theta"])
    s = L.Kalman_smoother(y, u, u, L.vec_to_theta(th, 3, 3))
    assert rel(s["lik"], g["lik"]) < LIK_RTOL
    assert np.max(np.abs(s["X"] - np.array(g["rec"]["X"]))) < 1e-11
    assert np.max(np.abs(np.exp(s["Y"] + mu) / np.array(g["rec"]["Q"]) - 1)) < 1e-11


# ---- batched EM against the oracle
def _np213():
    y, u, mu, inst = data.np_case(601, 1800)
    return y, u, mu, inst


def check_batch(series, group_series, held, fit_group, th0, niter, tol, **kw):
    g = em_variant(series, group_series, held, fit_group, th0, niter, tol, want_liks=True, **kw)
    o = O.em_batch(series, group_series, held, fit_group, th0, niter, tol)
    assert np.array_equal(g["status"], o["status"])
    assert np.array_equal(g["iters"], o["iters"]), np.nonzero(g["iters"] != o["iters"])
    assert np.allclose(g["lik"], o["lik"], rtol=LIK_RTOL, atol=0)
    assert_theta_close(g["theta"], o["theta"])
    assert np.array_equal(g["best"], o["best"])
    # trace: filled up to iters, NaN after
    for f in range(len(fit_group)):
        n = g["iters"][f]
        assert np.all(np.isfinite(g["liks"][f, :n])) and np.all(np.isnan(g["liks"][f, n:]))
        assert g["liks"][f, n - 1] == g["lik"][f]
    return g, o


# both EM kernels must agree with the oracle: 2 = lane-per-fit (em_kernel.cuh), 3 = time-split
# (em_split_kernel.cuh); 0 = whatever the plan picks
VARIANTS = [2, 3, 5]  # lane-per-fit, time-split, small-batch scan kernel (4 = wide-input kernel: wide tests)


def em_variant(*a, **kw):
    """_lib.em_batch; variants 4 / 5 exist for some widths, lengths and batch sizes only: skip where they do not."""
    try:
        return _lib.em_batch(*a, **kw)
    except _lib.LdsrError as e:
        if kw.get("variant") in (4, 5) and e.code == _lib.ERR_UNSUPPORTED:
            pytest.skip("kernel variant %d does not cover this case" % kw["variant"])
        raise


@pytest.mark.parametrize("variant", VARIANTS)
def test_em_batch_folds_restarts_np213(variant):
    y, u, mu, inst = _np213()
    rng = np.random.default_rng(11)
    n_folds, n_rest = 6, 20
    held = [np.sort(rng.choice(inst, 11, replace=False)) for _ in range(n_folds)]
    fg = np.repeat(np.arange(n_folds), n_rest)
    th0 = rand_theta0(rng, 3, 3, n_folds * n_rest)
    ser = [dict(y=y, u=u, v=u)]
    g, o = check_batch(ser, np.zeros(n_folds, dtype=int), held, fg, th0, 300, 1e-5, variant=variant)
    # winners' smoothed trajectories == oracle E-step with the winner's theta on the fold's y
    for k in range(n_folds):
        b = g["best"][k]
        yy = y.copy()
        yy[held[k]] = np.nan
        s = O.kalman_smoother(yy, u, u, o["theta"][b])
        row = slice(g["traj_ptr"][k], g["traj_ptr"][k + 1])
        assert np.allclose(g["X"][row], s["X"], rtol=1e-6, atol=1e-9)
        assert np.allclose(np.exp(g["Y"][row] + mu), np.exp(s["Y"] + mu), rtol=THETA_RTOL)
        assert np.allclose(g["V"][row], s["V"], rtol=1e-6) and np.allclose(g["J"][row], s["J"], rtol=1e-6)


@pytest.mark.parametrize("variant", VARIANTS)
def test_chunking_does_not_change_results(variant):
    y, u, mu, inst = _np213()
    rng = np.random.default_rng(5)
    th0 = rand_theta0(rng, 3, 3, 40)
    ser = [dict(y=y, u=u, v=u)]
    a = em_variant(ser, [0], None, np.zeros(40, dtype=int), th0, 150, 1e-5, chunk_iters=100, variant=variant)
    b = em_variant(ser, [0], None, np.zeros(40, dtype=int), th0, 150, 1e-5, chunk_iters=7, variant=variant)
    for k in ("theta", "lik", "iters", "best", "X", "Y", "V", "J"):
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("variant", VARIANTS)
def test_sentinels_unequal_dims_and_ensemble(variant):
    # test-LDS-EM.R:58-77, test-ensemble.R:9-18: u=NULL, v=NULL, nrow(u)!=nrow(v), list of u/v
    y, u, mu, inst = _np213()
    rng = np.random.default_rng(3)
    series = [dict(y=y, u=None, v=u, p=1, q=3), dict(y=y, u=u, v=None, p=3, q=1),
              dict(y=y, u=u[:2], v=u), dict(y=y, u=u, v=u)]
    stride = 12
    th0, fg = [], []
    for s_i, (p, q) in enumerate([(1, 3), (3, 1), (2, 3), (3, 3)]):
        for t in rand_theta0(rng, p, q, 5):
            th0.append(np.pad(t, (0, stride - t.size)))
            fg.append(s_i)
    held = [inst[:5], inst[5:9], np.array([], dtype=int), inst[-3:]]
    g, o = check_batch(series, [0, 1, 2, 3], held, fg, np.stack(th0), 120, 1e-5, variant=variant)
    assert np.all(g["theta"][0:5, 1] == 0)      # B == 0 without u
    assert np.all(g["theta"][5:10, 5] == 0)     # D == 0 without v


@pytest.mark.parametrize("variant", VARIANTS)
def test_fully_observed_p1_batch(variant):
    # every step observed (the reference's golden series, p=q=7): no unobserved word anywhere, so the
    # time-split kernel runs entirely on composed Moebius/affine maps of 8-step segments
    y, u, th0, kat = data.p1_case()
    rng = np.random.default_rng(21)
    th = np.vstack([th0[None], rand_theta0(rng, 7, 7, 37)])
    held = [np.array([], dtype=int), np.array([0, 1, 2, 40, 84])]
    fg = np.repeat([0, 1], 19)
    g, o = check_batch([dict(y=y, u=u, v=u)], [0, 0], held, fg, th, 100, 1e-5, variant=variant)
    assert g["iters"][0] == 68  # tests/testthat/test-LDS-EM.R:39


@pytest.mark.parametrize("variant", VARIANTS)
@pytest.mark.parametrize("T", [4, 5, 8, 9, 31, 32, 33, 40, 64, 65, 100, 257])
def test_ragged_lengths_and_scattered_observations(variant, T):
    # unit-table edge cases: T below / at / just above the 8-step segment and the 32-step word,
    # observations scattered so that U words and M segments interleave, first/last step missing
    rng = np.random.default_rng(100 + T)
    p, q = (1, 1) if T < 16 else (2, 3)  # a handful of steps cannot identify more inputs
    niter = 10 if T < 16 else 40
    u = rng.standard_normal((p, T))
    v = rng.standard_normal((q, T))
    x = np.zeros(T)
    for t in range(1, T):
        x[t] = 0.7 * x[t - 1] + 0.3 * u[0, t - 1] + 0.5 * rng.standard_normal()
    y = 0.8 * x + 0.2 * v[-1] + 0.3 * rng.standard_normal(T)
    ya = y.copy()  # sparse: bursts of observations separated by long gaps
    keep = np.zeros(T, dtype=bool)
    for s0 in range(3, T, 70):
        keep[s0:s0 + 9] = True
    keep[rng.integers(0, T, 2)] = True
    ya[~keep] = np.nan
    if np.isfinite(ya).sum() < 4:
        ya = y.copy()
    yb = y.copy()  # dense with random gaps; first and last step missing when long enough
    yb[rng.uniform(size=T) < 0.3] = np.nan
    if T > 8:
        yb[0] = yb[-1] = np.nan
    if np.isfinite(yb).sum() < 4:
        yb = y.copy()
    series = [dict(y=ya, u=u, v=v), dict(y=yb, u=u, v=v)]
    fg = np.repeat([0, 1], 5)
    th0 = rand_theta0(rng, p, q, 10)
    none = np.array([], dtype=int)
    check_batch(series, [0, 1], [none, none], fg, th0, niter, 1e-7, variant=variant)


@pytest.mark.parametrize("variant", VARIANTS + [0])
def test_cv_np413_sample(variant):
    # the bench workload in small: NP series T=413 (obs at steps 360..405), folds x restarts, 2 CTAs
    # of the time-split kernel with several groups per CTA (per-lane masks differ)
    y, u, mu, inst = data.np_case(401, 1600)
    assert y.size == 413
    rng = np.random.default_rng(413)
    n_folds, n_rest = 8, 6
    held = [np.sort(rng.choice(inst, 11, replace=False)) for _ in range(n_folds)]
    fg = np.repeat(np.arange(n_folds), n_rest)
    th0 = rand_theta0(rng, 3, 3, n_folds * n_rest)
    check_batch([dict(y=y, u=u, v=u)], np.zeros(n_folds, dtype=int), held, fg, th0, 400, 1e-5, variant=variant)


def test_long_series_np813_both_kernels_agree():
    y, u, mu, inst = data.np_case(1, 1200)
    rng = np.random.default_rng(813)
    th0 = rand_theta0(rng, 3, 3, 12)
    ser = [dict(y=y, u=u, v=u)]
    fg = np.zeros(12, dtype=int)
    check_batch(ser, [0], [np.array([], dtype=int)], fg, th0, 150, 1e-5, variant=3)
    a = _lib.em_batch(ser, [0], None, fg, th0, 150, 1e-5, variant=2)
    b = _lib.em_batch(ser, [0], None, fg, th0, 150, 1e-5, variant=3)
    assert np.array_equal(a["iters"], b["iters"]) and np.array_equal(a["best"], b["best"])
    assert np.allclose(a["lik"], b["lik"], rtol=LIK_RTOL, atol=0)


def test_api_restart_and_cv_shapes():
    d = data.load("np.json")
    Qa = dict(year=np.array(d["NPannual"]["year"]), Qa=np.array(d["NPannual"]["Qa"]))
    pc = np.array([d["NPpc"][k] for k in ("PC1", "PC9", "PC13")])[:, 600:]
    rng = np.random.default_rng(2)
    fit = L.LDS_reconstruction(Qa, pc, pc, start_year=1800, num_restarts=4, rng=rng, niter=200, return_raw=True)
    assert set(fit["rec"]) == {"year", "X", "Xl", "Xu", "Q", "Ql", "Qu"} and fit["rec"]["Q"].size == 213
    assert np.all(fit["rec"]["Ql"] < fit["rec"]["Q"]) and np.all(fit["rec"]["Q"] < fit["rec"]["Qu"])
    Z = L.make_Z(Qa["Qa"], 3, rng=rng)
    cv = L.cvLDS(Qa, pc, pc, start_year=1800, num_restarts=3, Z=Z, rng=rng, niter=200)
    assert cv["Ycv"].shape == (46, 3) and set(cv["metrics"]) == {"R2", "RE", "CE", "nRMSE", "KGE"}
    ens = L.LDS_reconstruction(Qa, [pc, pc[:2]], [pc, pc[:2]], start_year=1800, num_restarts=2, rng=rng, niter=100)
    assert len(ens["ensemble"]) == 2 and ens["rec"]["X"].size == 213
    cv2 = L.cvLDS(Qa, [pc, pc[:2]], [pc, pc[:2]], start_year=1800, num_restarts=2,
                  Z=L.make_Z(Qa["Qa"], 2, contiguous=False, rng=rng), rng=rng, niter=100)
    assert cv2["Ycv"].shape == (46, 2)
    for kw in (dict(u=None, v=pc), dict(u=pc, v=None), dict(u=pc[:2], v=pc)):
        f = L.LDS_reconstruction(Qa, kw["u"], kw["v"], start_year=1800, num_restarts=2, rng=rng, niter=100)
        assert np.isfinite(f["lik"])
    # test-LDS-EM.R:43-46 "Fixed restart works": init = make_init(nrow(u), nrow(v), 2), here drawn from R's
    # own stream (set.seed(5)) so that the run is the one a seeded R session would make; repeatable
    fa = L.LDS_reconstruction(Qa, pc, pc, start_year=1800, init=L.make_init(3, 3, 2, L.RRandom(5)), niter=150)
    fb = L.LDS_reconstruction(Qa, pc, pc, start_year=1800, init=L.make_init(3, 3, 2, L.RRandom(5)), niter=150)
    assert np.isfinite(fa["lik"]) and fa["lik"] == fb["lik"] and np.array_equal(fa["rec"]["Q"], fb["rec"]["Q"])


def test_propagate_and_rep_against_oracle():
    d = data.load("np.json")
    th = data.theta_of(d["theta"])
    y, u, mu, inst = data.np_case(1, 1200)
    g = L.propagate(L.vec_to_theta(th, 3, 3), u, u, y)
    o = O.propagate(th, u, u, y)
    assert rel(g["lik"], o["lik"]) < LIK_RTOL
    for k in "XYV":
        assert np.allclose(g[k], o[k], rtol=1e-12, atol=1e-14)
    rng = np.random.default_rng(9)
    n_reps, n = 7, 813
    z = rng.standard_normal((n_reps, 1 + 2 * n))
    r = L.LDS_rep(L.vec_to_theta(th, 3, 3), u, u, np.arange(1200, 2013), n_reps, mu=mu, z=z)
    for i in range(n_reps):
        oo = O.rep(th, u, u, n, z[i], mu=mu)
        sl = slice(i * n, (i + 1) * n)
        assert np.allclose(r["simX"][sl], oo["simX"], rtol=1e-10, atol=1e-12)
        assert np.allclose(r["simQ"][sl], oo["simQ"], rtol=1e-10)
    # device generator: right moments, reproducible, different per replicate
    r1 = L.LDS_rep(L.vec_to_theta(th, 3, 3), None, None, np.arange(2000), 2000, seed=1, exp_trans=False)
    r2 = L.LDS_rep(L.vec_to_theta(th, 3, 3), None, None, np.arange(2000), 2000, seed=1, exp_trans=False)
    assert np.array_equal(r1["simX"], r2["simX"])
    X = r1["simX"].reshape(2000, 2000)[:, 500:]
    a, q = th[0], th[8]
    assert abs(X.mean()) < 0.02 and rel(X.var(), q / (1 - a * a)) < 0.02


def test_singular_gram_block_is_flagged():
    y, u, mu, inst = _np213()
    uu = np.vstack([u[0], u[0], u[1]])  # duplicated row: Tuu singular -> arma::inv would throw
    th0 = rand_theta0(np.random.default_rng(0), 3, 3, 3)
    r = _lib.em_batch([dict(y=y, u=uu, v=u)], [0], None, [0, 0, 0], th0, 20, 1e-5)
    assert np.all(r["status"] == _lib.FIT_SINGULAR) and np.all(np.isnan(r["lik"])) and r["best"][0] == -1


def test_argument_errors():
    y, u, mu, inst = _np213()
    th0 = rand_theta0(np.random.default_rng(0), 3, 3, 2)
    with pytest.raises(_lib.LdsrError) as e:
        _lib.em_batch([dict(y=y, u=u, v=u)], [0], None, [0, 0], th0, 1, 1e-5)  # niter < 2
    assert e.value.code == _lib.ERR_ARG
    yy = y.copy()
    yy[170] = np.inf
    with pytest.raises(_lib.LdsrError):
        _lib.em_batch([dict(y=yy, u=u, v=u)], [0], None, [0, 0], th0, 10, 1e-5)
    with pytest.raises(_lib.LdsrError):
        _lib.em_batch([dict(y=y, u=u, v=u)], [0], [np.array([999])], [0, 0], th0, 10, 1e-5)


def test_poll_callback_interrupts():
    y, u, mu, inst = _np213()
    th0 = rand_theta0(np.random.default_rng(0), 3, 3, 8)
    calls = []
    with pytest.raises(_lib.LdsrError) as e:
        _lib.em_batch([dict(y=y, u=u, v=u)], [0], None, np.zeros(8, dtype=int), th0, 1000, 0.0, chunk_iters=10,
                      poll=lambda: calls.append(1) or len(calls) >= 3)
    assert e.value.code == _lib.ERR_INTERRUPTED and len(calls) == 3


def test_cv_metrics_kernel_matches_the_stored_cvLDS_result():
    # R/sysdata.rda::NPcv: Ycv, Z, target -> metrics.dist (30 folds x 5), the reference's own numbers
    g = data.load("npcv.json")
    n = len(g["target"]["y"])
    Y = np.array(g["Ycv"]["Y"]).reshape(-1, n)
    obs = np.array(g["target"]["y"])
    m = _lib.cv_metrics(Y, obs, g["Z"])
    for j, name in enumerate(_lib.METRIC_NAMES):
        assert np.allclose(m[:, j], np.array(g["metrics_dist"][name]), rtol=1e-10, atol=1e-12), name
    assert np.allclose(_lib.cv_metrics(np.log(Y), obs, g["Z"], exp_trans=True), m, rtol=1e-12)
    # against the oracle on ragged folds, NaN in obs, n not a multiple of 32
    rng = np.random.default_rng(8)
    n2, nf = 211, 37
    obs2 = np.exp(rng.standard_normal(n2))
    obs2[rng.choice(n2, 9, replace=False)] = np.nan
    ok = np.nonzero(~np.isnan(obs2))[0] + 1
    Z = [np.sort(rng.choice(ok, rng.integers(3, 40), replace=False)) for _ in range(nf)]
    sim = np.exp(np.log(np.nan_to_num(obs2, nan=1.0)) + 0.3 * rng.standard_normal((nf, n2)))
    assert np.allclose(_lib.cv_metrics(sim, obs2, Z), O.cv_metrics(sim, obs2, Z), rtol=1e-11, atol=1e-13)
    with pytest.raises(_lib.LdsrError):
        _lib.cv_metrics(sim, obs2, [np.array([0])] * nf)  # R indices are 1-based


def test_em_batch_across_two_devices_matches_single_device():
    # ldsr_em_batch shards groups over devices (no collective); results must not depend on the split
    if _lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    y, u, mu, inst = _np213()
    rng = np.random.default_rng(12)
    n_folds, n_rest = 7, 9
    held = [np.sort(rng.choice(inst, 11, replace=False)) for _ in range(n_folds)]
    fg = np.repeat(np.arange(n_folds), n_rest)
    th0 = rand_theta0(rng, 3, 3, n_folds * n_rest)
    ser = [dict(y=y, u=u, v=u)]
    a = _lib.em_batch(ser, np.zeros(n_folds, dtype=int), held, fg, th0, 200, 1e-5, n_devices=1)
    b = _lib.em_batch(ser, np.zeros(n_folds, dtype=int), held, fg, th0, 200, 1e-5, n_devices=2)
    for k in ("theta", "lik", "iters", "best", "X", "Y", "V", "J"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k


def _run_variant(fn, variant):
    """variant 4 (wide-input kernel) exists for widths >= 5 and only when its shared-memory plan fits."""
    try:
        return fn()
    except _lib.LdsrError as e:
        if variant in (4, 5) and e.code == _lib.ERR_UNSUPPORTED:
            pytest.skip("kernel variant %d does not cover this case (shared-memory plan / width / v != u)" % variant)
        raise


@pytest.mark.parametrize("variant", [2, 3, 4, 5, 0])
@pytest.mark.parametrize("p,q", [(5, 5), (7, 6), (10, 10), (12, 11), (16, 16), (18, 20), (32, 29)])
def test_wide_inputs(variant, p, q):
    # the padded widths 5 .. 32 (24 and 32 are built as several translation units)
    rng = np.random.default_rng(p * 100 + q)
    T = 150
    u = rng.standard_normal((p, T))
    v = rng.standard_normal((q, T)) if p != q else u
    x = np.zeros(T)
    for t in range(1, T):
        x[t] = 0.6 * x[t - 1] + 0.1 * u[0, t - 1] + 0.5 * rng.standard_normal()
    y = 0.8 * x + 0.05 * v[0] + 0.3 * rng.standard_normal(T)
    y[:60] = np.nan  # instrumental period = the last 90 steps
    th0 = rand_theta0(rng, p, q, 6)
    th0[:, 1:1 + p] *= 0.1
    th0[:, 2 + p:2 + p + q] *= 0.1
    held = [np.array([], dtype=int), np.arange(70, 90)]
    _run_variant(lambda: check_batch([dict(y=y, u=u, v=v)], [0, 0], held, np.repeat([0, 1], 3), th0, 25, 1e-6,
                                     variant=variant), variant)


@pytest.mark.parametrize("T", [8, 12, 16, 31, 32, 33, 40, 64, 65, 97, 150])
def test_wide_kernel_ragged_lengths(T):
    """em_wide_kernel on series shorter than a word, exactly one word, a word + a ragged tail ...: the
    slices of phases A / C, the piece bounds and what aliases the trajectory after phase C must hold for
    every length (fully observed and with an unobserved prefix; always enough steps for the Gram blocks
    of the p = 5 inputs to be invertible)."""
    rng = np.random.default_rng(T)
    p = 5
    u = rng.standard_normal((p, T))
    for lead in ((0,) if T < 16 else (0, T // 4)):
        y = 0.3 * rng.standard_normal(T)
        y[:lead] = np.nan
        if T >= 16:
            y[lead + 2] = np.nan
        th0 = rand_theta0(rng, p, p, 37)
        th0[:, 1:1 + p] *= 0.2
        th0[:, 2 + p:2 + 2 * p] *= 0.2
        held = [np.array([], dtype=int), np.array([T - 1]) if T >= 16 else np.array([], dtype=int)]
        check_batch([dict(y=y, u=u, v=u)], [0, 0], held, np.sort(rng.integers(0, 2, 37)), th0, 12, 1e-7, variant=4)


def test_wide_kernel_full_length_convergence_matches_oracle():
    """One station of BASELINE config 3 (T = 400, p = q = 10) x 2 folds x 50 restarts run to niter = 1000:
    the stop rule (EM.cpp:272) must fire at the SAME iteration as in the oracle after hundreds of
    iterations of the phase-split arithmetic; lik 1e-9, theta 1e-6, same selected restarts."""
    from ldsr_b200 import workloads as W
    w = W.synthetic_stations(n_stations=1, n_folds=2, n_restarts=50)
    g = _lib.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], 1000, 1e-5, variant=4)
    o = O.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], 1000, 1e-5)
    assert np.array_equal(g["iters"], o["iters"]), np.nonzero(g["iters"] != o["iters"])
    assert g["iters"].max() > 300
    assert np.allclose(g["lik"], o["lik"], rtol=LIK_RTOL, atol=0)
    assert_theta_close(g["theta"], o["theta"])
    assert np.array_equal(g["best"], o["best"])
    # and the time-split kernel of narrow inputs on the same job (the fallback when the plan does not fit)
    s = _lib.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], 1000, 1e-5, variant=3)
    assert np.array_equal(s["iters"], o["iters"]) and np.array_equal(s["best"], o["best"])


@pytest.mark.parametrize("variant", [2, 3, 5])
def test_result_of_a_fit_does_not_depend_on_its_neighbours(variant):
    """Every EM kernel classifies segments / units from the SERIES (is y finite?), never from a vote over the
    hold-out masks of the fits that happen to share a warp or CTA, so listing the groups in reverse order and
    changing the chunk length (another compaction pattern) gives bit-identical results -- for the lane-per-fit
    kernel too (ADVICE round 1: it used a warp vote)."""
    from ldsr_b200 import workloads as W
    w = W.np_cv(12, 20)
    a = em_variant(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], 150, 1e-5,
                   want_traj=False, variant=variant)
    ng = len(w["group_series"])
    perm = np.arange(ng)[::-1]
    src = np.concatenate([np.nonzero(w["fit_group"] == g)[0] for g in perm])
    fg2 = np.repeat(np.arange(ng), 20)
    b = em_variant(w["series"], w["group_series"][perm], [w["held"][g] for g in perm], fg2, w["theta0"][src], 150, 1e-5,
                   chunk_iters=13, want_traj=False, variant=variant)
    assert np.array_equal(b["iters"], a["iters"][src]) and np.array_equal(b["lik"], a["lik"][src])
    assert np.array_equal(b["theta"], a["theta"][src], equal_nan=True)


def test_full_size_cvlds_job_properties():
    """BASELINE config 2 at full size (10 000 fits: 100 folds x 100 restarts on NP-413), where the
    oracle would take minutes: size-independent properties instead.
      * EM never decreases the likelihood (trace of every fit, the E-step likelihood of each iteration);
      * the result of a fit does not depend on which other fits share its CTA / launch: reversing the
        order of the groups and changing the chunk length give bit-identical results;
      * the selected restart is the first maximum of lik among restarts with C > 0
        (R/LDS_reconstruction.R:50-58);
      * iteration counts respect the stop rule (EM.cpp:272): 3 <= iters <= niter."""
    from ldsr_b200 import workloads as W
    w = W.np_cv(100, 100)
    a = _lib.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], 1000, 1e-5,
                      want_liks=True, want_traj=False)
    it = a["iters"]
    assert it.min() >= 3 and it.max() <= 1000 and np.all(a["status"] == 0)
    liks = a["liks"]
    d = np.diff(liks, axis=1)
    valid = np.arange(999)[None, :] < (it[:, None] - 1)
    assert np.all(np.isfinite(liks[np.arange(1000)[None, :] < it[:, None]]))
    assert d[valid].min() > -1e-11, d[valid].min()  # monotone up to rounding
    assert np.allclose(liks[np.arange(it.size), it - 1], a["lik"], rtol=0, atol=0)
    # selection
    ng = len(w["group_series"])
    C = a["theta"][:, 1 + 3]
    for g in range(ng):
        idx = np.nonzero(w["fit_group"] == g)[0]
        pos = idx[C[idx] > 0]
        cand = pos if pos.size else idx
        assert a["best"][g] == cand[np.argmax(a["lik"][cand])]
    # order / chunking invariance (bitwise)
    perm_g = np.arange(ng)[::-1]
    fg_new, th_new, src = [], [], []
    for k, g in enumerate(perm_g):
        idx = np.nonzero(w["fit_group"] == g)[0]
        fg_new += [k] * idx.size
        src.append(idx)
    src = np.concatenate(src)
    b = _lib.em_batch(w["series"], [w["group_series"][g] for g in perm_g], [w["held"][g] for g in perm_g],
                      np.array(fg_new), w["theta0"][src], 1000, 1e-5, chunk_iters=250, want_traj=False)
    assert np.array_equal(b["iters"], it[src])
    assert np.array_equal(b["lik"], a["lik"][src])
    assert np.array_equal(b["theta"], a["theta"][src], equal_nan=True)


def test_task_loop_when_later_chunks_have_more_tasks_than_ctas():
    """A batch between two and three CTAs per SM: later chunks are launched with two CTAs per SM while
    more tasks are still live, so some CTAs take a second task (the task loop of both kernels).  The
    results must equal the single-launch run bit for bit."""
    from ldsr_b200 import workloads as W
    w = W.np_cv(120, 100)  # 12 000 fits = 375 tasks of 32
    for variant in (2, 3):
        a = _lib.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], 60, 1e-5,
                          chunk_iters=60, want_traj=False, variant=variant)
        b = _lib.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], 60, 1e-5,
                          chunk_iters=7, want_traj=False, variant=variant)
        for k in ("iters", "lik", "best"):
            assert np.array_equal(a[k], b[k]), (variant, k)
        assert np.array_equal(a["theta"], b["theta"], equal_nan=True)


def test_tasks_shared_by_iterations_equal_separate_runs():
    """Between one and four waves the time-split kernel's co-resident grid shares the tasks by iterations (a task's
    first iterations on one CTA, the rest on another, handed over through global memory and a flag: 375 and 313
    tasks on 296 CTAs).  The results must equal, bit for bit, those of the same fits run as two batches that
    each fit one wave (one CTA per task, no hand-over), and the call must report the time-split kernel."""
    from ldsr_b200 import workloads as W
    for folds, niter in ((120, 130), (100, 230)):
        w = W.np_cv(folds, 100)
        a = _lib.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], niter, 1e-5,
                          want_traj=False)
        st = _lib.Plan(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"]).em(niter=3)
        assert st["kernel"] == "em_split_kernel" and 0 < st["shared_slots"] < folds * 100 // 32
        for half in (np.arange(0, folds // 2), np.arange(folds // 2, folds)):
            h = W.take_groups(w, half)
            b = _lib.em_batch(h["series"], h["group_series"], h["held"], h["fit_group"], h["theta0"], niter, 1e-5,
                              want_traj=False)
            f = h["fits"]
            assert np.array_equal(b["iters"], a["iters"][f]) and np.array_equal(b["lik"], a["lik"][f])
            assert np.array_equal(b["theta"], a["theta"][f], equal_nan=True)
            assert np.array_equal(f[b["best"]], a["best"][half])


def test_repeated_runs_of_the_shared_launches_are_bit_identical():
    """Which CTA runs which iterations of which task depends on the run (hand-over between CTAs, CTAs that run ahead);
    the results must not: 25 runs of the full 10 000-fit job (313 tasks on 296 CTAs, then ranked launches) and of a
    12 000-fit job (375 tasks) give bit-identical theta, lik, iteration counts and selections -- a lost hand-over or
    a stale state read would show as a difference."""
    from ldsr_b200 import workloads as W
    for folds, niter, reps in ((100, 1000, 25), (120, 330, 10)):
        w = W.np_cv(folds, 100)
        plan = _lib.Plan(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"])
        ref = None
        for _ in range(reps):
            st = plan.em(niter=niter)
            assert st["shared_slots"] > 0
            r = plan.fetch(want_traj=False)
            if ref is None:
                ref = {k: np.array(r[k], copy=True) for k in ("theta", "lik", "iters", "best")}
            else:
                for k in ("lik", "iters", "best"):
                    assert np.array_equal(r[k], ref[k]), k
                assert np.array_equal(r["theta"], ref["theta"], equal_nan=True)


def test_ranked_assignment_with_several_series_equals_separate_runs():
    """Five stations of narrow inputs, 6 000 fits = 190 tasks: more than one task per SM, so the co-resident
    grid deals the tasks by progress and lets early CTAs run ahead (the iterations a fit advances per launch
    depend on the run).  Each station run alone is 38 tasks (one CTA per task, plain launches): results must
    agree bit for bit; and the first groups agree with the oracle."""
    from ldsr_b200 import workloads as W
    w = W.synthetic_stations(n_stations=5, T=200, p=3, n_folds=12, n_restarts=100, seed=77)
    niter = 260
    st = _lib.Plan(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"]).em(niter=3)
    assert st["kernel"] == "em_split_kernel" and st["shared_slots"] > 0
    a = _lib.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], niter, 1e-5, want_traj=False)
    for s_ in range(5):
        h = W.take_groups(w, np.arange(12 * s_, 12 * (s_ + 1)))
        b = _lib.em_batch(h["series"], h["group_series"], h["held"], h["fit_group"], h["theta0"], niter, 1e-5,
                          want_traj=False, variant=3)  # 1 200 fits would take the scan kernel by themselves
        f = h["fits"]
        assert np.array_equal(b["iters"], a["iters"][f]) and np.array_equal(b["lik"], a["lik"][f])
        assert np.array_equal(b["theta"], a["theta"][f], equal_nan=True)
    h = W.take_groups(w, np.arange(2))
    o = O.em_batch(h["series"], h["group_series"], h["held"], h["fit_group"], h["theta0"], niter, 1e-5)
    f = h["fits"]
    assert np.array_equal(a["iters"][f], o["iters"]) and np.array_equal(f[o["best"]], a["best"][:2])
    assert np.allclose(a["lik"][f], o["lik"], rtol=LIK_RTOL, atol=0)
    assert_theta_close(a["theta"][f], o["theta"])


# (T, p, q, v == u) of the synthetic winner-trajectory cases.  The scan kernel's trajectory mode takes widths up to 10
# (T <= 1024 up to width 4; T <= 512 and v == u from width 5); the others take smoother_kernel, one thread per winner.
WINNER_CASES = dict(narrow_separate_v=(150, 3, 2, False), wide10=(300, 10, 10, True),
                    wide10_separate_v=(120, 10, 4, False), long1500=(1500, 3, 3, True),
                    wide12=(300, 12, 12, True), wide16=(300, 16, 16, True), wide24=(300, 24, 24, True),
                    wide32=(300, 32, 32, True), wide6_separate_v=(200, 6, 3, False), pq4_long1100=(1100, 4, 4, True),
                    pq6_long600=(600, 6, 6, True), singular_group=(300, 12, 12, True))


def _winner_case(case):
    """The em_batch job of a winner-trajectory case (also built by the child process of the sequential-path run)."""
    rng = np.random.default_rng(21)
    if case == "np413":
        from ldsr_b200 import workloads as W
        return W.np_cv(4, 10)
    T, p, q, same = WINNER_CASES[case]
    u = rng.standard_normal((p, T))
    v = u if same else rng.standard_normal((q, T))
    x = np.zeros(T)
    for t in range(1, T):
        x[t] = 0.7 * x[t - 1] + 0.1 * u[0, t - 1] + 0.4 * rng.standard_normal()
    y = 0.6 * x + 0.05 * v[0] + 0.2 * rng.standard_normal(T)
    y[: T // 2] = np.nan
    y[T // 2 + 7] = np.nan
    inst = np.arange(T // 2, T)
    inst = inst[np.isfinite(y[inst])]
    held = [np.sort(rng.choice(inst, 9, replace=False)) for _ in range(3)] + [np.array([], dtype=int)]
    th0 = rand_theta0(rng, p, q, 4 * 6)
    th0[:, 1:1 + p] *= 0.2
    th0[:, 2 + p:2 + p + q] *= 0.2
    series, group_series = [dict(y=y, u=u, v=v)], np.zeros(4, dtype=np.int32)
    if case == "singular_group":
        # group 1 on a second series whose Tuu is exactly singular (two equal +-1 rows over the 64 steps t < T - 1):
        # all its fits are singular, it has no winner and its rows must be NaN; its neighbours are unaffected
        us = rng.standard_normal((p, 65))
        us[0] = us[1] = rng.choice([-1.0, 1.0], 65)
        ys = 0.3 * rng.standard_normal(65)
        series.append(dict(y=ys, u=us, v=us))
        group_series[1] = 1
        held[1] = np.array([], dtype=int)
    return dict(series=series, group_series=group_series, held=held, fit_group=np.repeat(np.arange(4), 6), theta0=th0)


@pytest.mark.parametrize("case", ["np413", "narrow_separate_v", "wide10", "wide10_separate_v", "long1500", "wide12",
                                  "wide16", "wide24", "wide32", "wide6_separate_v", "pq4_long1100", "pq6_long600",
                                  "singular_group"])
def test_winner_trajectories_equal_the_oracle_estep_with_the_same_theta(case, tmp_path):
    """X, Y, V, J returned by ldsr_em_batch are the E-step (EM.cpp:43-110) of the selected restart's theta on the
    group's y: compared with the oracle's smoother run with the GPU's OWN theta, so the tolerance is that of one
    E-step (1e-10), not of a whole EM run.  Covers both trajectory paths: the scan kernel's trajectory mode
    (narrow inputs, or wide with v == u, series up to 1024 / 512 steps) and the one-thread-per-winner kernel
    (wider inputs, v != u from width 5, longer series), whose rows are NaN for a group without a winner.
    Where the scan kernel applies (np413, wide10), the one-thread-per-winner kernel is also run on the same job
    (LDSR_SEQ_TRAJ=1, read once, so in a child process) and both paths must agree to 1e-10."""
    w = _winner_case(case)
    g = _lib.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], 40, 1e-5)
    for k in range(len(w["group_series"])):
        row = slice(g["traj_ptr"][k], g["traj_ptr"][k + 1])
        if case == "singular_group" and k == 1:
            assert np.all(g["status"][w["fit_group"] == 1] == _lib.FIT_SINGULAR) and g["best"][k] == -1
            for name in ("X", "Y", "V", "J"):
                assert np.isnan(g[name][row]).all(), name
            continue
        s0 = w["series"][w["group_series"][k]]
        yy = np.array(s0["y"], dtype=float)
        yy[w["held"][k]] = np.nan
        s = O.kalman_smoother(yy, s0["u"], s0["v"], g["theta"][g["best"][k]])
        for name in ("X", "Y", "V", "J"):
            assert np.allclose(g[name][row], s[name], rtol=1e-10, atol=1e-13), (k, name)
    if case in ("np413", "wide10"):
        import subprocess
        import sys
        f = str(tmp_path / "seq.npz")
        code = ("import sys, numpy as np; sys.path.insert(0, %r)\n"
                "from ldsr_b200 import _lib; from tests.test_gpu_parity import _winner_case\n"
                "w = _winner_case(sys.argv[2])\n"
                "r = _lib.em_batch(w['series'], w['group_series'], w['held'], w['fit_group'], w['theta0'], 40, 1e-5)\n"
                "np.savez(sys.argv[1], **r)\n") % ROOT
        subprocess.run([sys.executable, "-c", code, f, case], check=True, env=dict(os.environ, LDSR_SEQ_TRAJ="1"),
                       timeout=300)
        seq = np.load(f)
        assert np.array_equal(seq["theta"], g["theta"]) and np.array_equal(seq["best"], g["best"])
        for name in ("X", "Y", "V", "J"):
            assert np.allclose(seq[name], g[name], rtol=1e-10, atol=1e-13), name


def test_lds_rep_chunked_pipeline_equals_the_single_kernel_path(tmp_path):
    """ldsr_rep_batch simulates every replicate in one kernel when the output fits HBM and in pipelined chunks
    otherwise; the device generator is keyed by (seed, replicate, step), so both give the same bits.  The
    chunked path is forced through LDSR_REP_CHUNKED in a child process (the switch is read once).
    seed: n = 813, 9000 replicates (two chunks).  z, r_seed, three_chunks: n = 4000, 4000 replicates are chunks of
    1664, 1664 and 672 replicates, so the third chunk re-uses the first one's slot; the noise comes from the caller,
    from R's stream after set.seed, or from the device generator."""
    import subprocess
    import sys
    code = ("import sys, numpy as np; sys.path.insert(0, %r); from ldsr_b200 import _lib; from tests import data\n"
            "d = data.load('np.json'); th = data.theta_of(d['theta']); y, u, mu, inst = data.np_case(1, 1200)\n"
            "case = sys.argv[2]\n"
            "if case == 'seed':\n"
            "    r = _lib.rep_batch(th, u, u, y.size, 9000, seed=7, mu=mu)\n"
            "else:\n"
            "    n = 4000; rng = np.random.default_rng(40); u = rng.standard_normal((3, n))\n"
            "    kw = dict(z=rng.standard_normal((n, 1 + 2 * n))) if case == 'z' else (\n"
            "        dict(r_seed=11) if case == 'r_seed' else dict(seed=5))\n"
            "    r = _lib.rep_batch(th, u, u, n, n, mu=mu, want=('simQ',), **kw)\n"
            "np.save(sys.argv[1], np.stack([r[k] for k in ('simX', 'simY', 'simQ') if k in r]))\n") % ROOT
    for case in ("seed", "z", "r_seed", "three_chunks"):
        outs = []
        for k, env in enumerate(({}, {"LDSR_REP_CHUNKED": "1"})):
            f = str(tmp_path / ("rep_%s%d.npy" % (case, k)))
            subprocess.run([sys.executable, "-c", code, f, case], check=True, env=dict(os.environ, **env), timeout=300)
            outs.append(np.load(f))
        assert np.isfinite(outs[0]).all() and np.array_equal(outs[0], outs[1]), case


def test_construct_rec_kernel_reproduces_the_stored_reconstruction():
    # R/sysdata.rda::NPlds$rec (X, Xl, Xu, Q, Ql, Qu, T = 813) from the GPU E-step with the stored theta
    g = data.load("nplds.json")
    y, u, mu, inst = data.np_case(1, 1200)
    th = data.theta_of(g["theta"])
    s = L.Kalman_smoother(y, u, u, L.vec_to_theta(th, 3, 3))
    out, mean = _lib.construct_rec(s["X"], s["V"], s["Y"], th[4], th[9], mu, "log")
    for j, name in enumerate(_lib.REC_COLUMNS):
        assert np.allclose(out[0, j], np.array(g["rec"][name]), rtol=1e-10, atol=1e-11), name
    # ensemble of 3 members, all three transforms, against the oracle
    rng = np.random.default_rng(4)
    n, T = 3, 97
    X, Y = rng.standard_normal((n, T)), 0.3 * rng.standard_normal((n, T)) + 1.0
    V = rng.uniform(0.1, 2.0, (n, T))
    Cm, Rm = rng.uniform(0.1, 1.0, n), rng.uniform(0.01, 0.2, n)
    for tr, lam in (("log", 0.0), ("none", 0.0), ("boxcox", 0.3), ("boxcox", 0.0)):
        a, am = _lib.construct_rec(X, V, Y, Cm, Rm, 0.7, tr, lam)
        b, bm = O.construct_rec(X, V, Y, Cm, Rm, 0.7, tr, lam)
        assert np.allclose(a, b, rtol=1e-12, atol=1e-13) and np.allclose(am, bm, rtol=1e-12, atol=1e-13), tr


def test_objectives_of_the_experimental_learners():
    # penalized_likelihood / negLogLik / ssqTrain (R/LDS_GA.R:28-44, 136-147) for a population of thetas
    y, u, mu, inst = _np213()
    rng = np.random.default_rng(17)
    n = 40
    th = rand_theta0(rng, 3, 3, n)
    th[:, 8] = rng.uniform(0.2, 2.0, n)   # Q
    th[:, 9] = rng.uniform(0.05, 1.0, n)  # R
    ser = [dict(y=y, u=u, v=u)]
    none = [np.array([], dtype=int)]
    for kind, lam in (("penalized_likelihood", 1.0), ("penalized_likelihood", 0.25), ("negLogLik", 0.0), ("ssqTrain", 0.0)):
        g = _lib.objective_batch(ser, [0], none, np.zeros(n, dtype=int), th, kind, lam)
        o = np.array([O.objective(y, u, u, th[i], kind, lam) for i in range(n)])
        assert np.allclose(g, o, rtol=1e-9, atol=1e-12), (kind, np.max(np.abs(g - o)))


@pytest.mark.parametrize("variant", VARIANTS)
def test_unusual_initial_values(variant):
    # initial values outside make_init's ranges: negative / explosive A, negative C, tiny and large noise
    # variances.  The unobserved-unit shortcuts use powers of A and A^2 up to A^64: they must agree with
    # the step-by-step oracle for every sign and for |A| > 1 as well.
    y, u, mu, inst = data.np_case(401, 1600)  # T = 413, 360 unobserved steps before the first record
    base = np.array([0.5, 0.3, -0.2, 0.1, 0.5, 0.05, -0.1, 0.2, 1.0, 1.0, 0.0, 1.0])
    th = []
    for A in (-0.9, -0.3, 1e-3, 0.999, 1.02):
        for C in (0.7, -0.4):
            for Q, R in ((1.0, 1.0), (1e-3, 10.0), (25.0, 1e-3)):
                t = base.copy()
                t[0], t[4], t[8], t[9] = A, C, Q, R
                th.append(t)
    th = np.stack(th)
    fg = np.zeros(len(th), dtype=int)
    none = [np.array([], dtype=int)]
    g = em_variant([dict(y=y, u=u, v=u)], [0], none, fg, th, 4, 0.0, want_liks=True, variant=variant)
    o = O.em_batch([dict(y=y, u=u, v=u)], [0], none, fg, th, 4, 0.0)
    assert np.array_equal(g["iters"], o["iters"])
    # a stable start is held to the usual bars; an explosive one (A = 1.02: the predicted variance reaches
    # 1e7 Q before the first record, so the update (1 - K C) P cancels ~11 digits against R = 1e-3) is
    # ill-conditioned in the reference's own arithmetic and is held to the digits that survive
    stable = np.abs(th[:, 0]) < 1.0
    assert np.allclose(g["lik"][stable], o["lik"][stable], rtol=1e-9, atol=0)
    # The scan kernel (variant 5) forms the smoothed mean of step 0 -- the new mu1 -- by composing affine maps
    # over the whole series: its ABSOLUTE error is a few ulps of the O(1) terms composed, while the value itself
    # is ~A^360 here (the first record is 360 steps away; the sequential recursions carry that decay exactly).
    # mu1 only enters the next E-step additively, so 1e-12 absolute is far inside every other bar.
    assert_theta_close(g["theta"][stable], o["theta"][stable], 1e-6, floor=1e-6 if variant == 5 else 1e-8)
    assert np.allclose(g["lik"][~stable], o["lik"][~stable], rtol=1e-6, atol=0)
    assert_theta_close(g["theta"][~stable], o["theta"][~stable], 1e-5)


def test_repeated_calls_reuse_the_context_arenas_and_trim_releases_them():
    # a long R session calls the library thousands of times with batches of varying size: the
    # context's cache must stop growing once it has seen the largest call, repeated calls must give
    # identical results, and ldsr_ctx_trim must hand the cached blocks back
    import torch

    torch.cuda.init()
    y, u, mu, inst = _np213()
    ser = [dict(y=y, u=u, v=u)]
    none = [np.array([], dtype=int)]
    ctx = _lib.Ctx(devices=[0])
    sizes = [64, 7, 300, 33, 128, 300, 5, 64, 300, 17, 300, 64]
    first, free = {}, []
    for n in sizes:
        th = rand_theta0(np.random.default_rng(1000), 3, 3, 300)[:n]
        r = _lib.em_batch(ser, [0], none, np.zeros(n, dtype=int), th, 30, 1e-5, ctx=ctx, want_traj=False)
        key = n
        if key in first:
            assert np.array_equal(first[key]["theta"], r["theta"], equal_nan=True)
            assert np.array_equal(first[key]["lik"], r["lik"])
        first[key] = r
        free.append(torch.cuda.mem_get_info(0)[0])
    assert free[-1] == free[5], (free[5], free[-1])  # no growth after the largest batch has been seen twice
    freed, kept = ctx.trim()
    assert freed > 0 and kept == 0
    assert torch.cuda.mem_get_info(0)[0] >= free[-1] + freed - (1 << 20)
    r = _lib.em_batch(ser, [0], none, np.zeros(64, dtype=int),
                      rand_theta0(np.random.default_rng(1000), 3, 3, 300)[:64],
                      30, 1e-5, ctx=ctx, want_traj=False)
    assert np.array_equal(first[64]["lik"], r["lik"])
    ctx.close()


def test_wide_multi_station_batch_matches_oracle_and_is_order_invariant():
    # BASELINE config 3 in miniature: several stations of different length with ten inputs each (the
    # width at which B and D live in shared memory and one warp does the M-step), two folds per
    # station, a handful of restarts.  Against the oracle, and bit-identical when the stations are
    # listed in reverse and the chunk length changes (a CTA then walks different tasks in a different
    # order through the same shared-memory areas).
    from ldsr_b200 import workloads as W
    w = W.synthetic_stations(n_stations=3, T=200, p=10, n_folds=2, n_restarts=5, seed=77)
    for i, s in enumerate(w["series"]):  # ragged: shorten two of the three stations
        cut = (0, 37, 90)[i]
        if cut:
            s["y"], s["u"], s["v"] = s["y"][cut:], s["u"][:, cut:], s["v"][:, cut:]
            for g in np.nonzero(w["group_series"] == i)[0]:
                w["held"][g] = w["held"][g] - cut
    niter = 40
    a = _lib.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], niter, 1e-6,
                      want_traj=False)
    o = O.em_batch(w["series"], w["group_series"], w["held"], w["fit_group"], w["theta0"], niter, 1e-6)
    assert np.array_equal(a["iters"], o["iters"]) and np.array_equal(a["best"], o["best"])
    assert np.allclose(a["lik"], o["lik"], rtol=LIK_RTOL, atol=0)
    assert_theta_close(a["theta"], o["theta"])
    # reversed station order, different chunking
    ng = len(w["group_series"])
    ns = len(w["series"])
    perm = np.arange(ng)[::-1]
    fg2, th2, src = [], [], []
    for gnew, gold in enumerate(perm):
        idx = np.nonzero(w["fit_group"] == gold)[0]
        fg2 += [gnew] * idx.size
        th2.append(w["theta0"][idx])
        src.append(idx)
    src = np.concatenate(src)
    b = _lib.em_batch(w["series"][::-1], (ns - 1 - w["group_series"])[perm], [w["held"][g] for g in perm],
                      np.array(fg2), np.concatenate(th2), niter, 1e-6, chunk_iters=7, want_traj=False)
    assert np.array_equal(b["iters"], a["iters"][src]) and np.array_equal(b["lik"], a["lik"][src])
    assert np.array_equal(b["theta"], a["theta"][src], equal_nan=True)
