"""Many stations in one batched call (cvLDS_stations / LDS_reconstruction_stations and the ragged epilogues
ldsr_cv_metrics_stations / ldsr_construct_rec_stations) against the single-station calls, the entry points
they generalise, the reference's stored results and the CPU oracle."""
import numpy as np
import pytest

import ldsr_b200 as L
from ldsr_b200 import _lib, api
from oracle import oracle as O
from tests import data
from tests.test_gpu_parity import LIK_RTOL, THETA_RTOL, assert_theta_close

pytestmark = pytest.mark.gpu


def _np():
    d = data.load("np.json")
    years, qa = np.array(d["NPannual"]["year"]), np.array(d["NPannual"]["Qa"])
    pc = np.array([d["NPpc"][k] for k in ("PC1", "PC9", "PC13")])
    return years, qa, pc


def _stations():
    """Five stations that differ in T, p, q, instrumental period and start year: one without u, one
    two-member ensemble of unequal widths."""
    years, qa, pc = _np()
    rng = np.random.default_rng(31)
    qb = qa * np.exp(0.2 * rng.standard_normal(qa.size))  # a second gauge with its own flows
    return [dict(Qa=dict(year=years, Qa=qa), u=pc[:, 600:], v=pc[:, 600:], start_year=1800),
            dict(Qa=dict(year=years[6:], Qa=qb[6:]), u=None, v=pc[:2, 650:], start_year=1850),
            dict(Qa=dict(year=years[:-4], Qa=qa[:-4]), u=[pc[:, 480:], pc[:1, 480:]], v=[pc[:, 480:], pc[1:, 480:]],
                 start_year=1680),
            dict(Qa=dict(year=years[3:-3], Qa=qb[3:-3]), u=pc[:1, 700:], v=pc[:, 700:], start_year=1900),
            dict(Qa=dict(year=years, Qa=qb), u=pc[:2, 550:], v=pc[:1, 550:], start_year=1750)]


def _close(a, b, rtol, atol=0.0):
    assert np.allclose(a, b, rtol=rtol, atol=atol), np.max(np.abs(np.asarray(a) - np.asarray(b)))


@pytest.mark.parametrize("transform", ["log", "boxcox"])
def test_cvlds_stations_equal_per_station_calls(transform):
    st = _stations()
    st[3] = dict(st[3], Z=L.make_Z(st[3]["Qa"]["Qa"], 4, contiguous=False, rng=np.random.default_rng(1)))
    kw = dict(transform=transform, num_restarts=4, niter=300)
    many = L.cvLDS_stations([dict(s, Z=s.get("Z")) for s in st], rng=np.random.default_rng(5), **kw)
    rng = np.random.default_rng(5)
    one = [L.cvLDS(s["Qa"], s["u"], s["v"], s["start_year"], Z=s.get("Z"), rng=rng, **kw) for s in st]
    assert len(many) == len(st)
    for a, b in zip(many, one):
        assert set(a) == set(b) and len(a["Z"]) == len(b["Z"])
        assert all(np.array_equal(x, y) for x, y in zip(a["Z"], b["Z"]))
        assert np.array_equal(a["best"], b["best"]) and np.array_equal(a["iters"], b["iters"])
        _close(a["lik"], b["lik"], LIK_RTOL)
        assert a["Ycv"].shape == b["Ycv"].shape
        _close(a["Ycv"], b["Ycv"], THETA_RTOL)
        for k in _lib.METRIC_NAMES:
            _close(a["metrics_dist"][k], b["metrics_dist"][k], 1e-5, 1e-9)
        assert np.array_equal(a["target"]["y"], b["target"]["y"])


@pytest.mark.parametrize("transform", ["log", "boxcox"])
def test_reconstruction_stations_equal_per_station_calls(transform):
    st = _stations()
    kw = dict(transform=transform, num_restarts=4, niter=300, return_init=True, return_raw=True)
    many = L.LDS_reconstruction_stations(st, rng=np.random.default_rng(6), **kw)
    rng = np.random.default_rng(6)
    one = [L.LDS_reconstruction(s["Qa"], s["u"], s["v"], s["start_year"], rng=rng, **kw) for s in st]
    for a, b in zip(many, one):
        assert set(a) == set(b)
        ma, mb = a.get("ensemble", [a]), b.get("ensemble", [b])
        for x, y in zip(ma, mb):
            assert set(x) == set(y)
            _close(x["lik"], y["lik"], LIK_RTOL)
            assert_theta_close(api.theta_to_vec(x["theta"]), api.theta_to_vec(y["theta"]))
            assert np.array_equal(api.theta_to_vec(x["init"]), api.theta_to_vec(y["init"]))
            for r in ("rec", "rec2"):
                assert np.array_equal(x[r]["year"], y[r]["year"])
                for c in _lib.REC_COLUMNS:
                    _close(x[r][c], y[r][c], THETA_RTOL, 1e-9)
            if transform == "boxcox":
                assert x["lambda"] == y["lambda"]
        if "ensemble" in a:
            for r in ("rec", "rec_raw"):
                for c in ("X", "Q"):
                    _close(a[r][c], b[r][c], THETA_RTOL, 1e-9)
                    # the kernel's ensemble mean is numpy's member-order mean, bit for bit
                    assert np.array_equal(a[r][c], np.mean([m["rec" if r == "rec" else "rec2"][c] for m in ma], axis=0))


def _ragged_case(rng, sizes):
    sims, obss, Zs = [], [], []
    for n, nf in sizes:
        obs = np.exp(rng.standard_normal(n))
        obs[rng.choice(n, 3, replace=False)] = np.nan
        ok = np.nonzero(~np.isnan(obs))[0] + 1
        Zs.append([np.sort(rng.choice(ok, rng.integers(3, n // 3), replace=False)) for _ in range(nf)])
        sims.append(np.exp(np.log(np.nan_to_num(obs, nan=1.0)) + 0.3 * rng.standard_normal((nf, n))))
        obss.append(obs)
    return sims, obss, Zs


def test_ragged_epilogues_equal_the_existing_entry_points_bit_for_bit():
    rng = np.random.default_rng(12)
    sims, obss, Zs = _ragged_case(rng, [(46, 30), (211, 7), (33, 1), (97, 12)])
    many = _lib.cv_metrics_stations(sims, obss, Zs)
    for s in range(len(sims)):
        ref = _lib.cv_metrics(sims[s], obss[s], Zs[s])
        assert np.array_equal(_lib.cv_metrics_stations([sims[s]], [obss[s]], [Zs[s]])[0], ref)
        assert np.array_equal(many[s], ref)
        assert np.array_equal(_lib.cv_metrics_stations(np.log(sims[s])[None], [obss[s]], [Zs[s]], exp_trans=True)[0],
                              _lib.cv_metrics(np.log(sims[s]), obss[s], Zs[s], exp_trans=True))
    for tr in ("log", "none", "boxcox"):
        shapes = [(3, 97), (1, 213), (2, 40)]
        X = [rng.standard_normal(sh) for sh in shapes]
        V = [rng.uniform(0.1, 2.0, sh) for sh in shapes]
        Y = [0.3 * rng.standard_normal(sh) + 1.0 for sh in shapes]
        Cm = [rng.uniform(0.1, 1.0, sh[0]) for sh in shapes]
        Rm = [rng.uniform(0.01, 0.2, sh[0]) for sh in shapes]
        mus, lams = [0.7, 0.2, 1.1], ([0.3, 0.0, -0.4] if tr == "boxcox" else None)
        many = _lib.construct_rec_stations(X, V, Y, Cm, Rm, mus, tr, lams)
        for s in range(len(shapes)):
            lam = 0.0 if lams is None else lams[s]
            ref = _lib.construct_rec(X[s], V[s], Y[s], Cm[s], Rm[s], mus[s], tr, lam)
            one = _lib.construct_rec_stations([X[s]], [V[s]], [Y[s]], [Cm[s]], [Rm[s]], [mus[s]], tr, [lam])[0]
            for got in (one, many[s]):  # a negative lambda makes pow() NaN where y * lambda + 1 < 0, in both
                assert np.array_equal(got[0], ref[0], equal_nan=True), (tr, s)
                assert np.array_equal(got[1], ref[1], equal_nan=True), (tr, s)


def test_oracle_pins_hold_through_the_ragged_path():
    # R/sysdata.rda::NPcv metrics.dist, computed in one call together with another station
    g = data.load("npcv.json")
    n = len(g["target"]["y"])
    Y = np.array(g["Ycv"]["Y"]).reshape(-1, n)
    sims, obss, Zs = _ragged_case(np.random.default_rng(3), [(71, 5)])
    m = _lib.cv_metrics_stations(sims + [Y], obss + [np.array(g["target"]["y"])], Zs + [g["Z"]])
    for j, name in enumerate(_lib.METRIC_NAMES):
        assert np.allclose(m[1][:, j], np.array(g["metrics_dist"][name]), rtol=1e-10, atol=1e-12), name
    assert np.allclose(m[0], O.cv_metrics(sims[0], obss[0], Zs[0]), rtol=1e-11, atol=1e-13)
    # R/sysdata.rda::NPlds$rec from the GPU E-step with the stored theta, next to a shorter station
    g = data.load("nplds.json")
    y, u, mu, inst = data.np_case(1, 1200)
    th = data.theta_of(g["theta"])
    s = L.Kalman_smoother(y, u, u, L.vec_to_theta(th, 3, 3))
    s2 = L.Kalman_smoother(y[400:], u[:, 400:], u[:, 400:], L.vec_to_theta(th, 3, 3))
    rec = _lib.construct_rec_stations([s2["X"], s["X"]], [s2["V"], s["V"]], [s2["Y"], s["Y"]], [[th[4]], [th[4]]],
                                      [[th[9]], [th[9]]], [mu, mu], "log")
    for j, name in enumerate(_lib.REC_COLUMNS):
        assert np.allclose(rec[1][0][0, j], np.array(g["rec"][name]), rtol=1e-10, atol=1e-11), name


def _check_use_raw(res, stations, transform, num_restarts, niter, seed):
    """Every fold output of a use_raw run equals the oracle's open-loop propagate of the selected fit on the
    fold's y, member-averaged, and its metrics equal the oracle's calculate_metrics of those outputs."""
    P, B = api.cv_batch(stations, transform, num_restarts, np.random.default_rng(seed))
    r = _lib.em_batch(B["series"], B["group_series"], B["held"], B["fit_group"], B["theta0"], niter, 1e-5)
    for S, got in zip(P, res):
        nm, inst = len(S["series"]), S["inst"]
        sims = []
        for k in range(len(S["Z"])):
            cols = []
            for m in range(nm):
                g = S["g0"] + k * nm + m
                s = B["series"][B["group_series"][g]]
                y = s["y"].copy()
                y[B["held"][g]] = np.nan
                th = r["theta"][r["best"][g], :s["p"] + s["q"] + 6]
                cols.append(O.propagate(th, s["u"], s["v"], y, p=s["p"], q=s["q"])["Y"][inst] + S["mu"])
            sims.append(np.exp(np.mean(cols, axis=0)) if transform == "log" else np.mean(cols, axis=0))
        assert np.allclose(got["Ycv"], np.stack(sims, axis=1), rtol=1e-12, atol=0)
        o = O.cv_metrics(np.stack(sims), got["target"]["y"], S["Z"])
        for j, k in enumerate(_lib.METRIC_NAMES):
            assert np.allclose(got["metrics_dist"][k], o[:, j], rtol=1e-10, atol=1e-12), k


def test_use_raw():
    st = _stations()
    kw = dict(num_restarts=3, niter=200)
    for s in (st[0], st[2]):  # a single model and a two-member ensemble
        Z = L.make_Z(s["Qa"]["Qa"], 4, rng=np.random.default_rng(2))
        res = L.cvLDS(s["Qa"], s["u"], s["v"], s["start_year"], Z=Z, use_raw=True, rng=np.random.default_rng(9), **kw)
        smooth = L.cvLDS(s["Qa"], s["u"], s["v"], s["start_year"], Z=Z, rng=np.random.default_rng(9), **kw)
        assert np.array_equal(res["best"], smooth["best"]) and not np.allclose(res["Ycv"], smooth["Ycv"])
        _check_use_raw([res], [dict(s, Z=Z)], "log", 3, 200, 9)
    res = L.cvLDS_stations(st, use_raw=True, rng=np.random.default_rng(4), **kw)
    _check_use_raw(res, st, "log", 3, 200, 4)


def test_stations_on_two_devices_equal_one_device():
    if _lib.device_count() < 2:
        pytest.skip("needs two GPUs")
    st = _stations()
    kw = dict(num_restarts=4, niter=300)
    for fn, extra in ((L.cvLDS_stations, dict(use_raw=True)), (L.LDS_reconstruction_stations, dict(return_raw=True))):
        a = fn(st, rng=np.random.default_rng(8), n_devices=2, **kw, **extra)
        b = fn(st, rng=np.random.default_rng(8), n_devices=1, **kw, **extra)
        for x, y in zip(a, b):
            if fn is L.cvLDS_stations:
                for k in ("best", "iters", "lik", "Ycv"):
                    assert np.array_equal(x[k], y[k]), k
                for k in _lib.METRIC_NAMES:
                    assert np.array_equal(x["metrics_dist"][k], y["metrics_dist"][k]), k
            else:
                for mx, my in zip(x.get("ensemble", [x]), y.get("ensemble", [y])):
                    assert mx["lik"] == my["lik"]
                    for r in ("rec", "rec2"):
                        for c in _lib.REC_COLUMNS:
                            assert np.array_equal(mx[r][c], my[r][c]), (r, c)
