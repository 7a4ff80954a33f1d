"""Python mirror of the reference's R API for the EM path -- same function names, argument
meaning, defaults and error behaviour -- on top of the CUDA library (ldsr_b200/_lib.py).

R is not installed in the build image, so this module plays the role the R wrappers in
ldsr_b200/r/ play for an R user (see INTEGRATION.md); the parity tests are written against it
so that they read like tests/testthat/test-LDS-EM.R.

Conventions carried over from R:
  * u, v are [p, T] / [q, T] arrays (R matrices), or None (R: NULL -> `matrix(0)` sentinel,
    R/LDS_reconstruction.R:131-136); an ensemble is a list of such arrays.
  * theta is a dict with keys A, B, C, D, Q, R, mu1, V1 (R: list of 1x1 / 1xp matrices).
  * y is a length-T vector with NaN for missing (R: NA).
  * Random numbers: the reference draws initial values from R's global RNG (make_init) inside
    each worker.  Here the caller passes a numpy Generator; draws are made in the reference's
    order (fold-major, then restart, then A, B[1..p], C, D[1..q]) -- see LDS_EM_restart/cvLDS.
Every numeric result comes from the GPU; there is no CPU path in this module.
"""
import numpy as np

from . import _lib

_Z05 = 1.6448536269514722  # qnorm(0.95)


# ---------------------------------------------------------------------------------------------
# theta helpers
# ---------------------------------------------------------------------------------------------
def theta_to_vec(theta):
    """R/LDS_GA.R:6-16 order: [A, B, C, D, Q, R, mu1, V1]."""
    return np.concatenate([np.ravel(theta[k]) for k in ("A", "B", "C", "D", "Q", "R", "mu1", "V1")]).astype(float)


def vec_to_theta(vec, p, q):
    vec = np.asarray(vec, dtype=float)
    return dict(A=float(vec[0]), B=vec[1:1 + p].copy(), C=float(vec[1 + p]), D=vec[2 + p:2 + p + q].copy(),
                Q=float(vec[2 + p + q]), R=float(vec[3 + p + q]), mu1=float(vec[4 + p + q]),
                V1=float(vec[5 + p + q]))


def _dims(u, v):
    """nrow(u), nrow(v) with the matrix(0) sentinel counting as one row."""
    p = 1 if u is None else np.atleast_2d(u).shape[0]
    q = 1 if v is None else np.atleast_2d(v).shape[0]
    return p, q


def make_init(p, q, num_restarts, rng):
    """R/LDS_reconstruction.R:14-30: A~U(0,1), B~U(-1,1)^p, C~U(0,1), D~U(-1,1)^q, Q=R=V1=1, mu1=0,
    drawn per restart in that order."""
    out = []
    for _ in range(num_restarts):
        A = rng.uniform()
        B = rng.uniform(-1, 1, p)
        Cc = rng.uniform()
        D = rng.uniform(-1, 1, q)
        out.append(dict(A=A, B=B, C=Cc, D=D, Q=1.0, R=1.0, mu1=0.0, V1=1.0))
    return out


def make_Z(obs, nRuns=30, frac=0.1, contiguous=True, rng=None):
    """R/utils.R:83-101.  Returns 1-based index vectors like R (indices into obs)."""
    rng = rng or np.random.default_rng()
    obs = np.asarray(obs, dtype=float)
    obsInd = np.nonzero(~np.isnan(obs))[0] + 1
    if frac == 1:
        return [np.array([i]) for i in obsInd]
    n = obsInd.size
    k = int(np.floor(n * frac))
    if contiguous:
        maxInd = n - k
        if maxInd < nRuns:  # the reference's fallback (utils.R:92-95); negative k is its bug, we refuse
            maxInd = nRuns
            k = n - nRuns
            if k < 0 or maxInd + k > n:
                raise ValueError("make_Z: cannot make %d contiguous folds out of %d points "
                                 "(the reference misbehaves here, R/utils.R:92-95)" % (nRuns, n))
        starts = np.sort(rng.choice(np.arange(1, maxInd + 1), nRuns, replace=False))
        return [obsInd[x - 1:x + k] for x in starts]  # obsInd[x:(x+k)]: k+1 points
    return [np.sort(rng.choice(obsInd, k, replace=False)) for _ in range(nRuns)]


def _series(y, u, v):
    p, q = _dims(u, v)
    return dict(y=np.asarray(y, dtype=float).ravel(), u=None if u is None else np.atleast_2d(u),
                v=None if v is None else np.atleast_2d(v), p=p, q=q)


def _fit_dict(r, row, T):
    sl = slice(row, row + T)
    return dict(X=r["X"][sl].copy(), Y=r["Y"][sl].copy(), V=r["V"][sl].copy(), J=r["J"][sl].copy())


# ---------------------------------------------------------------------------------------------
# The reference's four .Call functions (R/RcppExports.R:15-59)
# ---------------------------------------------------------------------------------------------
def Kalman_smoother(y, u, v, theta, stdlik=True):
    s = _series(y, u, v)
    r = _lib.smoother_batch([s], [0], None, [0], theta_to_vec(theta)[None, :], stdlik)
    return dict(X=r["X"][0], Y=r["Y"][0], V=r["V"][0], J=r["J"][0], lik=float(r["lik"][0]))


def Mstep(y, u, v, fit):
    s = _series(y, u, v)
    r = _lib.mstep_batch([s], [0], None, [0], [fit["X"]], [fit["V"]], [fit["J"]], s["p"] + s["q"] + 6)
    if r["status"][0] == _lib.FIT_SINGULAR:
        raise _lib.LdsrError(_lib.ERR_ARG, "Mstep: inv(): matrix is singular")
    return vec_to_theta(r["theta"][0], s["p"], s["q"])


def LDS_EM(y, u, v, theta0, niter=1000, tol=1e-5):
    s = _series(y, u, v)
    r = _lib.em_batch([s], [0], None, [0], theta_to_vec(theta0)[None, :], niter, tol, want_liks=True)
    if r["status"][0] == _lib.FIT_SINGULAR:
        raise _lib.LdsrError(_lib.ERR_ARG, "LDS_EM: inv(): matrix is singular")
    n = int(r["iters"][0])
    fit = _fit_dict(r, 0, s["y"].size)
    fit["lik"] = float(r["lik"][0])
    return dict(theta=vec_to_theta(r["theta"][0], s["p"], s["q"]), fit=fit, liks=r["liks"][0, :n].copy(),
                lik=float(r["lik"][0]))


def propagate(theta, u, v, y, stdlik=True):
    s = _series(y, u, v)
    r = _lib.propagate_batch([s], [0], None, [0], theta_to_vec(theta)[None, :], stdlik)
    return dict(X=r["X"][0], Y=r["Y"][0], V=r["V"][0], lik=float(r["lik"][0]))


# ---------------------------------------------------------------------------------------------
# Restart / cross-validation fan-out: ONE batched GPU call instead of foreach %dopar%
# ---------------------------------------------------------------------------------------------
def LDS_EM_restart(y, u, v, init, niter=1000, tol=1e-5, return_init=True, n_devices=1):
    """R/LDS_reconstruction.R:42-62: all restarts as one batch, selection on the device."""
    s = _series(y, u, v)
    th0 = np.stack([theta_to_vec(t) for t in init])
    r = _lib.em_batch([s], [0], None, np.zeros(len(init), dtype=np.int32), th0, niter, tol,
                      n_devices=n_devices)
    if np.any(r["status"] == _lib.FIT_SINGULAR):
        raise _lib.LdsrError(_lib.ERR_ARG, "LDS_EM_restart: inv(): matrix is singular")
    b = int(r["best"][0])
    if b < 0:
        raise _lib.LdsrError(_lib.ERR_ARG, "LDS_EM_restart: no restart produced a finite likelihood")
    fit = _fit_dict(r, 0, s["y"].size)
    fit["lik"] = float(r["lik"][b])
    ans = dict(theta=vec_to_theta(r["theta"][b], s["p"], s["q"]), fit=fit, lik=float(r["lik"][b]),
               iters=int(r["iters"][b]), all_lik=r["lik"], all_iters=r["iters"], best=b)
    if return_init:
        ans["init"] = init[b]
    return ans


def _prep_uv(u, v):
    """Argument checks of LDS_reconstruction / cvLDS (R/LDS_reconstruction.R:128-157, :315-340).
    Returns (single, list of u, list of v, N)."""
    single = not isinstance(u, (list, tuple)) and not isinstance(v, (list, tuple))
    if single:
        if u is None and v is None:
            raise ValueError("u and v cannot both be NULL")
        if u is not None and v is not None and np.atleast_2d(u).shape[1] != np.atleast_2d(v).shape[1]:
            raise ValueError("u and v must have the same number of time steps.")
        N = np.atleast_2d(u if u is not None else v).shape[1]
        return True, [u], [v], N
    if u is None:
        u = [None] * len(v)
    if v is None:
        v = [None] * len(u)
    for a, b in zip(u, v):
        if a is not None and b is not None and np.atleast_2d(a).shape[1] != np.atleast_2d(b).shape[1]:
            raise ValueError("u and v must have the same number of time steps.")
    first = u[0] if u[0] is not None else v[0]
    return False, list(u), list(v), np.atleast_2d(first).shape[1]


def _boxcox_lambda(y):
    """MASS::boxcox(y ~ 1, plotit = FALSE): profile log-likelihood on lambda = seq(-2, 2, 0.1)."""
    y = np.asarray(y, dtype=float)
    n = y.size
    logy = np.log(y)
    ydot = np.exp(logy.mean())
    lam = np.round(np.arange(-2, 2.0001, 0.1), 10)
    ll = []
    for l in lam:
        yt = (np.log(y) * ydot) if abs(l) < 1e-12 else ((y / ydot) ** l - 1) / l * ydot
        rss = np.sum((yt - yt.mean()) ** 2)
        ll.append(-n / 2 * np.log(rss / n))
    return float(lam[int(np.argmax(ll))])


def _transform(Qa, transform):
    y = np.asarray(Qa, dtype=float)
    lam = None
    if transform == "log":
        y = np.log(y)
    elif transform == "boxcox":
        lam = _boxcox_lambda(y)
        if abs(lam) < 0.01:
            lam = 0.0
            y = np.log(y)
        else:
            y = (y ** lam - 1) / lam
    elif transform != "none":
        raise ValueError('Accepted transformations are "log", "boxcox" and "none" only.')
    return y, lam


def inv_boxcox(x, lam):
    return np.exp(x) if lam == 0 else (x * lam + 1) ** (1 / lam)


def _make_y(years_Qa, obs, start_year, N):
    """R/LDS_reconstruction.R:179-183: centre and NA-pad to the study horizon."""
    end_year = start_year + N - 1
    if end_year < years_Qa[-1]:
        raise ValueError("The last year of u is earlier than the last year of the instrumental period.")
    mu = float(np.nanmean(obs))
    y = np.concatenate([np.full(int(years_Qa[0] - start_year), np.nan), obs - mu,
                        np.full(int(end_year - years_Qa[-1]), np.nan)])
    years = np.arange(start_year, end_year + 1)
    return y, mu, years


def _station(st, transform):
    """Host-side set-up of one station, no random draws: the argument checks of LDS_reconstruction / cvLDS,
    the transform, and y centred and NA-padded to the station's horizon (R/LDS_reconstruction.R:128-183)."""
    single, us, vs, N = _prep_uv(st.get("u"), st.get("v"))
    obs, lam = _transform(st["Qa"]["Qa"], transform)
    qyears = np.asarray(st["Qa"]["year"])
    y, mu, years = _make_y(qyears, obs, st["start_year"], N)
    return dict(Qa=st["Qa"], single=single, N=N, obs=obs, lam=lam, qyears=qyears, mu=mu, years=years,
                series=[_series(y, a, b) for a, b in zip(us, vs)])


def _pack(P, groups):
    """One em_batch over all stations.  groups: per station, its (member, held-out steps, initial thetas)
    groups in batch order; series are numbered station-major, theta rows padded to the widest series.
    Sets each station's first series / group / fit (s0, g0, f0) and its fit end f1; returns the em_batch
    arguments."""
    series, group_series, held, fit_group, th0 = [], [], [], [], []
    for S, gs in zip(P, groups):
        S.update(s0=len(series), g0=len(group_series), f0=len(fit_group))
        for m, h, init in gs:
            for t in init:
                th0.append(theta_to_vec(t))
                fit_group.append(len(group_series))
            group_series.append(S["s0"] + m)
            held.append(np.asarray(h, dtype=np.int64))
        series += S["series"]
        S["f1"] = len(fit_group)
    stride = max(s["p"] + s["q"] + 6 for s in series)
    return dict(series=series, group_series=group_series, held=held, fit_group=fit_group,
                theta0=np.stack([np.pad(v, (0, stride - v.size)) for v in th0]))


def _selected_thetas(r, best, series, group_series):
    """The selected fits' theta rows for a propagate_batch: a narrower series' padding is zeroed."""
    th = r["theta"][best].copy()
    for i, g in enumerate(group_series):
        s = series[g]
        th[i, s["p"] + s["q"] + 6:] = 0.0
    return th


def reconstruction_batch(stations, transform="log", num_restarts=50, rng=None):
    """Host half of LDS_reconstruction_stations, usable without a device: prepares every station, then, station
    by station, draws what that station's own LDS_reconstruction call draws (make_init per member unless the
    station gives `init`) and packs one em_batch (one group per member).  Returns (stations, em_batch args)."""
    rng = rng or np.random.default_rng()
    P = [_station(st, transform) for st in stations]
    groups = []
    for S, st in zip(P, stations):
        init = st.get("init")
        if init is None:
            init = [make_init(s["p"], s["q"], num_restarts, rng) for s in S["series"]]
        elif S["single"]:
            init = [init]
        S["init"] = init
        groups.append([(m, [], ini) for m, ini in enumerate(init)])
    return P, _pack(P, groups)


def LDS_reconstruction_stations(stations, method="EM", transform="log", num_restarts=50, return_init=False,
                                niter=1000, tol=1e-5, return_raw=False, rng=None, n_devices=1):
    """LDS_reconstruction for many stations in one batched GPU call.  stations: list of
    dict(Qa=dict(year=, Qa=), u=, v=, start_year=[, init=]); u / v as in LDS_reconstruction (matrix, None or an
    ensemble list); stations may differ in T, p, q, instrumental period and start year.  The other arguments
    are shared.  Random numbers are drawn station by station exactly as the single-station calls would draw
    them in that order.  Returns one LDS_reconstruction result per station.
    Device calls: one em_batch, one propagate_batch (return_raw), one construct_rec_stations."""
    if method != "EM":
        raise ValueError("only method = 'EM' is implemented (GA/BFGS are experimental in the reference)")
    P, B = reconstruction_batch(stations, transform, num_restarts, rng)
    r = _lib.em_batch(B["series"], B["group_series"], None, B["fit_group"], B["theta0"], niter, tol,
                      n_devices=n_devices)
    if np.any(r["status"] == _lib.FIT_SINGULAR):
        raise _lib.LdsrError(_lib.ERR_ARG, "LDS_reconstruction: inv(): matrix is singular")
    best = r["best"]
    if np.any(best < 0):
        raise _lib.LdsrError(_lib.ERR_ARG, "no restart produced a finite likelihood")
    ns = len(B["series"])
    # one group per series (member): group g == series g, and its winner's rows start at traj_ptr[g]
    fits = [_fit_dict(r, int(r["traj_ptr"][g]), B["series"][g]["y"].size) for g in range(ns)]
    thetas = [vec_to_theta(r["theta"][best[g]], B["series"][g]["p"], B["series"][g]["q"]) for g in range(ns)]
    raws = None
    if return_raw:
        pr = _lib.propagate_batch(B["series"], np.arange(ns), None, np.arange(ns),
                                  _selected_thetas(r, best, B["series"], range(ns)))
        raws = [dict(X=pr["X"][g], Y=pr["Y"][g], V=pr["V"][g]) for g in range(ns)]
    # construct_rec of every station's members in one launch; the raw trajectories are a second set of stations
    blocks = [(fs, range(S["s0"], S["s0"] + len(S["series"])), S) for fs in ([fits, raws] if return_raw else [fits])
              for S in P]
    rec = _lib.construct_rec_stations([np.stack([fs[g]["X"] for g in gs]) for fs, gs, _ in blocks],
                                      [np.stack([fs[g]["V"] for g in gs]) for fs, gs, _ in blocks],
                                      [np.stack([fs[g]["Y"] for g in gs]) for fs, gs, _ in blocks],
                                      [[thetas[g]["C"] for g in gs] for _, gs, _ in blocks],
                                      [[thetas[g]["R"] for g in gs] for _, gs, _ in blocks],
                                      [S["mu"] for _, _, S in blocks], transform, [S["lam"] for _, _, S in blocks])
    out = []
    for j, S in enumerate(P):
        members = []
        years = S["years"]

        def cols(o, k):
            d = dict(year=years)
            d.update({c: o[k, i] for i, c in enumerate(_lib.REC_COLUMNS)})
            return d
        for k in range(len(S["series"])):
            g = S["s0"] + k
            b = int(best[g])
            ans = dict(rec=cols(rec[j][0], k), theta=thetas[g], lik=float(r["lik"][b]))
            if return_raw:
                ans["rec2"] = cols(rec[len(P) + j][0], k)
            if return_init:
                ans["init"] = S["init"][k][b - S["f0"] - sum(len(i) for i in S["init"][:k])]
            if transform == "boxcox":
                ans["lambda"] = S["lam"]
            members.append(ans)
        if S["single"]:
            out.append(members[0])
            continue
        mean = rec[j][1]
        res = dict(rec=dict(year=years, X=mean[0], Q=mean[1]), ensemble=members)
        if return_raw:
            mean = rec[len(P) + j][1]
            res["rec_raw"] = dict(year=years, X=mean[0], Q=mean[1])
        out.append(res)
    return out


def LDS_reconstruction(Qa, u, v, start_year, method="EM", transform="log", init=None, num_restarts=50,
                       return_init=False, niter=1000, tol=1e-5, return_raw=False, rng=None, n_devices=1):
    """R/LDS_reconstruction.R:122-258.  Qa: dict(year=..., Qa=...).  Single model or ensemble
    (u, v lists); all members x restarts go to the GPU as one batch.  The one-station case of
    LDS_reconstruction_stations."""
    return LDS_reconstruction_stations([dict(Qa=Qa, u=u, v=v, start_year=start_year, init=init)], method, transform,
                                       num_restarts, return_init, niter, tol, return_raw, rng, n_devices)[0]


def one_lds_cv(z, instPeriod, mu, y, u, v, method="EM", num_restarts=20, niter=1000, tol=1e-6, use_raw=False,
               rng=None):
    """R/LDS_reconstruction.R:270-285.  z: 1-based indices into the instrumental period;
    instPeriod: 1-based indices of the instrumental period in the whole record."""
    rng = rng or np.random.default_rng()
    y = np.array(y, dtype=float).ravel()
    y[np.asarray(instPeriod)[np.asarray(z) - 1] - 1] = np.nan
    init = make_init(*_dims(u, v), num_restarts, rng)
    res = LDS_EM_restart(y, u, v, init, niter, tol, return_init=False)
    idx = np.asarray(instPeriod) - 1
    if use_raw:
        return propagate(res["theta"], u, v, y)["Y"][idx] + mu
    return res["fit"]["Y"][idx] + mu


def _nse(sim, obs):
    return 1 - np.sum((sim - obs) ** 2) / np.sum((obs - obs.mean()) ** 2)


def calculate_metrics(sim, obs, z):
    """R/utils.R:56-70 with the metric definitions of src/utils.cpp:13-97.  z is 1-based."""
    sim, obs = np.asarray(sim, dtype=float), np.asarray(obs, dtype=float)
    zi = np.asarray(z) - 1
    keep = np.ones(obs.size, dtype=bool)
    keep[zi] = False
    tr_obs, tr_sim = obs[keep], sim[keep]
    ok = ~np.isnan(tr_obs)
    tr_obs, tr_sim = tr_obs[ok], tr_sim[ok]
    vs, vo = sim[zi], obs[zi]
    rmse = np.sqrt(np.mean((vs - vo) ** 2))
    r = np.corrcoef(vs, vo)[0, 1] if vs.size > 1 else np.nan
    alpha, beta = np.std(vs, ddof=1) / np.std(vo, ddof=1) if vs.size > 1 else np.nan, vs.mean() / vo.mean()
    return dict(R2=_nse(tr_sim, tr_obs),
                RE=1 - np.sum((vs - vo) ** 2) / np.sum((vo - tr_obs.mean()) ** 2),
                CE=_nse(vs, vo), nRMSE=rmse / np.nanmean(obs),
                KGE=1 - np.sqrt((r - 1) ** 2 + (alpha - 1) ** 2 + (beta - 1) ** 2))


def tbrm(x, C=9.0):
    """Tukey's biweight robust mean, one step from the median, as dplR::tbrm (the reference's default
    aggregator of metrics.dist, R/LDS_reconstruction.R:397-398).  dplR is not part of the reference tree
    and is not installed here: this follows its published definition (Mosteller & Tukey 1977; weights
    (1 - u^2)^2 with u = (x - median)/(C * MAD + 1e-6), |u| < 1) -- unpinned.  The reference's stored NPcv
    result was aggregated with the plain mean (its `metrics` equal colMeans(metrics.dist))."""
    x = np.asarray(x, dtype=float)
    x = x[~np.isnan(x)]
    if x.size == 0:
        return float("nan")
    m = np.median(x)
    u = (x - m) / (C * np.median(np.abs(x - m)) + 1e-6)
    w = np.where(np.abs(u) < 1, (1 - u * u) ** 2, 0.0)
    return float(np.sum(w * x) / np.sum(w))


def cv_batch(stations, transform="log", num_restarts=50, rng=None):
    """Host half of cvLDS_stations, usable without a device: prepares every station, then, station by station,
    draws what that station's own cvLDS call draws -- make_Z if its Z is None, then make_init fold-major and
    member-minor (the reference's nested foreach order, R/LDS_reconstruction.R:373-381) -- and packs one
    em_batch (groups station-major, fold-major, member-minor).  Returns (stations, em_batch args)."""
    rng = rng or np.random.default_rng()
    P = [_station(st, transform) for st in stations]
    groups = []
    for S, st in zip(P, stations):
        Z = st.get("Z")
        if Z is None:
            Z = make_Z(S["Qa"]["Qa"], rng=rng)
        if not isinstance(Z, (list, tuple)):
            raise ValueError("Please provide the cross-validation folds (Z) in a list.")
        S["Z"] = Z
        S["inst"] = np.nonzero(np.isin(S["years"], S["qyears"]))[0]  # 0-based instPeriod
        groups.append([(m, S["inst"][np.asarray(z) - 1], make_init(s["p"], s["q"], num_restarts, rng))
                       for z in Z for m, s in enumerate(S["series"])])
    return P, _pack(P, groups)


def cvLDS_stations(stations, method="EM", transform="log", num_restarts=50, metric_space="original", use_raw=False,
                   niter=1000, tol=1e-5, rng=None, n_devices=1, use_robust_mean=True):
    """cvLDS for many stations in one batched GPU call.  stations: list of
    dict(Qa=dict(year=, Qa=), u=, v=, start_year=[, Z=]); u / v as in cvLDS (matrix, None or an ensemble list);
    stations may differ in T, p, q, instrumental period and start year.  The other arguments are shared.
    Random numbers are drawn station by station exactly as the single-station calls would draw them in that
    order.  Returns one cvLDS result per station.
    Device calls: one em_batch, one propagate_batch (use_raw), one cv_metrics_stations."""
    if method != "EM":
        raise ValueError("only method = 'EM' is implemented")
    P, B = cv_batch(stations, transform, num_restarts, rng)
    r = _lib.em_batch(B["series"], B["group_series"], B["held"], B["fit_group"], B["theta0"], niter, tol,
                      n_devices=n_devices)
    if np.any(r["status"] == _lib.FIT_SINGULAR):
        raise _lib.LdsrError(_lib.ERR_ARG, "cvLDS: inv(): matrix is singular")
    best = r["best"]
    for S in P:
        nm = len(S["series"])
        bad = np.nonzero(best[S["g0"]:S["g0"] + len(S["Z"]) * nm] < 0)[0]
        if bad.size:
            raise _lib.LdsrError(_lib.ERR_ARG, "fold %d: no restart produced a finite likelihood" % (bad[0] // nm))
    ng = len(B["group_series"])
    if use_raw:  # propagate(theta_best, u, v, y_fold)$Y (:279-281): the selected fits, open loop, in one call
        pr = _lib.propagate_batch(B["series"], B["group_series"], B["held"], np.arange(ng),
                                  _selected_thetas(r, best, B["series"], B["group_series"]))
        Yg = pr["Y"]
    else:
        Yg = [r["Y"][int(r["traj_ptr"][g]):int(r["traj_ptr"][g + 1])] for g in range(ng)]
    sims, targets = [], []
    for S in P:
        nm, inst, mu = len(S["series"]), S["inst"], S["mu"]
        Ycv = []
        for k in range(len(S["Z"])):
            g0 = S["g0"] + k * nm
            Ycv.append(np.mean([Yg[g0 + m][inst] + mu for m in range(nm)], axis=0))  # fit$Y[instPeriod] + mu,
        if metric_space == "original":                                              # .final = rowMeans (:379)
            if transform == "log":
                Ycv = [np.exp(a) for a in Ycv]
            elif transform == "boxcox":
                Ycv = [inv_boxcox(a, S["lam"]) for a in Ycv]
            target = np.asarray(S["Qa"]["Qa"], dtype=float)
        else:
            target = S["obs"]
        S["Ycv"], S["target"] = Ycv, target
        sims.append(np.stack(Ycv))
        targets.append(target)
    # mapply(calculate_metrics, ...) (:395) for all folds of all stations in one device call
    dists = _lib.cv_metrics_stations(sims, targets, [S["Z"] for S in P])
    keys = _lib.METRIC_NAMES
    mean_func = tbrm if use_robust_mean else np.mean  # R/LDS_reconstruction.R:397
    out = []
    for S, dist in zip(P, dists):
        metrics_dist = {k: dist[:, j].copy() for j, k in enumerate(keys)}
        g0, g1 = S["g0"], S["g0"] + len(S["Z"]) * len(S["series"])
        out.append(dict(metrics_dist=metrics_dist, metrics={k: float(mean_func(metrics_dist[k])) for k in keys},
                        target=dict(year=S["qyears"], y=S["target"]), Ycv=np.stack(S["Ycv"], axis=1), Z=S["Z"],
                        best=best[g0:g1] - S["f0"], lik=r["lik"][S["f0"]:S["f1"]], iters=r["iters"][S["f0"]:S["f1"]]))
    return out


def cvLDS(Qa, u, v, start_year, method="EM", transform="log", num_restarts=50, Z=None, metric_space="original",
          use_raw=False, niter=1000, tol=1e-5, rng=None, n_devices=1, use_robust_mean=True):
    """R/LDS_reconstruction.R:308-409.  All folds x members x restarts run as ONE batch; initial
    values are drawn fold-major exactly as `foreach(z = Z) ... one_lds_cv` would under
    registerDoSEQ (:373-381, :275).  use_raw: the fold output is the selected fit's open-loop
    propagate(theta, u, v, y_fold)$Y[instPeriod] + mu (:279-281).  The one-station case of cvLDS_stations."""
    return cvLDS_stations([dict(Qa=Qa, u=u, v=v, start_year=start_year, Z=Z)], method, transform, num_restarts,
                          metric_space, use_raw, niter, tol, rng, n_devices, use_robust_mean)[0]


# ---------------------------------------------------------------------------------------------
# Stochastic replicates (R/stochastics.R)
# ---------------------------------------------------------------------------------------------
def LDS_rep(theta, u=None, v=None, years=None, num_reps=100, mu=0.0, exp_trans=True, seed=0, z=None, r_seed=None):
    """R/stochastics.R:58-63.  Returns long-format columns like the reference's data.table
    (year, simX, simY, simQ, rep).  Noise: r_seed = s gives the replicates of `set.seed(s); LDS_rep(...)`
    in R (R's own stream, generated on the device); z (optional): [num_reps, 1+2n] standard normals in
    the reference's draw order; otherwise the counter-based device generator keyed by `seed`."""
    n = len(years)
    if u is None:  # is.null(u): both input terms are dropped (stochastics.R:28-32)
        v = None
    p, q = (0 if u is None else np.atleast_2d(u).shape[0]), (0 if v is None else np.atleast_2d(v).shape[0])
    th = np.concatenate([[theta["A"]], np.ravel(theta["B"])[:p], [theta["C"]], np.ravel(theta["D"])[:q],
                         [theta["Q"], theta["R"], theta["mu1"], theta["V1"]]]).astype(float)
    r = _lib.rep_batch(th, u, v, n, num_reps, z=z, seed=seed, mu=mu, exp_trans=exp_trans, p=p, q=q, r_seed=r_seed)
    return dict(year=np.tile(np.asarray(years), num_reps), simX=r["simX"].ravel(), simY=r["simY"].ravel(),
                simQ=r["simQ"].ravel(), rep=np.repeat(np.arange(1, num_reps + 1), n))


def LDS_rep_posterior(theta, Qa, u, v, start_year, transform="log", num_reps=100, seed=0, z=None):
    """Replicates conditioned on the observed record (beyond the reference): whole trajectories drawn from the
    smoothing distribution p(x | y, theta) of the model LDS_reconstruction fitted (forward filtering, backward
    sampling).  Each replicate passes through the observed flows, and its year-wise spread is the reconstruction's
    band, so path statistics (runs below a threshold, worst n-year means) can be read off them.
    theta: the fitted model (LDS_reconstruction(...)["theta"]), or a list of them for an ensemble with u / v lists.
    y, mu and lambda are prepared exactly as LDS_reconstruction prepares them.  Inputs follow Kalman_smoother:
    u = None drops B u and v = None drops D v (unlike LDS_rep, where u = None drops both).
    Noise: the device's counter-based generator keyed by (seed, member, replicate), or z: 2 * num_reps * sum(T)
    standard normals, member by member and replicate by replicate, T state draws then T observation draws each.
    Returns LDS_rep's long format (year, simX, simY, simQ, rep) over the station's horizon, one dict per member for
    an ensemble.  simY is on the centred, transformed scale; simQ = back-transform(simY + mu).  One device call."""
    S = _station(dict(Qa=Qa, u=u, v=v, start_year=start_year), transform)
    thetas = [theta] if S["single"] else list(theta)
    if len(thetas) != len(S["series"]):
        raise ValueError("theta must be one model per ensemble member (%d)" % len(S["series"]))
    rows = [theta_to_vec(t) for t in thetas]
    stride = max(s["p"] + s["q"] + 6 for s in S["series"])
    for s, r in zip(S["series"], rows):
        if r.size != s["p"] + s["q"] + 6:
            raise ValueError("theta has %d entries, the member's inputs need %d" % (r.size, s["p"] + s["q"] + 6))
    n = len(rows)
    r = _lib.posterior_rep_batch(S["series"], np.arange(n), None, np.arange(n),
                                 np.stack([np.pad(v, (0, stride - v.size)) for v in rows]), num_reps, z=z, seed=seed,
                                 mu=np.full(n, S["mu"]), transform=transform,
                                 lams=None if transform != "boxcox" else np.full(n, S["lam"]))
    years = S["years"]
    out = [dict(year=np.tile(years, num_reps), simX=r["simX"][k].ravel(), simY=r["simY"][k].ravel(),
                simQ=r["simQ"][k].ravel(), rep=np.repeat(np.arange(1, num_reps + 1), years.size)) for k in range(n)]
    return out[0] if S["single"] else out


def one_LDS_rep(rep_num, theta, u=None, v=None, years=None, mu=0.0, exp_trans=True, seed=0, z=None):
    """R/stochastics.R:18-47."""
    out = LDS_rep(theta, u, v, years, 1, mu, exp_trans, seed=seed + rep_num, z=None if z is None else z[None, :])
    out["rep"][:] = rep_num
    return out


def Kalman_smoother_d(y, u, v, theta, stdlik=True, method=1):
    """Kalman / RTS smoother for a state of dimension d = nrow(theta$A) in 2..4 (d = 1 works too).
    No counterpart in the reference, whose state is scalar (src/EM.cpp:20); same conventions as
    Kalman_smoother (src/EM.cpp:22-131).  theta: dict(A [d,d], B [d,p], C [d], D [q], Q [d,d], R, mu1 [d],
    V1 [d,d]).  method 1 = associative scan over time, 0 = sequential.  Returns dict(X [d,T], Y [T],
    V [T,d,d], lik) -- mirrors ldsr_b200.R::Kalman_smoother_d."""
    A = np.atleast_2d(np.asarray(theta["A"], dtype=float))
    d = A.shape[0]
    blocks = [A.ravel()]
    if u is not None:
        blocks.append(np.asarray(theta["B"], dtype=float).reshape(d, -1).ravel())
    blocks.append(np.asarray(theta["C"], dtype=float).ravel())
    if v is not None:
        blocks.append(np.asarray(theta["D"], dtype=float).ravel())
    blocks += [np.asarray(theta["Q"], dtype=float).reshape(d, d).ravel(), [float(np.ravel(theta["R"])[0])],
               np.asarray(theta["mu1"], dtype=float).ravel(), np.asarray(theta["V1"], dtype=float).reshape(d, d).ravel()]
    r = _lib.smoother_d(d, np.ravel(y), u, v, np.concatenate(blocks), stdlik=stdlik, method=method)
    return dict(X=r["X"][0].T, Y=r["Y"][0], V=r["V"][0], lik=float(r["lik"][0]))
