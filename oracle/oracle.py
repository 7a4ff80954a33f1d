"""ctypes front-end of oracle/libldsr_oracle.so (see the header of ldsr_oracle.c).

TEST INFRASTRUCTURE ONLY: importable from tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs.  The product package never imports this module.
"""
import ctypes as C
import os
import subprocess

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_SO = os.path.join(_HERE, "libldsr_oracle.so")
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)


def build(force=False):
    srcs = [os.path.join(_HERE, f) for f in ("ldsr_oracle.c", "ldsr_oracle_d.c")]
    if force or not os.path.exists(_SO) or os.path.getmtime(_SO) < max(os.path.getmtime(f) for f in srcs):
        subprocess.check_call(["make", "-C", _HERE, "-s"])
    return _SO


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        _lib = C.CDLL(_SO)
        for name in ("kalman_smoother", "mstep", "em", "select", "em_batch", "propagate", "rep",
                     "max_threads", "smoother_d", "cv_metrics", "construct_rec"):
            getattr(_lib, "ldsr_oracle_" + name).restype = C.c_int
    return _lib


def _d(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _i(a):
    return None if a is None else a.ctypes.data_as(_ip)


def _mat(m):
    """R-style p x T matrix (numpy [p, T]) -> column-major flat copy; None stays None."""
    if m is None:
        return None, 0
    m = np.asarray(m, dtype=np.float64)
    return np.ascontiguousarray(m.T).ravel(), m.shape[0]


def theta_flat(A, B, Cc, D, Q, R, mu1, V1):
    return np.concatenate([[A], np.ravel(B), [Cc], np.ravel(D), [Q, R, mu1, V1]]).astype(np.float64)


def theta_split(th, p, q):
    th = np.asarray(th)
    return dict(A=th[0], B=th[1:1 + p].copy(), C=th[1 + p], D=th[2 + p:2 + p + q].copy(),
                Q=th[2 + p + q], R=th[3 + p + q], mu1=th[4 + p + q], V1=th[5 + p + q])


def kalman_smoother(y, u, v, theta, p=None, q=None, stdlik=True):
    y = np.ascontiguousarray(y, dtype=np.float64).ravel()
    T = y.size
    uf, pu = _mat(u)
    vf, qv = _mat(v)
    p = pu if p is None else p
    q = qv if q is None else q
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    assert theta.size == p + q + 6
    X, Y, V, J = (np.empty(T) for _ in range(4))
    lik = C.c_double()
    rc = lib().ldsr_oracle_kalman_smoother(_d(y), _d(uf), _d(vf), T, p, q, _d(theta), int(stdlik),
                                           _d(X), _d(Y), _d(V), _d(J), C.byref(lik))
    if rc:
        raise RuntimeError("oracle kalman_smoother rc=%d" % rc)
    return dict(X=X, Y=Y, V=V, J=J, lik=lik.value)


def mstep(y, u, v, fit, p=None, q=None):
    y = np.ascontiguousarray(y, dtype=np.float64).ravel()
    T = y.size
    uf, pu = _mat(u)
    vf, qv = _mat(v)
    p = pu if p is None else p
    q = qv if q is None else q
    th = np.empty(p + q + 6)
    X, V, J = (np.ascontiguousarray(fit[k], dtype=np.float64) for k in ("X", "V", "J"))
    rc = lib().ldsr_oracle_mstep(_d(y), _d(uf), _d(vf), T, p, q, _d(X), _d(V), _d(J), _d(th))
    if rc:
        raise RuntimeError("oracle mstep rc=%d" % rc)
    return th


def em(y, u, v, theta0, niter=1000, tol=1e-5, p=None, q=None):
    y = np.ascontiguousarray(y, dtype=np.float64).ravel()
    T = y.size
    uf, pu = _mat(u)
    vf, qv = _mat(v)
    p = pu if p is None else p
    q = qv if q is None else q
    theta0 = np.ascontiguousarray(theta0, dtype=np.float64)
    assert theta0.size == p + q + 6
    th = np.empty(p + q + 6)
    X, Y, V, J = (np.empty(T) for _ in range(4))
    liks = np.full(niter, np.nan)
    n = C.c_int()
    lik = C.c_double()
    rc = lib().ldsr_oracle_em(_d(y), _d(uf), _d(vf), T, p, q, _d(theta0), int(niter),
                              C.c_double(tol), _d(th), _d(X), _d(Y), _d(V), _d(J), _d(liks),
                              C.byref(n), C.byref(lik))
    if rc:
        raise RuntimeError("oracle em rc=%d" % rc)
    return dict(theta=th, fit=dict(X=X, Y=Y, V=V, J=J, lik=lik.value), liks=liks[:n.value].copy(),
                lik=lik.value)


def select(liks, Cs):
    liks = np.ascontiguousarray(liks, dtype=np.float64)
    Cs = np.ascontiguousarray(Cs, dtype=np.float64)
    return lib().ldsr_oracle_select(_d(liks), _d(Cs), liks.size)


def em_batch(series, group_series, held, fit_group, theta0, niter=1000, tol=1e-5, n_threads=0):
    """series: list of dict(y=[T], u=[p,T]|None, v=[q,T]|None, p=, q=) ; held: list of int arrays
    (0-based step indices per group); theta0: [n_fits, th_stride].  Returns dict of arrays."""
    ns = len(series)
    ys, us, vs, Ts, ps, qs = [], [], [], [], [], []
    for s in series:
        y = np.ascontiguousarray(s["y"], dtype=np.float64).ravel()
        uf, pu = _mat(s.get("u"))
        vf, qv = _mat(s.get("v"))
        ys.append(y)
        us.append(uf)
        vs.append(vf)
        Ts.append(y.size)
        ps.append(s.get("p", pu))
        qs.append(s.get("q", qv))
    Ta, pa, qa = (np.asarray(a, dtype=np.int32) for a in (Ts, ps, qs))
    PP = _dp * ns
    yp = PP(*[_d(a) for a in ys])
    up = PP(*[C.cast(_d(a), _dp) if a is not None else C.cast(None, _dp) for a in us])
    vp = PP(*[C.cast(_d(a), _dp) if a is not None else C.cast(None, _dp) for a in vs])
    group_series = np.ascontiguousarray(group_series, dtype=np.int32)
    ng = group_series.size
    hp = np.zeros(ng + 1, dtype=np.int32)
    hp[1:] = np.cumsum([len(h) for h in held])
    hi = (np.concatenate([np.asarray(h, dtype=np.int32) for h in held]) if hp[-1] > 0
          else np.zeros(1, dtype=np.int32)).astype(np.int32)
    fit_group = np.ascontiguousarray(fit_group, dtype=np.int32)
    nf = fit_group.size
    theta0 = np.ascontiguousarray(theta0, dtype=np.float64)
    stride = theta0.shape[1]
    th = np.full_like(theta0, np.nan)
    lik = np.empty(nf)
    iters = np.empty(nf, dtype=np.int32)
    status = np.empty(nf, dtype=np.int32)
    best = np.empty(ng, dtype=np.int32)
    rc = lib().ldsr_oracle_em_batch(ns, _i(Ta), _i(pa), _i(qa), yp, up, vp, ng, _i(group_series),
                                    _i(hp), _i(hi), nf, _i(fit_group), _d(theta0), stride,
                                    int(niter), C.c_double(tol), _d(th), _d(lik), _i(iters),
                                    _i(status), _i(best), int(n_threads))
    if rc:
        raise RuntimeError("oracle em_batch rc=%d" % rc)
    return dict(theta=th, lik=lik, iters=iters, status=status, best=best)


def propagate(theta, u, v, y, p=None, q=None, stdlik=True, T=None):
    y = np.ascontiguousarray(y, dtype=np.float64).ravel()
    uf, pu = _mat(u)
    vf, qv = _mat(v)
    p = pu if p is None else p
    q = qv if q is None else q
    T = y.size if T is None else T
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    X, Y, V = (np.empty(T) for _ in range(3))
    lik = C.c_double()
    rc = lib().ldsr_oracle_propagate(_d(theta), _d(uf), _d(vf), _d(y), T, p, q, int(stdlik), _d(X),
                                     _d(Y), _d(V), C.byref(lik))
    if rc:
        raise RuntimeError("oracle propagate rc=%d" % rc)
    return dict(X=X, Y=Y, V=V, lik=lik.value)


def rep(theta, u, v, n, z, mu=0.0, exp_trans=True, p=None, q=None):
    uf, pu = _mat(u)
    vf, qv = _mat(v)
    p = pu if p is None else p
    q = qv if q is None else q
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    z = np.ascontiguousarray(z, dtype=np.float64)
    assert z.size == 1 + 2 * n
    sx, sy, sq = (np.empty(n) for _ in range(3))
    lib().ldsr_oracle_rep(_d(theta), _d(uf), _d(vf), n, p, q, _d(z), C.c_double(mu), int(exp_trans),
                          _d(sx), _d(sy), _d(sq))
    return dict(simX=sx, simY=sy, simQ=sq)


def max_threads():
    return lib().ldsr_oracle_max_threads()


def theta_d_flat(A, B, Cc, D, Q, R, mu1, V1):
    """General-d theta: [A d*d | B d*p | C d | D q | Q d*d | R | mu1 d | V1 d*d] (row-major blocks)."""
    return np.concatenate([np.ravel(A), np.ravel(B), np.ravel(Cc), np.ravel(D), np.ravel(Q), [R],
                           np.ravel(mu1), np.ravel(V1)]).astype(np.float64)


def smoother_d(d, y, u, v, theta, stdlik=True):
    """General state dimension d (ldsr_oracle_d.c).  u [p,T] | None, v [q,T] | None."""
    y = np.ascontiguousarray(y, dtype=np.float64).ravel()
    T = y.size
    uf, p = _mat(u)
    vf, q = _mat(v)
    th = np.ascontiguousarray(theta, dtype=np.float64)
    assert th.size == 2 * d * d + d * p + d + q + 1 + d + d * d, th.size
    X = np.empty((T, d))
    V = np.empty((T, d, d))
    Y = np.empty(T)
    lik = C.c_double()
    rc = lib().ldsr_oracle_smoother_d(int(d), T, int(p), int(q), _d(y), _d(uf), _d(vf), _d(th), int(bool(stdlik)),
                                      _d(X), _d(V), _d(Y), C.byref(lik))
    if rc != 0:
        raise RuntimeError("ldsr_oracle_smoother_d failed: %d" % rc)
    return dict(X=X, V=V, Y=Y, lik=lik.value)


METRIC_NAMES = ("R2", "RE", "CE", "nRMSE", "KGE")


def cv_metrics(sim, obs, Z, exp_trans=False):
    """calculate_metrics for every fold (R/utils.R:56-70, src/utils.cpp:13-97).  sim [n_folds, n];
    obs [n]; Z list of 1-based index vectors.  Returns [n_folds, 5] in METRIC_NAMES order."""
    sim = np.ascontiguousarray(sim, dtype=np.float64)
    obs = np.ascontiguousarray(obs, dtype=np.float64)
    nf, n = sim.shape
    zp = np.zeros(nf + 1, dtype=np.int32)
    zp[1:] = np.cumsum([len(z) for z in Z])
    zi = np.concatenate([np.asarray(z, dtype=np.int32) for z in Z]).astype(np.int32)
    out = np.empty((nf, 5))
    rc = lib().ldsr_oracle_cv_metrics(int(n), int(nf), _d(sim), _d(obs), _i(zp), _i(zi), int(bool(exp_trans)), _d(out))
    if rc != 0:
        raise RuntimeError("ldsr_oracle_cv_metrics failed: %d" % rc)
    return out


REC_COLUMNS = ("X", "Xl", "Xu", "Q", "Ql", "Qu")
TRANSFORMS = {"none": 0, "log": 1, "boxcox": 2}


def construct_rec(X, V, Y, C_, R_, mu, transform="log", lam=0.0):
    """construct_rec for every ensemble member + the year-wise ensemble mean of X and Q
    (R/LDS_reconstruction.R:190-212, 247-248).  X, V, Y: [n, T]; C_, R_: [n].  Returns
    (out [n, 6, T] in REC_COLUMNS order, mean [2, T])."""
    X, V, Y = (np.ascontiguousarray(np.atleast_2d(a), dtype=np.float64) for a in (X, V, Y))
    n, T = X.shape
    Cv = np.ascontiguousarray(np.broadcast_to(np.asarray(C_, dtype=np.float64).ravel(), (n,)))
    Rv = np.ascontiguousarray(np.broadcast_to(np.asarray(R_, dtype=np.float64).ravel(), (n,)))
    out = np.empty((n, 6, T))
    mean = np.empty((2, T))
    rc = lib().ldsr_oracle_construct_rec(int(n), int(T), _d(X), _d(V), _d(Y), _d(Cv), _d(Rv), C.c_double(mu),
                                         int(TRANSFORMS[transform]), C.c_double(lam), _d(out), _d(mean))
    if rc != 0:
        raise RuntimeError("ldsr_oracle_construct_rec failed: %d" % rc)
    return out, mean


def objective(y, u, v, theta_vec, kind, lam=1.0, p=None, q=None):
    """The experimental learners' objectives (R/LDS_GA.R:28-44, 136-147) from the oracle's
    Kalman_smoother / propagate.  theta_vec is the reference's flat order (vec_to_list, R/LDS_GA.R:6-16);
    p / q give its widths when u / v is None but theta still has B / D entries."""
    y = np.asarray(y, dtype=np.float64).ravel()
    if kind == "penalized_likelihood":
        s = kalman_smoother(y, u, v, theta_vec, p=p, q=q, stdlik=False)
        p = (0 if u is None else np.asarray(u).shape[0]) if p is None else p
        A, B = theta_vec[0], np.asarray(theta_vec[1:1 + p])
        X = s["X"]
        Bu = B @ np.asarray(u)[:, :-1] if u is not None else 0.0
        return s["lik"] - lam * float(np.sum((X[1:] - A * X[:-1] - Bu) ** 2))
    pr = propagate(theta_vec, u, v, y, p=p, q=q)
    if kind == "negLogLik":
        return -pr["lik"]
    return float(np.nansum((y - pr["Y"]) ** 2))
