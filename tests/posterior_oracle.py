"""CPU reference for replicates conditioned on the observed record (forward filtering, backward sampling), used by
tests/test_posterior_rep_host.py and tests/test_gpu_posterior_rep.py.  Never imported by the product.

The filter restates Kalman_smoother's forward pass (src/EM.cpp:43-90, the operation order of oracle/ldsr_oracle.c's
smoother_core): Xp_0 = mu1, Vp_0 = V1, u with one step of lag, v without, the update only where y is not NaN.
Then, for t = T-1 down to 0 (x_T taken as 0):
    J_t = Vu_t A / Vp_{t+1},  m_t = Xu_t - J_t Xp_{t+1},  s_t = sqrt(Vu_t Q / Vp_{t+1});  t = T-1: 0, Xu, sqrt(Vu)
    x_t = m_t + J_t x_{t+1} + s_t zeta_t
    simY_t = y_t where observed, else C x_t + D v_t + sqrt(R) eps_t
    simQ_t = back-transform(simY_t + mu): none, exp, or inverse Box-Cox (lambda; 0 means exp)
The backward walk is vectorised over replicates."""
import numpy as np


def _filter(y, u, v, th, p, q):
    A, B, C = th[0], th[1:1 + p], th[1 + p]
    D, Q, R, mu1, V1 = th[2 + p:2 + p + q], th[2 + p + q], th[3 + p + q], th[4 + p + q], th[5 + p + q]
    T = y.size
    Xp, Vp, Xu, Vu, Dv = (np.empty(T) for _ in range(5))
    for k in range(T):
        Dv[k] = sum(D[j] * v[j, k] for j in range(q)) if v is not None else 0.0
        if k == 0:
            Xp[k], Vp[k] = mu1, V1
        else:
            Bu = sum(B[j] * u[j, k - 1] for j in range(p)) if u is not None else 0.0
            Xp[k] = A * Xu[k - 1] + Bu
            Vp[k] = A * Vu[k - 1] * A + Q
        if np.isnan(y[k]):
            Xu[k], Vu[k] = Xp[k], Vp[k]
        else:
            K = Vp[k] * C * (1.0 / (C * Vp[k] * C + R))
            Xu[k] = Xp[k] + K * (y[k] - (C * Xp[k] + Dv[k]))
            Vu[k] = (1.0 - K * C) * Vp[k]
    return Xp, Vp, Xu, Vu, Dv


def posterior_rep(theta, y, u, v, z, mu=0.0, transform="log", lam=0.0, held=None, p=None, q=None):
    """theta: flat [A, B, C, D, Q, R, mu1, V1]; y [T] with NaN = missing; held: steps also treated as missing;
    u [p, T] / v [q, T] or None (p / q give theta's widths then); z [..., 2T]: T state draws, then T observation
    draws per replicate.  Returns simX, simY, simQ shaped like z[..., :T]."""
    y = np.array(y, dtype=float).ravel()
    if held is not None and len(held):
        y[np.asarray(held, dtype=np.int64)] = np.nan
    T = y.size
    u = None if u is None else np.atleast_2d(np.asarray(u, dtype=float))
    v = None if v is None else np.atleast_2d(np.asarray(v, dtype=float))
    p = u.shape[0] if p is None else p
    q = v.shape[0] if q is None else q
    th = np.asarray(theta, dtype=float)
    assert th.size == p + q + 6
    A, C, Q, R = th[0], th[1 + p], th[2 + p + q], th[3 + p + q]
    Xp, Vp, Xu, Vu, Dv = _filter(y, u, v, th, p, q)
    z = np.asarray(z, dtype=float)
    assert z.shape[-1] == 2 * T
    simX, simY = np.empty(z.shape[:-1] + (T,)), np.empty(z.shape[:-1] + (T,))
    x1 = np.zeros(z.shape[:-1])
    for k in range(T - 1, -1, -1):
        if k == T - 1:
            J, m, s = 0.0, Xu[k], np.sqrt(Vu[k])
        else:
            J = Vu[k] * A / Vp[k + 1]
            m = Xu[k] - J * Xp[k + 1]
            s = np.sqrt(Vu[k] * Q / Vp[k + 1])
        x = m + J * x1 + s * z[..., k]
        simX[..., k] = x
        simY[..., k] = C * x + Dv[k] + np.sqrt(R) * z[..., T + k] if np.isnan(y[k]) else y[k]
        x1 = x
    yq = simY + mu
    if transform == "none":
        simQ = yq
    elif transform == "log" or lam == 0.0:
        simQ = np.exp(yq)
    else:
        with np.errstate(invalid="ignore"):
            simQ = (yq * lam + 1.0) ** (1.0 / lam)
    return dict(simX=simX, simY=simY, simQ=simQ)
