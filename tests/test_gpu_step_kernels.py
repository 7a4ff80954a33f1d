"""The single-step kernels of aux_kernels.cuh -- smoother_kernel (Kalman_smoother, penalized_likelihood),
mstep_kernel (Mstep), propagate_kernel (propagate, negLogLik, ssqTrain) and rep_kernel (LDS_rep) -- at every
compiled input width, against the oracle on the same inputs.

Each width case is one batch: several series of different lengths (below, at and above the smoother's block of
BK steps and the 32-step mask word), groups listed out of series order, a different hold-out set per group and
several theta per group, so that the host-side row mapping (internal vs caller order) is exercised as well.
Each call is one pass of a recursion, not an EM run, so the bars are those of one E-step:
  rows X, Y, V, J: relative 1e-10, with an absolute floor of 1e-12 x the row's largest |value| (Y can cancel);
  lik and objectives: relative 1e-10;  M-step theta: relative 1e-9 with a floor of 1e-8.
Run with -s to see the largest deviation from the oracle per width and kernel."""
import numpy as np
import pytest

from ldsr_b200 import _lib
from oracle import oracle as O

pytestmark = pytest.mark.gpu

ROW_RTOL, ROW_FLOOR = 1e-10, 1e-12
LIK_RTOL = 1e-10
THETA_RTOL, THETA_FLOOR = 1e-9, 1e-8

PQ_LIST = (1, 2, 3, 4, 5, 6, 7, 8, 10, 12, 16, 24, 32)  # the compiled widths (build.py)

# (p, q, form): every padded width, every steps-per-block class of smoother_kernel, exact and padded widths, and
# v == u (one input set read twice: SeriesDev.same_uv) as well as v != u.  "unone": u = None with p = 1 declared
# (theta still carries a B entry); "vnone": v = None with q declared.
WIDTHS = [(1, 1, "vu"), (2, 1, "sep"), (3, 3, "vu"), (1, 3, "unone"), (3, 2, "vnone"), (4, 2, "sep"), (5, 5, "vu"),
          (6, 3, "sep"), (7, 7, "vu"), (8, 5, "sep"), (9, 9, "vu"), (11, 4, "sep"), (13, 13, "vu"), (16, 16, "vu"),
          (20, 17, "sep"), (24, 24, "vu"), (29, 32, "sep"), (32, 32, "vu")]
HOLD_KINDS = ("none", "first", "last", "word", "scattered", "fewobs")


def case_id(w):
    return "p%dq%d_%s" % w


def padded_width(p, q, form):
    need = max(1, 0 if form == "unone" else p, 0 if form == "vnone" else q)
    return next(w for w in PQ_LIST if w >= need)


def steps_per_block(pq):
    return 8 if pq <= 3 else (4 if pq <= 6 else (2 if pq <= 12 else 1))  # BK of smoother_kernel


def rand_theta(rng, p, q):
    sign = rng.choice([-1.0, 1.0])
    return np.concatenate([[rng.uniform(-0.9, 0.9)], rng.uniform(-1, 1, p) * 0.5 / np.sqrt(p),
                           [sign * rng.uniform(0.3, 1.2)], rng.uniform(-1, 1, q) * 0.5 / np.sqrt(q),
                           [rng.uniform(0.2, 1.5), rng.uniform(0.3, 1.0), rng.normal(), rng.uniform(0.5, 2.0)]])


def make_series(rng, p, q, form, T):
    u = rng.standard_normal((p, T))
    v = u if form == "vu" else rng.standard_normal((q, T))
    x = np.zeros(T)
    for t in range(1, T):
        x[t] = 0.7 * x[t - 1] + 0.2 * u[0, t - 1] + 0.5 * rng.standard_normal()
    y = 0.8 * x + 0.1 * v[0] + 0.3 * rng.standard_normal(T)
    if T >= 31:  # an unobserved lead (the reconstruction period) and a gap inside the record
        y[:T // 3] = np.nan
        y[T // 2] = np.nan
    return dict(y=y, u=None if form == "unone" else u, v=None if form == "vnone" else v, p=p, q=q)


def holdout(rng, y, kind):
    T = y.size
    if kind == "first":
        h = [0]
    elif kind == "last":
        h = [T - 1]
    elif kind == "word" and T > 32:
        h = list(range(32, 64)) if T >= 65 else list(range(32))
    elif kind in ("word", "scattered"):
        h = list(rng.choice(T, max(1, T // 5), replace=False))
    elif kind == "fewobs":  # all but three observed steps
        obs = np.nonzero(np.isfinite(y))[0]
        h = list(np.setdiff1d(obs, rng.choice(obs, min(3, obs.size), replace=False)))
    else:
        h = []
    h = np.unique(np.asarray(h, dtype=int))
    left = np.setdiff1d(np.nonzero(np.isfinite(y))[0], h)
    if left.size == 0:  # keep one observed step, so that the likelihood is defined
        h = h[h != np.nonzero(np.isfinite(y))[0][-1]]
    return h


def make_case(p, q, form, seed):
    rng = np.random.default_rng(seed)
    bk = steps_per_block(padded_width(p, q, form))
    Ts = sorted({T for T in (2, 3, bk - 1, bk, bk + 1, 31, 32, 33, 65, 213) if T >= 2})
    series = [make_series(rng, p, q, form, T) for T in Ts]
    pairs = []
    for s, T in enumerate(Ts):
        kinds = HOLD_KINDS if T >= 65 else [HOLD_KINDS[(s + k) % len(HOLD_KINDS)] for k in range(3)]
        pairs += [(s, k) for k in kinds]
    rng.shuffle(pairs)  # groups out of series order
    group_series = np.array([s for s, _ in pairs], dtype=np.int32)
    held = [holdout(rng, series[s]["y"], k) for s, k in pairs]
    fit_group = np.repeat(np.arange(len(pairs)), [2 + g % 2 for g in range(len(pairs))])
    theta = np.stack([rand_theta(rng, p, q) for _ in fit_group])
    return dict(series=series, group_series=group_series, held=held, fit_group=fit_group, theta=theta)


def group_y(c, g):
    s = c["series"][c["group_series"][g]]
    y = np.array(s["y"], dtype=float)
    y[c["held"][g]] = np.nan
    return s, y


def oracle_smoother(c, f, stdlik=True):
    s, y = group_y(c, c["fit_group"][f])
    return O.kalman_smoother(y, s["u"], s["v"], c["theta"][f], p=s["p"], q=s["q"], stdlik=stdlik)


def row_dev(a, b):
    """Largest |a - b| in units of max(|b|, 1e-2 x max|b|): below ROW_RTOL means relative 1e-10 with an absolute
    floor of 1e-12 x the row's largest value.  NaN must be in the same places."""
    a, b = np.asarray(a), np.asarray(b)
    assert a.shape == b.shape and np.array_equal(np.isnan(a), np.isnan(b))
    ok = ~np.isnan(b)
    if not ok.any():
        return 0.0
    top = np.max(np.abs(b[ok]))
    if top == 0.0:
        return 0.0 if np.array_equal(a[ok], b[ok]) else np.inf
    return float(np.max(np.abs(a[ok] - b[ok]) / np.maximum(np.abs(b[ok]), ROW_FLOOR / ROW_RTOL * top)))


def rel_dev(a, b):
    a, b = np.asarray(a, dtype=float), np.asarray(b, dtype=float)
    return float(np.max(np.abs(a - b) / np.abs(b)))


def report(kernel, width, dev):
    print("\n[max deviation] %s %s PQ=%d: %s" % (kernel, case_id(width), padded_width(*width),
                                                 ", ".join("%s %.1e" % kv for kv in dev.items())))


def width_seed(width):
    return 1000 + WIDTHS.index(width)


@pytest.mark.parametrize("stdlik", [True, False])
@pytest.mark.parametrize("width", WIDTHS, ids=case_id)
def test_smoother_batch_matches_the_oracle(width, stdlik):
    c = make_case(*width, seed=width_seed(width))
    g = _lib.smoother_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], stdlik=stdlik)
    dev = dict(X=0.0, Y=0.0, V=0.0, J=0.0, lik=0.0)
    for f in range(len(c["fit_group"])):
        o = oracle_smoother(c, f, stdlik)
        for k in "XYVJ":
            d = row_dev(g[k][f], o[k])
            assert d < ROW_RTOL, (f, k, d)
            dev[k] = max(dev[k], d)
        d = rel_dev(g["lik"][f], o["lik"])
        assert d < LIK_RTOL, (f, d)
        dev["lik"] = max(dev["lik"], d)
    report("smoother stdlik=%d" % stdlik, width, dev)


def _singular_series(rng, p, q, form):
    """A series whose Gram block of u (or of v, without u) is exactly singular: its first two input rows are the same
    +-1 vector (one row: all zeros) and 64 steps enter each block, so the Cholesky pivot is exactly 0 whatever the
    summation order.  T = 65 with y[0] missing: Tuu sums t < T - 1, Svv the 64 observed steps."""
    s = make_series(rng, p, q, form, 65)
    y = 0.3 * rng.standard_normal(65)
    y[0] = np.nan
    s["y"] = y
    m = s["u"] if s["u"] is not None else s["v"]
    if m.shape[0] == 1:
        m[0] = 0.0
    else:
        m[0] = m[1] = rng.choice([-1.0, 1.0], 65)
    return s


@pytest.mark.parametrize("width", WIDTHS, ids=case_id)
def test_mstep_batch_matches_the_oracle(width):
    p, q, form = width
    rng = np.random.default_rng(width_seed(width) + 500)
    c = make_case(p, q, form, seed=width_seed(width))
    # groups with at least 3 max(p, q) observed steps and transitions: well-conditioned Gram blocks
    need = 3 * max(p, q)
    keep = [g for g in range(len(c["group_series"]))
            if np.isfinite(group_y(c, g)[1]).sum() >= need and c["series"][c["group_series"][g]]["y"].size - 1 >= need]
    assert len(keep) >= 2
    series = c["series"] + [_singular_series(rng, p, q, form)]
    gs = [c["group_series"][g] for g in keep]
    held = [c["held"][g] for g in keep]
    gs.insert(1, len(series) - 1)  # the singular group between two others
    held.insert(1, np.array([], dtype=int))
    groups = [np.nonzero(c["fit_group"] == g)[0] for g in keep]
    th = [c["theta"][f] for f in groups[0]] + [rand_theta(rng, p, q) for _ in range(2)] + \
         [c["theta"][f] for fs in groups[1:] for f in fs]
    fg = np.repeat(np.arange(len(gs)), [groups[0].size, 2] + [fs.size for fs in groups[1:]])
    m = dict(series=series, group_series=np.array(gs, dtype=np.int32), held=held, fit_group=fg, theta=np.stack(th))
    rows = [oracle_smoother(m, f) for f in range(fg.size)]
    g = _lib.mstep_batch(series, m["group_series"], held, fg, [r["X"] for r in rows], [r["V"] for r in rows],
                         [r["J"] for r in rows], p + q + 6)
    dev = 0.0
    for f in range(fg.size):
        if fg[f] == 1:
            assert g["status"][f] == _lib.FIT_SINGULAR, f
            continue
        assert g["status"][f] == _lib.FIT_OK, f
        s, y = group_y(m, fg[f])
        o = O.mstep(y, s["u"], s["v"], rows[f], p=p, q=q)
        d = float(np.max(np.abs(g["theta"][f] - o) / np.maximum(np.abs(o), THETA_FLOOR)))
        assert d < THETA_RTOL, (f, d, np.argmax(np.abs(g["theta"][f] - o) / np.maximum(np.abs(o), THETA_FLOOR)))
        dev = max(dev, d)
    report("mstep", width, dict(theta=dev))


@pytest.mark.parametrize("stdlik", [True, False])
@pytest.mark.parametrize("width", WIDTHS, ids=case_id)
def test_propagate_batch_matches_the_oracle(width, stdlik):
    c = make_case(*width, seed=width_seed(width))
    g = _lib.propagate_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], stdlik=stdlik)
    dev = dict(X=0.0, Y=0.0, V=0.0, lik=0.0)
    for f in range(len(c["fit_group"])):
        s, y = group_y(c, c["fit_group"][f])
        o = O.propagate(c["theta"][f], s["u"], s["v"], y, p=s["p"], q=s["q"], stdlik=stdlik)
        for k in "XYV":
            d = row_dev(g[k][f], o[k])
            assert d < ROW_RTOL, (f, k, d)
            dev[k] = max(dev[k], d)
        d = rel_dev(g["lik"][f], o["lik"])
        assert d < LIK_RTOL, (f, d)
        dev["lik"] = max(dev["lik"], d)
    report("propagate stdlik=%d" % stdlik, width, dev)


@pytest.mark.parametrize("width", WIDTHS, ids=case_id)
def test_objectives_match_the_oracle(width):
    p, q, _ = width
    c = make_case(*width, seed=width_seed(width))
    dev = {}
    for kind in ("penalized_likelihood", "negLogLik", "ssqTrain"):
        for lam in (1.0, 0.25):
            g = _lib.objective_batch(c["series"], c["group_series"], c["held"], c["fit_group"], c["theta"], kind, lam)
            o = []
            for f in range(len(c["fit_group"])):
                s, y = group_y(c, c["fit_group"][f])
                o.append(O.objective(y, s["u"], s["v"], c["theta"][f], kind, lam, p=p, q=q))
            d = rel_dev(g, o)
            assert d < LIK_RTOL, (kind, lam, d)
            dev["%s/%g" % (kind, lam)] = d
    report("objective", width, dev)


REP_WIDTHS = [(3, 3, "vu"), (1, 3, "unone"), (3, 2, "vnone"), (5, 5, "vu"), (6, 3, "sep"), (9, 9, "vu"),
              (11, 4, "sep"), (16, 16, "vu"), (29, 32, "sep"), (32, 32, "vu")]
ALL_OUT = ("simX", "simY", "simQ")
# (n, n_reps, exp_trans, want): n against the 16-step tile, n_reps for partial warps and several CTAs of 128,
# fewer requested outputs than three (the output indexing)
REP_RUNS = [(1, 33, True, ALL_OUT), (15, 129, False, ("simQ",)), (16, 1, True, ("simX", "simQ")),
            (17, 31, False, ALL_OUT), (33, 300, True, ("simX", "simQ")), (813, 129, False, ("simQ",)),
            (813, 31, True, ALL_OUT)]


@pytest.mark.parametrize("width", REP_WIDTHS, ids=case_id)
def test_rep_batch_with_caller_noise_matches_the_oracle(width):
    p, q, form = width
    rng = np.random.default_rng(width_seed(width) + 900)
    dev = dict.fromkeys(ALL_OUT, 0.0)
    for n, n_reps, exp_trans, want in REP_RUNS:
        u = None if form == "unone" else rng.standard_normal((p, n))
        v = None if form == "vnone" else (u if form == "vu" else rng.standard_normal((q, n)))
        th = rand_theta(rng, p, q)
        mu = 0.37 if exp_trans else -1.3
        z = rng.standard_normal((n_reps, 1 + 2 * n))
        r = _lib.rep_batch(th, u, v, n, n_reps, z=z, mu=mu, exp_trans=exp_trans, p=p, q=q, want=want)
        assert set(r) == set(want) | {"device_ms"}
        for i in range(n_reps):
            o = O.rep(th, u, v, n, z[i], mu=mu, exp_trans=exp_trans, p=p, q=q)
            for k in want:
                d = row_dev(r[k][i], o[k])
                assert d < ROW_RTOL, (n, n_reps, i, k, d)
                dev[k] = max(dev[k], d)
    report("rep", width, dev)
