"""CPU reference for the per-step quantiles of w-step mean flows over conditioned replicates
(ldsr_posterior_quantile_batch), used by tests/test_posterior_quantile_host.py and tests/test_gpu_posterior_quantile.py.
Never imported by the product.

From a [n_reps, T] array of back-transformed flows Q and a step range [lo, hi), per window w and start t with
lo <= t <= hi - w: the window value of each replicate is S / w, where S is the kernel's running sum replayed step by
step (one IEEE add, one subtract and one divide, in the kernel's order, so the values are the kernel's bit for bit):
S starts at 0 at step hi - 1 and walks downwards, at step t S = (S + qf_t) - qf_{t+w}, the subtraction only once more
than w steps have been walked, qf being Q with non-finite flows replaced by 0.  A window that holds a non-finite flow
has no value.  The quantile at level p is the r-th smallest of the n values, r = max(1, ceil(p n)) (numpy's
method="inverted_cdf"); NaN when n = 0.  Outside the range and at starts past hi - w: q NaN, nonfinite -1."""
import math

import numpy as np


def window_means(Q, w, lo, hi):
    """Q [n, T] -> (M [n, hi - lo - w + 1], ok [same]): the kernel's window values at starts lo .. hi - w and whether
    the window's flows are all finite."""
    Qr = np.asarray(Q, dtype=np.float64)[:, lo:hi]
    fin = np.isfinite(Qr)
    qf = np.where(fin, Qr, 0.0)
    n, m = Qr.shape
    M = np.full((n, m - w + 1), np.nan)
    S = np.zeros(n)
    for j in range(m - 1, -1, -1):  # step lo + j; m - j steps of the range walked
        seen = m - j
        S = S + qf[:, j]
        if seen > w:
            S = S - qf[:, j + w]
        if seen >= w:
            M[:, j] = S / float(w)
    ok = np.lib.stride_tricks.sliding_window_view(fin, w, axis=1).all(axis=2)
    return M, ok


def rank(p, n):
    """The 1-based rank of level p among n values, in IEEE double as the library evaluates it."""
    return max(1, int(math.ceil(float(p) * float(n))))


def quantiles(Q, windows, levels, lo, hi):
    """Q [n_reps, T] -> dict(q [n_windows, n_levels, T], nonfinite [n_windows, T] int64)."""
    Q = np.atleast_2d(np.asarray(Q, dtype=np.float64))
    n_reps, T = Q.shape
    q = np.full((len(windows), len(levels), T), np.nan)
    nonfinite = np.full((len(windows), T), -1, np.int64)
    for k, w in enumerate(windows):
        if w > hi - lo:
            continue
        M, ok = window_means(Q, w, lo, hi)
        vals = np.sort(np.where(ok, M, np.inf), axis=0)  # the values first, ascending, per start
        cnt = ok.sum(axis=0)
        nonfinite[k, lo:hi - w + 1] = n_reps - cnt
        for j in range(M.shape[1]):
            if cnt[j] == 0:
                continue
            for l, p in enumerate(levels):
                q[k, l, lo + j] = vals[rank(p, cnt[j]) - 1, j]
    return dict(q=q, nonfinite=nonfinite)


def assert_match(got, Q, windows, levels, lo, hi, where=""):
    """Outputs of one fit from the library or the emulator (q [n_windows, n_levels, T], nonfinite [n_windows, T]; any
    may be missing) against the reference on its replicates' flows Q [n_reps, T]: bit for bit (NaN where NaN)."""
    ref = quantiles(Q, windows, levels, lo, hi)
    if "q" in got:
        g = np.asarray(got["q"])
        assert g.shape == ref["q"].shape, (where, g.shape, ref["q"].shape)
        same = (g == ref["q"]) | (np.isnan(g) & np.isnan(ref["q"]))
        assert same.all(), (where, "q", np.argwhere(~same)[:5], g[~same][:5], ref["q"][~same][:5])
    if "nonfinite" in got:
        assert np.array_equal(np.asarray(got["nonfinite"]), ref["nonfinite"]), (where, "nonfinite")
    return ref
