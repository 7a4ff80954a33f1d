"""CPU reference for the drought statistics of conditioned replicates (ldsr_posterior_stats_batch), used by
tests/test_posterior_stats_host.py and tests/test_gpu_posterior_stats.py.  Never imported by the product.

From a [n_reps, T] array of back-transformed flows Q and a step range [lo, hi), per replicate:
  * per window w, the minimum and maximum over starts lo <= t <= hi - w of the mean of Q_t .. Q_{t+w-1} and their
    starts (the smallest on a tie); w > hi - lo: NaN and -1;
  * the runs of Q_t < thr inside the range: the longest run's length and first step, the largest deficit
    sum(thr - Q_t) and its run's first step, the number of runs (the earliest run on a tie; none: 0, 0, -1, -1, 0);
  * a replicate with a non-finite Q in the range: NaN for every double output, -1 for every int output.
Window sums come from cumulative sums; runs are scanned step by step, upwards (the kernel walks downwards)."""
import numpy as np


def window_stats(Q, w, lo, hi):
    """Q [n_reps, T] -> (wmin, wmin_at, wmax, wmax_at, sums): means, first arg-extremes and the window sums
    [n_reps, hi - lo - w + 1] (for tie analysis)."""
    Q = np.atleast_2d(np.asarray(Q, dtype=float))
    n = Q.shape[0]
    nan, neg = np.full(n, np.nan), np.full(n, -1, dtype=np.int32)
    bad = ~np.isfinite(Q[:, lo:hi]).all(axis=1)
    if w > hi - lo:
        return nan, neg, nan.copy(), neg.copy(), np.zeros((n, 0))
    c = np.concatenate([np.zeros((n, 1)), np.cumsum(np.where(np.isfinite(Q[:, lo:hi]), Q[:, lo:hi], 0.0), axis=1)],
                       axis=1)
    sums = c[:, w:] - c[:, :-w]
    means = sums / w
    imin, imax = np.argmin(means, axis=1), np.argmax(means, axis=1)  # first occurrence: the smallest start
    r = np.arange(n)
    wmin, wmax = means[r, imin], means[r, imax]
    amin, amax = (lo + imin).astype(np.int32), (lo + imax).astype(np.int32)
    wmin[bad] = wmax[bad] = np.nan
    amin[bad] = amax[bad] = -1
    return wmin, amin, wmax, amax, sums


def run_stats(Q, thr, lo, hi):
    """Q [n_reps, T] -> dict(run_len, run_at, deficit, deficit_at, n_runs), one value per replicate.  The steps of
    the range are scanned in increasing order (vectorised over replicates); a run is closed at the first step not
    below thr, or at hi."""
    Q = np.atleast_2d(np.asarray(Q, dtype=float))
    n = Q.shape[0]
    run_len, run_at = np.zeros(n, np.int32), np.full(n, -1, np.int32)
    deficit, deficit_at, n_runs = np.zeros(n), np.full(n, -1, np.int32), np.zeros(n, np.int32)
    cur_len, cur_at, cur_def = np.zeros(n, np.int32), np.full(n, -1, np.int32), np.zeros(n)

    def close(m):
        n_runs[m] += 1
        longer = m & (cur_len > run_len)  # strictly: an earlier run keeps a tie
        run_len[longer], run_at[longer] = cur_len[longer], cur_at[longer]
        larger = m & (cur_def > deficit)
        deficit[larger], deficit_at[larger] = cur_def[larger], cur_at[larger]
        cur_len[m], cur_def[m] = 0, 0.0

    for t in range(lo, hi):
        below = Q[:, t] < thr
        start = below & (cur_len == 0)
        cur_at[start] = t
        cur_len[below] += 1
        cur_def[below] += thr - Q[below, t]
        close(~below & (cur_len > 0))
    close(cur_len > 0)
    bad = ~np.isfinite(Q[:, lo:hi]).all(axis=1)
    run_len[bad] = run_at[bad] = deficit_at[bad] = n_runs[bad] = -1
    deficit[bad] = np.nan
    return dict(run_len=run_len, run_at=run_at, deficit=deficit, deficit_at=deficit_at, n_runs=n_runs)


def stats(Q, windows, thr, lo, hi):
    """Every statistic of one fit: window outputs stacked [n_windows, n_reps], run outputs [n_reps] (thr None: no run
    outputs)."""
    ws = [window_stats(Q, w, lo, hi) for w in windows]
    out = {k: np.stack([x[j] for x in ws]) if ws else np.zeros((0, np.atleast_2d(Q).shape[0]))
           for j, k in enumerate(("wmin", "wmin_at", "wmax", "wmax_at"))}
    out["sums"] = [x[4] for x in ws]
    if thr is not None:
        out.update(run_stats(Q, thr, lo, hi))
    return out


RTOL = 1e-12


def assert_match(got, Q, windows, thr, lo, hi, where=""):
    """Statistics of one fit from the library or the emulator (window outputs [n_windows, n_reps], run outputs
    [n_reps]) against the reference on its replicates' flows Q [n_reps, T].  Counts, lengths and run steps exactly;
    means and deficits to RTOL relative to the larger of the value and the replicate's largest |Q| in the range (a
    running sum's rounding scales with the flows it has seen); a window's start may differ from the reference's only
    where the reference's means at the two starts are that close.  Returns the largest relative deviation."""
    ref = stats(Q, windows, thr, lo, hi)
    Qr = np.atleast_2d(Q)[:, lo:hi]
    with np.errstate(invalid="ignore"):
        scale = np.max(np.abs(np.where(np.isfinite(Qr), Qr, 0.0)), axis=1)
    dev = 0.0

    def close(a, b, k):
        nonlocal dev
        a, b = np.asarray(a), np.asarray(b)
        assert np.array_equal(np.isnan(a), np.isnan(b)), (where, k)
        ok = ~np.isnan(b)
        d = np.abs(a[ok] - b[ok]) / np.maximum(np.maximum(np.abs(b[ok]), scale[ok]), 1e-300)
        if d.size:
            dev = max(dev, float(d.max()))
            assert d.max() <= RTOL, (where, k, float(d.max()))

    for j, w in enumerate(windows):
        for v, a in (("wmin", "wmin_at"), ("wmax", "wmax_at")):
            close(got[v][j], ref[v][j], (v, w))
            ga, ra = np.asarray(got[a][j]), np.asarray(ref[a][j])
            diff = np.nonzero(ga != ra)[0]
            if diff.size:  # only a near tie of the reference's candidates may pick another start
                assert (ra[diff] >= 0).all() and (ga[diff] >= 0).all(), (where, a, w)
                means = ref["sums"][j] / w
                m_g, m_r = means[diff, ga[diff] - lo], means[diff, ra[diff] - lo]
                assert (np.abs(m_g - m_r) <= RTOL * np.maximum(np.abs(m_r), scale[diff])).all(), (where, a, w)
    if thr is not None:
        for k in ("run_len", "run_at", "deficit_at", "n_runs"):
            assert np.array_equal(got[k], ref[k]), (where, k)
        close(got["deficit"], ref["deficit"], "deficit")
    return dev
