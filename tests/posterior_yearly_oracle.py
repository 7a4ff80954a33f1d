"""CPU reference for the year-by-year drought counts of conditioned replicates (ldsr_posterior_yearly_batch), used by
tests/test_posterior_yearly_host.py and tests/test_gpu_posterior_yearly.py.  Never imported by the product.

From a [n_reps, T] array of back-transformed flows Q, a threshold thr and a step range [lo, hi), per step t of the
range, the number of replicates with:
  * below:      Q_t < thr (a non-finite Q_t is not below);
  * in_run[k]:  t inside a run of length >= lengths[k], a run being a maximal stretch of below steps of the range;
  * wbelow[k]:  Q_t .. Q_{t+w-1} all finite and summing to less than w thr (w = windows[k]), for lo <= t <= hi - w;
  * nonfinite:  Q_t not finite.
Steps outside the range, and window starts past hi - w, are -1.  Runs are found by an explicit scan, upwards and
downwards (the kernel decides each step with a delay in its downward walk); window sums are exact (math.fsum)
wherever a rounded sum lies near w thr."""
import math

import numpy as np

NEAR = 1e-9  # a window whose exact sum is this close to w thr (relative) may be counted either way


def run_lengths(below):
    """below [n, m] bool -> [n, m] int: the length of the run each below step lies in (0 where not below)."""
    n, m = below.shape
    up, down = np.zeros((n, m), np.int64), np.zeros((n, m), np.int64)
    cur = np.zeros(n, np.int64)
    for t in range(m):  # below steps ending at t
        cur = np.where(below[:, t], cur + 1, 0)
        down[:, t] = cur
    cur[:] = 0
    for t in range(m - 1, -1, -1):  # below steps starting at t
        cur = np.where(below[:, t], cur + 1, 0)
        up[:, t] = cur
    return np.where(below, up + down - 1, 0)


def window_sums(Q, w, thr):
    """Q [n, m] (finite values, zeros in place of non-finite ones) -> sums [n, m - w + 1] of every w consecutive
    values, exact (math.fsum) wherever the rounded sum lies within 1e-6 of w thr, and their scale sum |Q|."""
    v = np.lib.stride_tricks.sliding_window_view(Q, w, axis=1)
    sums, scale = v.sum(axis=2), np.abs(v).sum(axis=2)
    for i, j in zip(*np.nonzero(np.abs(sums - w * thr) <= 1e-6 * np.maximum(abs(w * thr), scale))):
        sums[i, j] = math.fsum(v[i, j])
    return sums, scale


def counts(Q, thr, windows, lengths, lo, hi):
    """Q [n_reps, T] -> dict of int64 rows: below [T], in_run [n_lengths, T], wbelow [n_windows, T], nonfinite [T],
    and wbelow_lo / wbelow_hi [n_windows, T]: the window counts with every window near w thr (NEAR) left out / put
    in (equal to wbelow where there is none)."""
    Q = np.atleast_2d(np.asarray(Q, dtype=float))
    n, T = Q.shape
    Qr = Q[:, lo:hi]
    fin = np.isfinite(Qr)
    with np.errstate(invalid="ignore"):
        bel = Qr < thr
    out = {k: np.full(T, -1, np.int64) for k in ("below", "nonfinite")}
    out["below"][lo:hi] = bel.sum(axis=0)
    out["nonfinite"][lo:hi] = (~fin).sum(axis=0)
    rl = run_lengths(bel)
    out["in_run"] = np.full((len(lengths), T), -1, np.int64)
    for k, L in enumerate(lengths):
        out["in_run"][k, lo:hi] = (rl >= L).sum(axis=0)
    for key in ("wbelow", "wbelow_lo", "wbelow_hi"):
        out[key] = np.full((len(windows), T), -1, np.int64)
    for k, w in enumerate(windows):
        if w > hi - lo:
            continue
        sums, scale = window_sums(np.where(fin, Qr, 0.0), w, thr)
        ok = np.lib.stride_tricks.sliding_window_view(fin, w, axis=1).all(axis=2)
        tol = NEAR * np.maximum(abs(w * thr), scale)
        s = slice(lo, hi - w + 1)
        out["wbelow"][k, s] = (ok & (sums < w * thr)).sum(axis=0)
        out["wbelow_lo"][k, s] = (ok & (sums < w * thr - tol)).sum(axis=0)
        out["wbelow_hi"][k, s] = (ok & (sums < w * thr + tol)).sum(axis=0)
    return out


def assert_match(got, Q, thr, windows, lengths, lo, hi, where=""):
    """Counts of one fit from the library or the emulator (below / nonfinite [T], in_run [n_lengths, T], wbelow
    [n_windows, T]; any may be missing) against the reference on its replicates' flows Q [n_reps, T]: below, in_run
    and nonfinite exactly, wbelow exactly except where windows lie near w thr, where it must lie between the counts
    with those windows left out and put in.  Returns the number of steps where the window bounds differ."""
    ref = counts(Q, thr, windows, lengths, lo, hi)
    for k in ("below", "in_run", "nonfinite"):
        if k in got:
            assert np.array_equal(np.asarray(got[k]), ref[k]), (where, k)
    if "wbelow" not in got:
        return 0
    g = np.asarray(got["wbelow"])
    assert ((ref["wbelow_lo"] <= g) & (g <= ref["wbelow_hi"])).all(), (where, "wbelow")
    assert np.array_equal(g < 0, ref["wbelow"] < 0), (where, "wbelow")
    return int((ref["wbelow_lo"] != ref["wbelow_hi"]).sum())
