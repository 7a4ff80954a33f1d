"""The EM kernels' and the single-step kernels' SOURCE run on the CPU by a coroutine-per-thread emulator
(tests/host_simt/): checks, without a GPU and without compute-sanitizer (closed on the GPU pool), that
  * the kernels' control flow, shared-memory carve-up and cross-warp exchanges reproduce the oracle,
  * results are BIT-IDENTICAL under different orders of resuming the CTA's threads between
    synchronisation points -- a shared-memory race (two accesses to one word that no barrier orders)
    shows up as a difference (the racecheck stand-in),
  * no thread reads shared memory that was never written (it starts as NaN) or past its end (traps).
The arithmetic differs from the GPU build only in the reciprocal seed (lds_math.cuh, fast_rcp)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import oracle as O
from tests import data

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_simt")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SO = os.path.join(HERE, "libldsr_hostsim.so")
_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int)


def _lib():
    srcs = [os.path.join(HERE, f) for f in ("sim_em.cpp", "host_simt.h")]
    csrc = os.path.join(ROOT, "ldsr_b200", "csrc")
    srcs += [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith(".cuh")]
    if not os.path.exists(SO) or any(os.path.getmtime(s) > os.path.getmtime(SO) for s in srcs):
        wide = ["-DLDSR_HAVE_WIDE"] if os.path.exists(os.path.join(csrc, "em_wide_kernel.cuh")) else []
        wide += ["-DLDSR_HAVE_SCAN"] if os.path.exists(os.path.join(csrc, "em_scan_kernel.cuh")) else []
        subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-DLDSR_HOST_SIM", "-Wno-unknown-pragmas", "-mfma",
                        "-ffp-contract=off", "-shared", "-fPIC"] + wide +
                       [os.path.join(HERE, "sim_em.cpp"), "-o", SO], check=True)
    return C.CDLL(SO)


def sim_em(kind, y, u, v, held, fit_group, theta0, niter, tol=1e-5, chunk=100, order=0, grid_cap=0):
    L = _lib()
    y = np.ascontiguousarray(y, dtype=np.float64)
    T = y.size
    uf = None if u is None else np.ascontiguousarray(np.asarray(u, dtype=np.float64).T)
    vf = None if v is None else np.ascontiguousarray(np.asarray(v, dtype=np.float64).T)
    p = 1 if uf is None else uf.shape[1]
    q = 1 if vf is None else vf.shape[1]
    hp = np.zeros(len(held) + 1, dtype=np.int32)
    hp[1:] = np.cumsum([len(h) for h in held])
    hi = np.ascontiguousarray(np.concatenate([np.asarray(h, dtype=np.int32) for h in held] + [np.zeros(1, np.int32)]))
    fg = np.ascontiguousarray(fit_group, dtype=np.int32)
    th0 = np.ascontiguousarray(theta0, dtype=np.float64)
    nf = fg.size
    th = np.full_like(th0, np.nan)
    lik = np.empty(nf)
    it = np.empty(nf, dtype=np.int32)
    d = lambda a: None if a is None else a.ctypes.data_as(_dp)
    i = lambda a: a.ctypes.data_as(_ip)
    rc = L.hostsim_em(kind, T, p, q, d(y), d(uf), d(vf), len(held), i(hp), i(hi), nf, i(fg), d(th0), niter,
                      C.c_double(tol), chunk, order, grid_cap, d(th), d(lik), i(it))
    assert rc == 0, rc
    return dict(theta=th, lik=lik, iters=it)


def sim_em_traj(y, u, v, held, fit_group, theta0, niter, tol=1e-5, chunk=100, order=0, grid_cap=0):
    """The scan kernel's EM, then its trajectory mode on every fit's final theta (last fit: 'no winner')."""
    L = _lib()
    y = np.ascontiguousarray(y, dtype=np.float64)
    T = y.size
    uf = np.ascontiguousarray(np.asarray(u, dtype=np.float64).T)
    vf = np.ascontiguousarray(np.asarray(v, dtype=np.float64).T)
    hp = np.zeros(len(held) + 1, dtype=np.int32)
    hp[1:] = np.cumsum([len(h) for h in held])
    hi = np.ascontiguousarray(np.concatenate([np.asarray(h, dtype=np.int32) for h in held] + [np.zeros(1, np.int32)]))
    fg = np.ascontiguousarray(fit_group, dtype=np.int32)
    th0 = np.ascontiguousarray(theta0, dtype=np.float64)
    nf = fg.size
    th, lik, it = np.full_like(th0, np.nan), np.empty(nf), np.empty(nf, dtype=np.int32)
    traj = np.full((4, nf, T), 12345.0)
    d = lambda a: a.ctypes.data_as(_dp)
    i = lambda a: a.ctypes.data_as(_ip)
    rc = L.hostsim_em_traj(T, uf.shape[1], vf.shape[1], d(y), d(uf), d(vf), len(held), i(hp), i(hi), nf, i(fg), d(th0),
                           niter, C.c_double(tol), chunk, order, grid_cap, d(th), d(lik), i(it), d(traj))
    assert rc == 0, rc
    return dict(theta=th, lik=lik, iters=it, X=traj[0], Y=traj[1], V=traj[2], J=traj[3])


def rand_theta0(rng, p, q, n):
    return np.stack([np.concatenate([[rng.uniform()], rng.uniform(-1, 1, p), [rng.uniform()],
                                     rng.uniform(-1, 1, q), [1, 1, 0, 1]]) for _ in range(n)])


def _np_job(n_folds=3, n_rest=14, seed=5):
    y, u, mu, inst = data.np_case(601, 1800)  # T = 213
    rng = np.random.default_rng(seed)
    held = [np.sort(rng.choice(inst, 11, replace=False)) for _ in range(n_folds)]
    fg = np.repeat(np.arange(n_folds), n_rest)
    return y, u, held, fg, rand_theta0(rng, 3, 3, n_folds * n_rest)


def _check_vs_oracle(r, y, u, v, held, fg, th0, niter):
    o = O.em_batch([dict(y=y, u=u, v=v)], np.zeros(len(held), dtype=int), held, fg, th0, niter, 1e-5)
    assert np.array_equal(r["iters"], o["iters"])
    assert np.allclose(r["lik"], o["lik"], rtol=1e-9, atol=0)
    assert np.allclose(r["theta"], o["theta"], rtol=1e-6, atol=1e-12)


@pytest.mark.parametrize("kind", [3, 2])
def test_emulated_kernel_matches_oracle_and_is_schedule_independent(kind):
    y, u, held, fg, th0 = _np_job()
    niter = 7
    base = sim_em(kind, y, u, u, held, fg, th0, niter, chunk=4, order=0)
    _check_vs_oracle(base, y, u, u, held, fg, th0, niter)
    for order in (1, 2, 3):
        r = sim_em(kind, y, u, u, held, fg, th0, niter, chunk=4, order=order)
        for k in ("theta", "lik", "iters"):
            assert np.array_equal(base[k], r[k]), (order, k)


def test_emulated_task_loop_reuses_shared_memory_safely():
    # one CTA takes both tasks in turn (grid_cap = 1): the arena is re-used across tasks
    y, u, held, fg, th0 = _np_job(n_folds=3, n_rest=14)  # 42 fits = 2 tasks of the time-split kernel
    a = sim_em(3, y, u, u, held, fg, th0, 5, chunk=5, order=2, grid_cap=1)
    b = sim_em(3, y, u, u, held, fg, th0, 5, chunk=5, order=0, grid_cap=0)
    for k in ("theta", "lik", "iters"):
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("slots,chunk,n_rest", [(2, 5, 35), (2, 4, 35), (4, 5, 35), (3, 5, 70)])
def test_emulated_tasks_shared_by_iterations(slots, chunk, n_rest):
    """Iteration-level task sharing (SplitParams.flags): 3 tasks on 2 CTAs -- a task's first iterations at the
    start of one CTA's slot, the rest at the end of the previous one's --, on more CTAs than tasks, and 5 tasks
    on 3 CTAs (the middle CTA: end of one task, a whole task, start of another); results are bit-identical to
    one CTA per task, whatever the chunk length."""
    y, u, held, fg, th0 = _np_job(n_folds=2, n_rest=n_rest)  # 70 fits = 3 tasks, 140 = 5
    a = sim_em(3, y, u, u, held, fg, th0, 7, chunk=chunk, order=2, grid_cap=-slots)
    b = sim_em(3, y, u, u, held, fg, th0, 7, chunk=7, order=0, grid_cap=0)
    for k in ("theta", "lik", "iters"):
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("slots,order", [(4, 0), (6, 3), (2, 1)])
def test_emulated_ranked_assignment_and_extra_iterations(slots, order):
    """At most one task per CTA, two CTAs per (emulated) SM: tasks are dealt by progress and by where the CTAs
    landed, and a CTA keeps iterating past its chunk while others have not finished theirs (the emulator runs
    the CTAs one after the other, so the first ones run their fits to the end).  Results equal the plain run's."""
    y, u, held, fg, th0 = _np_job(n_folds=2, n_rest=35)  # 3 tasks; slots = 2: the first launch shares by iterations
    a = sim_em(3, y, u, u, held, fg, th0, 9, chunk=4, order=order, grid_cap=-slots)
    b = sim_em(3, y, u, u, held, fg, th0, 9, chunk=9, order=0, grid_cap=0)
    for k in ("theta", "lik", "iters"):
        assert np.array_equal(a[k], b[k]), k


def _wide_job(p=10, T=150, n_fits=40, seed=3, first_obs=60):
    rng = np.random.default_rng(seed)
    u = rng.standard_normal((p, T)) * np.sqrt(4.0 / np.arange(1, p + 1))[:, None]
    x = np.zeros(T)
    for t in range(1, T):
        x[t] = 0.6 * x[t - 1] + 0.1 * u[0, t - 1] + 0.5 * rng.standard_normal()
    y = 0.8 * x + 0.05 * u[0] + 0.3 * rng.standard_normal(T)
    y[:first_obs] = np.nan
    y[first_obs + 9] = np.nan  # a gap inside the instrumental period
    held = [np.array([first_obs + 3, first_obs + 4, T - 1]), np.array([], dtype=int), np.array([T - 2])]
    fg = np.sort(rng.integers(0, 3, n_fits))
    return y, u, held, fg, rand_theta0(rng, p, p, n_fits)


@pytest.mark.parametrize("p,T,first_obs", [(10, 150, 60), (10, 77, 5), (3, 213, None), (6, 130, 70)])
def test_emulated_wide_kernel(p, T, first_obs):
    """em_wide_kernel (phase A / scalar recursions / phase C): oracle parity and schedule independence,
    incl. a series observed almost everywhere (no unobserved word), a ragged tail and a narrow width."""
    if first_obs is None:
        y, u, held, fg, th0 = _np_job()
    else:
        y, u, held, fg, th0 = _wide_job(p, T, 40, seed=p * T, first_obs=first_obs)
    niter = 6
    base = sim_em(4, y, u, u, held, fg, th0, niter, chunk=4, order=0)
    _check_vs_oracle(base, y, u, u, held, fg, th0, niter)
    for order in (1, 5):
        r = sim_em(4, y, u, u, held, fg, th0, niter, chunk=4, order=order)
        for k in ("theta", "lik", "iters"):
            assert np.array_equal(base[k], r[k]), (order, k)


def test_emulated_wide_kernel_separate_v_and_task_loop():
    y, u, held, fg, th0 = _wide_job(10, 120, 70, seed=9, first_obs=40)
    rng = np.random.default_rng(1)
    v = rng.standard_normal((7, 120))
    th0 = rand_theta0(rng, 10, 7, 70)
    a = sim_em(4, y, u, v, held, fg, th0, 5, chunk=5, order=0)
    _check_vs_oracle(a, y, u, v, held, fg, th0, 5)
    b = sim_em(4, y, u, v, held, fg, th0, 5, chunk=2, order=3, grid_cap=1)  # 3 tasks on one CTA, 3 launches
    for k in ("theta", "lik", "iters"):
        assert np.array_equal(a[k], b[k]), k


@pytest.mark.parametrize("T", [213, 40, 129, 14])
def test_emulated_scan_kernel(T):
    """em_scan_kernel (one CTA per fit, one thread per 4 steps, the recursions as scans): oracle parity and
    schedule independence; lengths that leave the last warp ragged, fill one warp exactly or not at all."""
    y, u, held, fg, th0 = _np_job(n_folds=2, n_rest=3)
    if T != 213:
        y, u = y[213 - T:], u[:, 213 - T:]
        if T == 14:
            y = np.array([0.1, -0.2, np.nan, 0.3, 0.05, 0.2, -0.1, 0.15, np.nan, -0.3, 0.25, 0.1, -0.05, 0.12])
        held = [np.array([T - 1]), np.array([], dtype=int)]
    niter = 9
    base = sim_em(5, y, u, u, held, fg, th0, niter, chunk=4, order=0)
    _check_vs_oracle(base, y, u, u, held, fg, th0, niter)
    for order in (1, 4):
        r = sim_em(5, y, u, u, held, fg, th0, niter, chunk=4, order=order, grid_cap=2 if order == 4 else 0)
        for k in ("theta", "lik", "iters"):
            assert np.array_equal(base[k], r[k]), (order, k)
    # two steps per thread (the LDSR_SCAN_L=2 build): orders >= 8 select it in the harness
    r4 = sim_em(5, y, u, u, held, fg, th0, niter, chunk=4, order=8)
    _check_vs_oracle(r4, y, u, u, held, fg, th0, niter)
    r4b = sim_em(5, y, u, u, held, fg, th0, niter, chunk=4, order=9)
    for k in ("theta", "lik", "iters"):
        assert np.array_equal(r4[k], r4b[k]), k


@pytest.mark.parametrize("p,T", [(10, 150), (7, 85), (6, 40)])
def test_emulated_scan_kernel_wide_inputs(p, T):
    """The scan kernel with 5..10 inputs (v == u, two steps per thread, 32 + 16-value sum reduction, the M-step's
    matrix-vector rows spread over the lanes)."""
    y, u, held, fg, th0 = _wide_job(p, T, 9, seed=100 + p, first_obs=T // 3)
    th0[:, 1:1 + p] *= 0.2
    th0[:, 2 + p:2 + 2 * p] *= 0.2
    niter = 8
    base = sim_em(5, y, u, u, held, fg, th0, niter, chunk=5, order=0)
    _check_vs_oracle(base, y, u, u, held, fg, th0, niter)
    r = sim_em(5, y, u, u, held, fg, th0, niter, chunk=5, order=3)
    for k in ("theta", "lik", "iters"):
        assert np.array_equal(base[k], r[k]), k


@pytest.mark.parametrize("case", ["np213", "np40_separate_v", "wide10", "wide7_ragged"])
def test_emulated_scan_kernel_trajectory_mode(case):
    """em_scan_kernel<.., EMIT>: the smoothed X, Y, V, J of a (group, theta) pair against the oracle's E-step with the
    same theta on the group's y (held-out steps missing); a job without a winner gives NaN rows; schedule
    independence; CTAs that take several jobs."""
    rng = np.random.default_rng(3)
    if case.startswith("np"):
        y, u, held, fg, th0 = _np_job(n_folds=2, n_rest=3)
        v = u
        if case == "np40_separate_v":
            y, u = y[213 - 40:], u[:, 213 - 40:]
            v = rng.standard_normal((2, 40))
            held = [np.array([39]), np.array([], dtype=int)]
            th0 = rand_theta0(rng, 3, 2, 6)
    else:
        p, T = (10, 150) if case == "wide10" else (7, 85)
        y, u, held, fg, th0 = _wide_job(p, T, 7, seed=50 + p, first_obs=T // 3)
        th0[:, 1:1 + p] *= 0.2
        th0[:, 2 + p:2 + 2 * p] *= 0.2
        v = u
    a = sim_em_traj(y, u, v, held, fg, th0, 6, chunk=6, order=0)
    nf = fg.size
    for f in range(nf - 1):
        yy = np.array(y, dtype=float)
        yy[held[fg[f]]] = np.nan
        s = O.kalman_smoother(yy, u, v, a["theta"][f])
        for k in ("X", "Y", "V", "J"):
            assert np.allclose(a[k][f], s[k], rtol=1e-10, atol=1e-13), (f, k, np.max(np.abs(a[k][f] - s[k])))
    for k in ("X", "Y", "V", "J"):
        assert np.isnan(a[k][nf - 1]).all()
    b = sim_em_traj(y, u, v, held, fg, th0, 6, chunk=6, order=3, grid_cap=2)
    for k in ("X", "Y", "V", "J"):
        assert np.array_equal(a[k], b[k], equal_nan=True), k


# ---- the single-step kernels (aux_kernels.cuh) -------------------------------------------------------------------
# Case generators of tests/test_gpu_step_kernels.py; here one series per case, padded to width 3, 5 or 16 (steps per
# smoother block 8, 4 and 1), with one group per hold-out kind and two theta per group.
from tests import test_gpu_step_kernels as SK  # noqa: E402

STEP_WIDTHS = [(3, 3, "vu"), (3, 2, "sep"), (1, 3, "unone"), (5, 5, "vu"), (4, 2, "sep"), (13, 13, "vu"),
               (16, 9, "sep")]


def _held_arrays(held):
    hp = np.zeros(len(held) + 1, dtype=np.int32)
    hp[1:] = np.cumsum([len(h) for h in held])
    hi = np.ascontiguousarray(np.concatenate([np.asarray(h, dtype=np.int32) for h in held] + [np.zeros(1, np.int32)]))
    return hp, hi


def sim_step(kind, s, held, job_group, theta=None, job_theta=None, stdlik=True, rows=None, order=0):
    """hostsim_step: kind 0 smoother, 1 propagate, 2 M-step (from rows X, V, J).  s: dict(y, u, v, p, q)."""
    L = _lib()
    y = np.ascontiguousarray(s["y"], dtype=np.float64)
    T, p, q = y.size, s["p"], s["q"]
    uf = None if s["u"] is None else np.ascontiguousarray(np.asarray(s["u"], dtype=np.float64).T)
    vf = None if s["v"] is None else np.ascontiguousarray(np.asarray(s["v"], dtype=np.float64).T)
    hp, hi = _held_arrays(held)
    jg = np.ascontiguousarray(job_group, dtype=np.int32)
    nj = jg.size
    jt = np.ascontiguousarray(np.arange(nj) if job_theta is None else job_theta, dtype=np.int32)
    th = None if theta is None else np.ascontiguousarray(theta, dtype=np.float64)
    # one guard row past the last job's: a write beyond a job's T steps lands there (or in the next job's row)
    X, Y, V, J = (np.full((nj + 1, T), 12345.0) for _ in range(4))
    if rows is not None:
        for k, a in (("X", X), ("V", V), ("J", J)):
            a[:nj] = [r[k] for r in rows]
    lik, aux = np.full(nj, 12345.0), np.full(nj, 12345.0)
    th_out, st = np.full((nj, p + q + 6), np.nan), np.full(nj, -1, dtype=np.int32)
    d = lambda a: None if a is None else a.ctypes.data_as(_dp)
    i = lambda a: a.ctypes.data_as(_ip)
    rc = L.hostsim_step(kind, T, p, q, d(y), d(uf), d(vf), len(held), i(hp), i(hi), nj, i(jg), i(jt), d(th),
                        int(stdlik), order, d(X), d(Y), d(V), d(J), d(lik), d(aux), d(th_out), i(st))
    assert rc == 0, rc
    for k, a in (("X", X), ("Y", Y), ("V", V), ("J", J)):
        assert np.all(a[nj] == 12345.0), "%s written past the last job's row" % k
    return dict(X=X[:nj], Y=Y[:nj], V=V[:nj], J=J[:nj], lik=lik, aux=aux, theta=th_out, status=st)


def _step_case(p, q, form, seed, T=150):
    rng = np.random.default_rng(seed)
    s = SK.make_series(rng, p, q, form, T)
    held = [SK.holdout(rng, s["y"], k) for k in SK.HOLD_KINDS]
    job_group = np.repeat(np.arange(len(held)), 2)
    return s, held, job_group, np.stack([SK.rand_theta(rng, p, q) for _ in job_group])


def _y_of(s, held, g):
    y = np.array(s["y"], dtype=float)
    y[held[g]] = np.nan
    return y


@pytest.mark.parametrize("width", STEP_WIDTHS, ids=SK.case_id)
def test_emulated_smoother_and_propagate_match_the_oracle(width):
    """smoother_kernel (incl. a job without theta: NaN rows) and propagate_kernel from their source, against the
    oracle: rows, lik, and the per-job sums of the experimental learners' objectives."""
    p, q, _ = width
    s, held, jg, th = _step_case(*width, seed=100 * p + q)
    jt = np.arange(jg.size)
    jt[3] = -1
    sm = sim_step(0, s, held, jg, th, job_theta=jt, stdlik=True)
    pr = sim_step(1, s, held, jg, th, stdlik=False)
    for j in range(jg.size):
        y = _y_of(s, held, jg[j])
        if jt[j] < 0:
            assert all(np.isnan(sm[k][j]).all() for k in "XYVJ") and np.isnan(sm["lik"][j])
            continue
        o = O.kalman_smoother(y, s["u"], s["v"], th[j], p=p, q=q, stdlik=True)
        for k in "XYVJ":
            assert SK.row_dev(sm[k][j], o[k]) < SK.ROW_RTOL, (j, k, SK.row_dev(sm[k][j], o[k]))
        assert SK.rel_dev(sm["lik"][j], o["lik"]) < SK.LIK_RTOL, j
        Bu = th[j][1:1 + p] @ s["u"][:, :-1] if s["u"] is not None else 0.0
        ssq = np.sum((o["X"][1:] - th[j][0] * o["X"][:-1] - Bu) ** 2)
        assert SK.rel_dev(sm["aux"][j], ssq) < SK.LIK_RTOL, j
        o = O.propagate(th[j], s["u"], s["v"], y, p=p, q=q, stdlik=False)
        for k in "XYV":
            assert SK.row_dev(pr[k][j], o[k]) < SK.ROW_RTOL, (j, k)
        assert SK.rel_dev(pr["lik"][j], o["lik"]) < SK.LIK_RTOL, j
        assert SK.rel_dev(pr["aux"][j], np.nansum((y - o["Y"]) ** 2)) < SK.LIK_RTOL, j


@pytest.mark.parametrize("width", STEP_WIDTHS, ids=SK.case_id)
def test_emulated_mstep_matches_the_oracle(width):
    """mstep_kernel from its source on the oracle smoother's rows, for the groups with at least 3 max(p, q) observed
    steps (well-conditioned Gram blocks)."""
    p, q, _ = width
    s, held, jg, th = _step_case(*width, seed=100 * p + q)
    rows = [O.kalman_smoother(_y_of(s, held, jg[j]), s["u"], s["v"], th[j], p=p, q=q) for j in range(jg.size)]
    r = sim_step(2, s, held, jg, rows=rows)
    checked = 0
    for j in range(jg.size):
        y = _y_of(s, held, jg[j])
        if np.isfinite(y).sum() < 3 * max(p, q):
            continue
        assert r["status"][j] == 0, j
        o = O.mstep(y, s["u"], s["v"], rows[j], p=p, q=q)
        d = np.max(np.abs(r["theta"][j] - o) / np.maximum(np.abs(o), SK.THETA_FLOOR))
        assert d < SK.THETA_RTOL, (j, d)
        checked += 1
    assert checked >= 6


REP_HOST_WIDTHS = [(3, 3, "vu"), (1, 3, "unone"), (3, 2, "vnone"), (5, 5, "vu"), (4, 2, "sep"), (16, 16, "vu"),
                   (13, 9, "sep")]


def sim_rep(p, q, u, v, n, z, theta, mu, exp_trans, want, order=0):
    L = _lib()
    n_reps = z.shape[0]
    uf = None if u is None else np.ascontiguousarray(np.asarray(u, dtype=np.float64).T)
    vf = None if v is None else np.ascontiguousarray(np.asarray(v, dtype=np.float64).T)
    outs = {k: np.full((n_reps, n), 12345.0) for k in want}
    d = lambda a: None if a is None else a.ctypes.data_as(_dp)
    rc = L.hostsim_rep(p, q, d(uf), d(vf), n, n_reps, d(np.ascontiguousarray(z)), d(np.ascontiguousarray(theta)),
                       C.c_double(mu), int(exp_trans), order, *(d(outs.get(k)) for k in ("simX", "simY", "simQ")))
    assert rc == 0, rc
    return outs


@pytest.mark.parametrize("width", REP_HOST_WIDTHS, ids=SK.case_id)
def test_emulated_rep_kernel_matches_the_oracle_and_is_schedule_independent(width):
    """rep_kernel with caller noise from its source: oracle parity replicate by replicate, and bit-identical outputs
    under several thread schedules -- its tile transposes are the one cross-lane shared-memory exchange among the
    single-step kernels, ordered by __syncwarp.  n is not a multiple of the 16-step tile, n_reps not one of 32."""
    p, q, form = width
    rng = np.random.default_rng(p * 100 + q)
    for n, n_reps, exp_trans, want in ((17, 33, True, ("simX", "simY", "simQ")), (40, 70, False, ("simQ",)),
                                       (1, 5, True, ("simX", "simQ"))):
        u = None if form == "unone" else rng.standard_normal((p, n))
        v = None if form == "vnone" else (u if form == "vu" else rng.standard_normal((q, n)))
        th = SK.rand_theta(rng, p, q)
        mu = 0.37 if exp_trans else -1.3
        z = rng.standard_normal((n_reps, 1 + 2 * n))
        base = sim_rep(p, q, u, v, n, z, th, mu, exp_trans, want)
        for i in range(n_reps):
            o = O.rep(th, u, v, n, z[i], mu=mu, exp_trans=exp_trans, p=p, q=q)
            for k in want:
                assert SK.row_dev(base[k][i], o[k]) < SK.ROW_RTOL, (n, i, k)
        for order in (1, 2, 3):
            r = sim_rep(p, q, u, v, n, z, th, mu, exp_trans, want, order=order)
            for k in want:
                assert np.array_equal(r[k], base[k]), (n, order, k)
