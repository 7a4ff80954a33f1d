"""Replicates conditioned on the observed record (forward filtering, backward sampling), without a GPU:
  * the reference (tests/posterior_oracle.py) with zero noise is the oracle's smoother (X everywhere, Y at unobserved steps) and copies y at observed
    steps, and on the NPlds fixture its back-transformed flows are the stored reconstruction's Q;
  * smoother_kernel's coefficient mode and posterior_rep_kernel, run from source by the CPU emulator at widths
    3, 5 and 16 with caller noise, match the oracle replicate by replicate and are bit-identical under four
    thread schedules and when cut into several launches;
  * ldsr_posterior_rep_batch checks its arguments before it looks for a device."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np
import pytest

from ldsr_b200 import _lib
from oracle import oracle as O
from tests import data
from tests import posterior_oracle as PO
from tests import test_gpu_step_kernels as SK

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "host_simt")
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ldsr_b200", "csrc")
_hostsim = None


def hostsim_lib():
    """tests/host_simt/sim_posterior.cpp built for the CPU (as test_host_simt.py builds sim_em.cpp), into the
    temporary directory under a name keyed by its sources."""
    global _hostsim
    if _hostsim is None:
        srcs = [os.path.join(HERE, f) for f in ("sim_posterior.cpp", "sim_em.cpp", "host_simt.h")]
        srcs += sorted(os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith(".cuh"))
        key = hashlib.sha256(b"".join(open(f, "rb").read() for f in srcs)).hexdigest()[:16]
        so = os.path.join(tempfile.gettempdir(), "ldsr_hostsim_post_%s_%d.so" % (key, os.getuid()))
        if not os.path.exists(so):
            tmp = so + ".%d.tmp" % os.getpid()
            subprocess.run(["g++", "-O1", "-g", "-std=c++17", "-DLDSR_HOST_SIM", "-Wno-unknown-pragmas", "-mfma",
                            "-ffp-contract=off", "-shared", "-fPIC", "-DLDSR_HAVE_WIDE", "-DLDSR_HAVE_SCAN",
                            srcs[0], "-o", tmp], check=True)
            os.replace(tmp, so)
        _hostsim = C.CDLL(so)
    return _hostsim

_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int)
TRANSFORMS = (("log", 0.0), ("none", 0.0), ("boxcox", 0.35), ("boxcox", 0.0))


def _zero_noise_cases():
    rng = np.random.default_rng(11)
    out = []
    for p, q, form in ((3, 3, "vu"), (4, 2, "sep"), (1, 3, "unone"), (3, 2, "vnone")):
        for T in (2, 17, 65, 213):
            s = SK.make_series(rng, p, q, form, T)
            for kind in ("none", "first", "last", "scattered"):
                out.append((s, SK.holdout(rng, s["y"], kind), SK.rand_theta(rng, p, q)))
    return out


def test_oracle_with_zero_noise_is_the_smoother():
    for s, held, th in _zero_noise_cases():
        y = np.array(s["y"], dtype=float)
        y[held] = np.nan
        T = y.size
        r = PO.posterior_rep(th, s["y"], s["u"], s["v"], np.zeros(2 * T), mu=0.0, transform="none", held=held,
                             p=s["p"], q=s["q"])
        sm = O.kalman_smoother(y, s["u"], s["v"], th, p=s["p"], q=s["q"])
        un = np.isnan(y)
        assert SK.row_dev(r["simX"], sm["X"]) < SK.ROW_RTOL
        if un.any():
            assert SK.row_dev(r["simY"][un], sm["Y"][un]) < SK.ROW_RTOL
        assert np.array_equal(r["simY"][~un], y[~un])  # bit for bit
        assert np.array_equal(r["simQ"], r["simY"])    # transform none, mu = 0


def test_oracle_with_zero_noise_reproduces_the_stored_reconstruction():
    # R/sysdata.rda::NPlds: stored theta, T = 813, 46 observed years; rec$Q = exp(Y + mu) at the 767 others
    g = data.load("nplds.json")
    y, u, mu, inst = data.np_case(1, 1200)
    th = data.theta_of(g["theta"])
    r = PO.posterior_rep(th, y, u, u, np.zeros(2 * y.size), mu=mu, transform="log")
    un = np.isnan(y)
    assert un.sum() == 767
    Q = np.array(g["rec"]["Q"])
    assert np.max(np.abs(r["simQ"][un] - Q[un]) / Q[un]) < 1e-10
    assert np.array_equal(r["simY"][~un], y[~un])


def sim_posterior(s, held, fit_group, theta, n_reps, z, mu, transform, lam, order=0, chunk_blk=0,
                  want=("simX", "simY", "simQ")):
    L = hostsim_lib()
    y = np.ascontiguousarray(s["y"], dtype=np.float64)
    T = y.size
    uf = None if s["u"] is None else np.ascontiguousarray(np.asarray(s["u"], dtype=np.float64).T)
    vf = None if s["v"] is None else np.ascontiguousarray(np.asarray(s["v"], dtype=np.float64).T)
    hp = np.zeros(len(held) + 1, dtype=np.int32)
    hp[1:] = np.cumsum([len(h) for h in held])
    hi = np.ascontiguousarray(np.concatenate([np.asarray(h, dtype=np.int32) for h in held] + [np.zeros(1, np.int32)]))
    fg = np.ascontiguousarray(fit_group, dtype=np.int32)
    nf = fg.size
    th = np.ascontiguousarray(theta, dtype=np.float64)
    mu = np.ascontiguousarray(mu, dtype=np.float64)
    lam = np.ascontiguousarray(lam, dtype=np.float64)
    outs = {k: np.full((nf, n_reps, T), 12345.0) for k in want}
    d = lambda a: None if a is None else a.ctypes.data_as(_dp)
    i = lambda a: a.ctypes.data_as(_ip)
    rc = L.hostsim_posterior_rep(T, s["p"], s["q"], d(y), d(uf), d(vf), len(held), i(hp), i(hi), nf, i(fg), d(th),
                                 n_reps, d(np.ascontiguousarray(z)), d(mu), _lib.TRANSFORMS[transform], d(lam), order,
                                 chunk_blk, *(d(outs.get(k)) for k in ("simX", "simY", "simQ")))
    assert rc == 0, rc
    return outs


# widths 3 (8 smoother steps per block), 5 (4) and 16 (1); v == u, v != u, u = None, v = None
HOST_WIDTHS = [(3, 3, "vu"), (2, 3, "unone"), (5, 4, "sep"), (4, 3, "vnone"), (16, 16, "vu"), (9, 13, "sep")]


@pytest.mark.parametrize("width", HOST_WIDTHS, ids=SK.case_id)
def test_emulated_posterior_kernels_match_the_oracle_and_are_schedule_independent(width):
    """T not a multiple of the 16-step tile, replicate counts not a multiple of 32, hold-outs (one group each),
    several fits per group, per-fit mu, all three transforms and output subsets."""
    p, q, form = width
    rng = np.random.default_rng(p * 100 + q)
    for T, n_reps, (tr, lam), want in ((17, 33, TRANSFORMS[0], ("simX", "simY", "simQ")),
                                       (40, 70, TRANSFORMS[2], ("simQ",)),
                                       (2, 5, TRANSFORMS[1], ("simX", "simY")),
                                       (65, 3, TRANSFORMS[3], ("simY", "simQ"))):
        s = SK.make_series(rng, p, q, form, T)
        held = [SK.holdout(rng, s["y"], k) for k in ("none", "scattered", "last")]
        fit_group = np.array([0, 1, 1, 2, 2, 2])[:2 + T % 4]
        nf = fit_group.size
        theta = np.stack([SK.rand_theta(rng, p, q) for _ in range(nf)])
        mu = rng.uniform(0.5, 1.5, nf) + (3.0 if tr == "boxcox" else 0.0)  # Box-Cox: (y + mu) lam + 1 > 0
        lams = np.full(nf, lam)
        z = rng.standard_normal((nf, n_reps, 2 * T))
        base = sim_posterior(s, held, fit_group, theta, n_reps, z, mu, tr, lams, want=want)
        for f in range(nf):
            hy = held[fit_group[f]]
            obs = np.isfinite(s["y"]) & ~np.isin(np.arange(T), hy)
            o = PO.posterior_rep(theta[f], s["y"], s["u"], s["v"], z[f], mu=mu[f], transform=tr, lam=lam, held=hy,
                                 p=p, q=q)
            for r in range(n_reps):
                for k in want:
                    assert SK.row_dev(base[k][f, r], o[k][r]) < SK.ROW_RTOL, (T, f, r, k)
                if "simY" in want:
                    assert np.array_equal(base["simY"][f, r][obs], s["y"][obs]), (T, f, r)
        for order in (1, 2, 3):
            out = sim_posterior(s, held, fit_group, theta, n_reps, z, mu, tr, lams, order=order, want=want)
            for k in want:
                assert np.array_equal(out[k], base[k]), (T, order, k)
        # launches of a few (fit, 32 replicates) blocks each, every one writing from its own output offset
        out = sim_posterior(s, held, fit_group, theta, n_reps, z, mu, tr, lams, chunk_blk=1 + T % 3, want=want)
        for k in want:
            assert np.array_equal(out[k], base[k]), (T, "chunked", k)


def _small_batch():
    y = np.array([0.1, np.nan, -0.2, 0.3])
    return _lib.PackedBatch([dict(y=y, u=np.ones((1, 4)), v=None, p=1, q=1)], [0], None, [0],
                            np.array([[0.5, 0.1, 0.8, 0.0, 1.0, 0.5, 0.0, 1.0]]))


def _call(pb, n_reps=4, transform=1, lam=None, out=None):
    err = C.create_string_buffer(256)
    lam_a = None if lam is None else np.ascontiguousarray(lam, dtype=np.float64)
    o = np.empty(max(n_reps, 1) * 4) if out is None else out
    rc = _lib.lib().ldsr_posterior_rep_batch(None, C.byref(pb.c), int(n_reps), None, C.c_ulonglong(0), None,
                                             int(transform), _lib._d(lam_a), _lib._d(o), None, None, err, 256)
    return rc, err.value.decode()


def test_argument_errors_come_before_the_device():
    pb = _small_batch()
    for kw in (dict(n_reps=0), dict(n_reps=-3), dict(transform=3), dict(transform=-1), dict(transform=2)):
        rc, msg = _call(pb, **kw)
        assert rc == _lib.ERR_ARG, (kw, rc, msg)
    bad = _lib.PackedBatch([dict(y=np.array([0.1, 0.2]), u=None, v=None, p=1, q=1)], [0], None, [0],
                           np.array([[0.5, 0.0, 0.8, 0.0, 1.0, -0.5, 0.0, 1.0]]))  # R < 0
    assert _call(bad)[0] == _lib.ERR_ARG
    if _lib.device_count() == 0:  # a valid call finds no device
        rc, msg = _call(pb, transform=2, lam=[0.3])
        assert rc == _lib.ERR_CUDA, msg
