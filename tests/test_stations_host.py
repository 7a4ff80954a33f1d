"""Host-side checks of the multi-station functions (no GPU needed): the ragged epilogues validate their
arguments before any device is touched, cvLDS_stations keeps the single-station argument errors, and a
stations call draws exactly what the single-station calls draw one after another on the same generator."""
import ctypes as C

import numpy as np
import pytest

import ldsr_b200 as L
from ldsr_b200 import _lib, api
from tests import data


def _stations():
    d = data.load("np.json")
    years, qa = np.array(d["NPannual"]["year"]), np.array(d["NPannual"]["Qa"])
    pc = np.array([d["NPpc"][k] for k in ("PC1", "PC9", "PC13")])
    return [dict(Qa=dict(year=years, Qa=qa), u=pc[:, 600:], v=pc[:, 600:], start_year=1800),
            dict(Qa=dict(year=years[10:], Qa=qa[10:]), u=None, v=pc[:2, 650:], start_year=1850),
            dict(Qa=dict(year=years[:-5], Qa=qa[:-5]), u=[pc[:, 500:], pc[:1, 500:]], v=[pc[:, 500:], None],
                 start_year=1700)]


def _rc(fn, *args):
    err = C.create_string_buffer(256)
    return fn(*args, err, 256), err.value.decode()


def _i(*v):
    return (C.c_int * len(v))(*v)


def _d(n):
    return (C.c_double * n)()


def test_ragged_epilogue_argument_errors_come_before_the_device():
    lib = _lib.lib()
    n, sim, out = _i(5, 4), _d(64), _d(64)
    z_ptr, z_idx = _i(0, 1, 2, 3), _i(1, 2, 3)
    cases = [
        (_i(0, 2, 1), z_ptr, z_idx, n),        # fold_ptr not monotone
        (_i(1, 2, 3), z_ptr, z_idx, n),        # fold_ptr[0] != 0
        (_i(0, 2, 3), _i(0, 2, 1, 3), z_idx, n),  # z_ptr not monotone
        (_i(0, 2, 3), z_ptr, _i(1, 2, 5), n),  # 5 is inside station 0's target (n = 5) but not station 1's (n = 4)
        (_i(0, 2, 3), z_ptr, _i(0, 2, 3), n),  # R indices are 1-based
        (_i(0, 2, 3), z_ptr, z_idx, _i(5, 1)),  # a target of length 1
        (_i(0, 0, 0), _i(0), z_idx, n),        # no fold at all
    ]
    for fold_ptr, zp, zi, nn in cases:
        rc, msg = _rc(lib.ldsr_cv_metrics_stations, 0, 2, nn, fold_ptr, sim, sim, zp, zi, 0, out)
        assert rc == _lib.ERR_ARG, msg
    T, m = _i(4, 3), _d(64)
    cases = [
        (T, _i(0, 2, 1), 0, m),   # member_ptr not increasing
        (T, _i(0, 2, 2), 0, m),   # a station without members
        (T, _i(1, 2, 3), 0, m),   # member_ptr[0] != 0
        (_i(4, 0), _i(0, 1, 2), 0, m),  # T < 1
        (T, _i(0, 1, 2), 3, m),   # unknown transform
        (T, _i(0, 1, 2), 2, None),  # boxcox without lambda
    ]
    for TT, mp, tr, lam in cases:
        rc, msg = _rc(lib.ldsr_construct_rec_stations, 0, 2, TT, mp, sim, sim, sim, sim, sim, sim, lam, tr, out, out)
        assert rc == _lib.ERR_ARG, msg
    with pytest.raises(_lib.LdsrError) as e:  # through the wrapper: index 6 is beyond the second station's target
        _lib.cv_metrics_stations([np.ones((1, 8)), np.ones((1, 5))], [np.ones(8), np.ones(5)],
                                 [[np.array([6])], [np.array([6])]])
    assert e.value.code == _lib.ERR_ARG
    if _lib.device_count() == 0:  # valid arguments and no device: no CPU fallback
        with pytest.raises(_lib.LdsrError) as e:
            _lib.cv_metrics_stations([np.ones((1, 8))], [np.ones(8)], [[np.array([2, 3])]])
        assert e.value.code == _lib.ERR_CUDA
        with pytest.raises(_lib.LdsrError) as e:
            _lib.construct_rec_stations([np.ones((1, 8))], [np.ones((1, 8))], [np.ones((1, 8))], [[1.0]], [[1.0]],
                                        [0.0])
        assert e.value.code == _lib.ERR_CUDA


def test_stations_reject_mismatched_inputs_with_the_single_station_messages():
    st = _stations()
    bad = dict(st[0], v=st[0]["v"][:, 1:])
    for fn in (L.cvLDS_stations, L.LDS_reconstruction_stations):
        with pytest.raises(ValueError, match="u and v must have the same number of time steps."):
            fn([st[1], bad], num_restarts=2, niter=10)
        with pytest.raises(ValueError, match="u and v must have the same number of time steps."):
            fn([st[1], dict(st[2], v=[st[2]["v"][0][:, 1:], None])], num_restarts=2, niter=10)
        with pytest.raises(ValueError, match="u and v cannot both be NULL"):
            fn([st[1], dict(st[0], u=None, v=None)], num_restarts=2, niter=10)
    with pytest.raises(ValueError, match="The last year of u is earlier"):
        L.cvLDS_stations([st[1], dict(st[0], start_year=1700)], num_restarts=2, niter=10)


def _draws(P, B):
    """Per station: its folds (if any) and its initial-value rows, unpadded."""
    out = []
    for S in P:
        th = [B["theta0"][f, :B["series"][B["group_series"][B["fit_group"][f]]]["p"]
                              + B["series"][B["group_series"][B["fit_group"][f]]]["q"] + 6]
              for f in range(S["f0"], S["f1"])]
        out.append(([np.asarray(z) for z in S.get("Z", [])], th))
    return out


def test_random_number_contract_with_r_random():
    st = _stations()
    st[1] = dict(st[1], Z=L.make_Z(st[1]["Qa"]["Qa"], 5, rng=L.RRandom(3)))  # given folds draw nothing
    for batch in (api.cv_batch, api.reconstruction_batch):
        together = _draws(*batch(st, num_restarts=3, rng=L.RRandom(2024)))
        rng = L.RRandom(2024)
        alone = [_draws(*batch([s], num_restarts=3, rng=rng))[0] for s in st]
        for (za, ta), (zb, tb) in zip(together, alone):
            assert len(za) == len(zb) and all(np.array_equal(a, b) for a, b in zip(za, zb))
            assert len(ta) == len(tb) and all(np.array_equal(a, b) for a, b in zip(ta, tb))
    # and what they draw is the reference's order: make_Z, then make_init fold-major, member-minor
    rng = L.RRandom(7)
    P, B = api.cv_batch(st[2:], num_restarts=2, rng=L.RRandom(7))
    Z = L.make_Z(st[2]["Qa"]["Qa"], rng=rng)
    assert all(np.array_equal(a, b) for a, b in zip(P[0]["Z"], Z))
    expect = [api.theta_to_vec(t) for _ in Z for p, q in ((3, 3), (1, 1)) for t in L.make_init(p, q, 2, rng)]
    assert all(np.array_equal(a, b) for a, b in zip(_draws(P, B)[0][1], expect))
    # stations are numbered station-major, groups fold-major / member-minor, theta rows padded to the widest
    assert B["theta0"].shape == (len(Z) * 2 * 2, 12) and B["group_series"][:4] == [0, 1, 0, 1]
