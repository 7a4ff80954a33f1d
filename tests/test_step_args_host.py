"""The single-step entry points (ldsr_smoother_batch, ldsr_propagate_batch, ldsr_mstep_batch and
ldsr_objective_batch) check their arguments before they look for a device: a malformed call is reported as
LDSR_ERR_ARG with or without a GPU, never as LDSR_ERR_CUDA."""
import ctypes as C

import numpy as np
import pytest

from ldsr_b200 import _lib

Y4 = np.array([0.1, np.nan, -0.2, 0.3])
TH = np.array([[0.5, 0.1, 0.8, 0.0, 1.0, 0.5, 0.0, 1.0]])  # p = q = 1: p + q + 6 = 8 entries


def _series(y):
    return [dict(y=y, u=np.ones((1, y.size)), v=None, p=1, q=1)]


MALFORMED = {  # (series, held, theta)
    "series_of_one_step": (_series(np.array([0.1])), None, TH),
    "infinite_y": (_series(np.array([0.1, np.inf, -0.2, 0.3])), None, TH),
    "held_out_step_past_the_end": (_series(Y4), [np.array([7])], TH),
    "theta_stride_below_p_q_6": (_series(Y4), None, TH[:, :7]),
}


def _code(call):
    with pytest.raises(_lib.LdsrError) as e:
        call()
    return e.value.code


@pytest.mark.parametrize("case", sorted(MALFORMED))
def test_malformed_batch_is_an_argument_error(case):
    series, held, theta = MALFORMED[case]
    T = series[0]["y"].size
    rows = [np.zeros(T)]
    assert _code(lambda: _lib.smoother_batch(series, [0], held, [0], theta)) == _lib.ERR_ARG
    assert _code(lambda: _lib.propagate_batch(series, [0], held, [0], theta)) == _lib.ERR_ARG
    assert _code(lambda: _lib.mstep_batch(series, [0], held, [0], rows, rows, rows, theta.shape[1])) == _lib.ERR_ARG
    for kind in _lib.OBJECTIVES:
        assert _code(lambda: _lib.objective_batch(series, [0], held, [0], theta, kind)) == _lib.ERR_ARG, kind


def test_missing_outputs_are_an_argument_error():
    pb = _lib.PackedBatch(_series(Y4), [0], None, [0], TH)
    L, err = _lib.lib(), C.create_string_buffer(256)
    rows, lik = np.zeros(Y4.size), np.zeros(1)
    d = _lib._d
    assert L.ldsr_smoother_batch(None, C.byref(pb.c), 1, None, d(rows), d(rows), None, d(lik), err, 256) == _lib.ERR_ARG
    assert L.ldsr_propagate_batch(None, C.byref(pb.c), 1, d(rows), None, d(rows), d(lik), err, 256) == _lib.ERR_ARG
    assert L.ldsr_mstep_batch(None, C.byref(pb.c), d(rows), d(rows), d(rows), None, None, err, 256) == _lib.ERR_ARG
