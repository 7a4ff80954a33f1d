"""ldsr_b200 -- B200-native (sm_100a, FP64, hand-written CUDA) batched EM engine behind ldsr's API.

Layout:
  csrc/      CUDA kernels + the C ABI (include/ldsr_b200.h) -> libldsr_b200.so
  _lib.py    ctypes binding of the C ABI
  api.py     Python mirror of the reference's R functions for this path
  r/         R-side shim sources (.Call glue + drop-in R wrappers); not buildable here (no R)
  build.py   in-tree nvcc build
There is no CPU implementation in this package; oracle/ (test infrastructure) is never imported.
"""
from . import _lib  # noqa: F401
from .api import (Kalman_smoother, Mstep, LDS_EM, LDS_EM_restart, LDS_reconstruction, cvLDS,  # noqa: F401
                  LDS_reconstruction_stations, cvLDS_stations,
                  one_lds_cv, propagate, LDS_rep, one_LDS_rep, LDS_rep_posterior, make_init, make_Z, calculate_metrics,
                  LDS_rep_posterior_stats, LDS_rep_posterior_yearly, LDS_rep_posterior_quantiles,
                  theta_to_vec, vec_to_theta, Kalman_smoother_d, tbrm)
from ._lib import RRandom  # noqa: F401  (R's generators after set.seed: reproducible restarts / replicates)
