"""ctypes binding of libldsr_b200.so (include/ldsr_b200.h).  No fallback of any kind: if the
library is missing or no CUDA device is present, calls raise."""
import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.environ.get("LDSR_SO") or os.path.join(HERE, "libldsr_b200.so")  # LDSR_SO: development builds

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)

OK, ERR_ARG, ERR_CUDA, ERR_INTERRUPTED, ERR_UNSUPPORTED = 0, 1, 2, 3, 4
FIT_OK, FIT_SINGULAR, FIT_NONFINITE = 0, 1, 2

# every symbol include/ldsr_b200.h declares (checked by tests/test_abi_symbols.py)
EXPORTS = ("ldsr_abi_version", "ldsr_device_count", "ldsr_ctx_create", "ldsr_ctx_destroy", "ldsr_ctx_trim",
           "ldsr_em_batch", "ldsr_plan_create", "ldsr_plan_em", "ldsr_plan_set_theta0",
           "ldsr_plan_fetch", "ldsr_plan_destroy", "ldsr_smoother_batch", "ldsr_mstep_batch",
           "ldsr_propagate_batch", "ldsr_rep_batch", "ldsr_shard_groups", "ldsr_measure_fp64_peak",
           "ldsr_smoother_d_batch", "ldsr_cv_metrics_batch", "ldsr_construct_rec_batch",
           "ldsr_objective_batch", "ldsr_rep_batch_r", "ldsr_r_rng_create", "ldsr_r_rng_unif", "ldsr_r_rng_norm",
           "ldsr_r_rng_sample", "ldsr_r_rng_destroy", "ldsr_r_rnorm_device", "ldsr_last_device_ms",
           "ldsr_cv_metrics_stations", "ldsr_construct_rec_stations", "ldsr_posterior_rep_batch",
           "ldsr_posterior_stats_batch")


class LdsrError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("ldsr_b200 error %d: %s" % (code, msg))
        self.code = code


class Batch(C.Structure):
    _fields_ = [("n_series", C.c_int), ("T", _ip), ("p", _ip), ("q", _ip),
                ("y", C.POINTER(_dp)), ("u", C.POINTER(_dp)), ("v", C.POINTER(_dp)),
                ("n_groups", C.c_int), ("group_series", _ip), ("held_ptr", _ip), ("held_idx", _ip),
                ("n_fits", C.c_int), ("fit_group", _ip), ("theta0", _dp), ("theta_stride", C.c_int)]


class EmResult(C.Structure):
    _fields_ = [("theta", _dp), ("lik", _dp), ("iters", _ip), ("status", _ip), ("liks", _dp),
                ("best", _ip), ("X", _dp), ("Y", _dp), ("V", _dp), ("J", _dp)]


class StatsSpec(C.Structure):
    _fields_ = [("n_windows", C.c_int), ("windows", _ip), ("threshold", _dp), ("range", _ip)]


class StatsOut(C.Structure):
    _fields_ = [("wmin", _dp), ("wmin_at", _ip), ("wmax", _dp), ("wmax_at", _ip), ("run_len", _ip), ("run_at", _ip),
                ("deficit", _dp), ("deficit_at", _ip), ("n_runs", _ip)]


POLL_FN = C.CFUNCTYPE(C.c_int, C.c_void_p)


class Options(C.Structure):
    _fields_ = [("n_devices", C.c_int), ("devices", _ip), ("chunk_iters", C.c_int),
                ("poll", POLL_FN), ("poll_arg", C.c_void_p), ("variant", C.c_int),
                ("trace_liks", C.c_int)]


_lib = None


def lib():
    """Load the CUDA shared library; raises if it has not been built (no silent fallback)."""
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise LdsrError(ERR_CUDA, "%s not built: run `python -m ldsr_b200.build` "
                                      "(or __graft_entry__.build())" % SO_PATH)
        L = C.CDLL(SO_PATH)
        for name in EXPORTS:
            getattr(L, name).restype = C.c_int
        L.ldsr_ctx_destroy.restype = None
        L.ldsr_ctx_trim.restype = C.c_longlong
        L.ldsr_r_rng_destroy.restype = None
        L.ldsr_plan_destroy.restype = None
        L.ldsr_last_device_ms.restype = C.c_double
        _lib = L
    return _lib


def device_count():
    return lib().ldsr_device_count()


def _d(a):
    return None if a is None else a.ctypes.data_as(_dp)


def _i(a):
    return None if a is None else a.ctypes.data_as(_ip)


def _colmajor(m):
    """R-style [p, T] matrix -> flat column-major copy (time step contiguous)."""
    if m is None:
        return None, 0
    m = np.asarray(m, dtype=np.float64)
    if m.ndim == 1:
        m = m[None, :]
    return np.ascontiguousarray(m.T).ravel(), m.shape[0]


class PackedBatch:
    """Keeps every numpy buffer a C `ldsr_batch` points to alive."""

    def __init__(self, series, group_series, held, fit_group, theta0):
        ns = len(series)
        self.ys, self.us, self.vs = [], [], []
        Ts, ps, qs = [], [], []
        for s in series:
            y = np.ascontiguousarray(s["y"], dtype=np.float64).ravel()
            uf, pu = _colmajor(s.get("u"))
            vf, qv = _colmajor(s.get("v"))
            if uf is not None and uf.size != pu * y.size:
                raise ValueError("u must have %d columns" % y.size)
            if vf is not None and vf.size != qv * y.size:
                raise ValueError("v must have %d columns" % y.size)
            self.ys.append(y)
            self.us.append(uf)
            self.vs.append(vf)
            Ts.append(y.size)
            ps.append(int(s.get("p", pu)))
            qs.append(int(s.get("q", qv)))
        self.T = np.asarray(Ts, dtype=np.int32)
        self.p = np.asarray(ps, dtype=np.int32)
        self.q = np.asarray(qs, dtype=np.int32)
        PP = _dp * ns
        null = C.cast(None, _dp)
        self.yp = PP(*[_d(a) for a in self.ys])
        self.up = PP(*[_d(a) if a is not None else null for a in self.us])
        self.vp = PP(*[_d(a) if a is not None else null for a in self.vs])
        self.group_series = np.ascontiguousarray(group_series, dtype=np.int32)
        ng = self.group_series.size
        self.held_ptr = self.held_idx = None
        if held is not None:
            hp = np.zeros(ng + 1, dtype=np.int32)
            hp[1:] = np.cumsum([len(h) for h in held])
            self.held_ptr = hp
            if hp[-1] > 0:  # one conversion of the concatenation, not one per group
                self.held_idx = np.ascontiguousarray(np.concatenate(held, axis=None), dtype=np.int32)
            else:
                self.held_idx = np.zeros(1, dtype=np.int32)
        self.fit_group = np.ascontiguousarray(fit_group, dtype=np.int32)
        self.theta0 = np.ascontiguousarray(theta0, dtype=np.float64)
        if self.theta0.ndim != 2 or self.theta0.shape[0] != self.fit_group.size:
            raise ValueError("theta0 must be [n_fits, theta_stride]")
        self.n_fits = self.fit_group.size
        self.n_groups = ng
        self.stride = self.theta0.shape[1]
        self.traj_ptr = np.zeros(ng + 1, dtype=np.int64)
        self.traj_ptr[1:] = np.cumsum(self.T[self.group_series])
        self._fit_ptr = None
        self.c = Batch(ns, _i(self.T), _i(self.p), _i(self.q), self.yp, self.up, self.vp,
                       ng, _i(self.group_series), _i(self.held_ptr), _i(self.held_idx),
                       self.n_fits, _i(self.fit_group), _d(self.theta0), self.stride)


def _fit_ptr(self):
    """Row offsets of per-FIT trajectories (smoother / propagate outputs); made on first use."""
    if self._fit_ptr is None:
        self._fit_ptr = np.zeros(self.n_fits + 1, dtype=np.int64)
        self._fit_ptr[1:] = np.cumsum(self.T[self.group_series[self.fit_group]])
    return self._fit_ptr


PackedBatch.fit_ptr = property(_fit_ptr)


def _check(rc, err):
    if rc != OK:
        raise LdsrError(rc, err.value.decode("utf-8", "replace"))


def _options(n_devices=0, devices=None, chunk_iters=0, poll=None, trace_liks=False, keep=None, variant=None):
    o = Options()
    # kernel variant (ldsr_options.variant): 0 auto; development override through LDSR_VARIANT
    o.variant = int(os.environ.get("LDSR_VARIANT", "0")) if variant is None else int(variant)
    o.n_devices = int(n_devices)
    if devices is not None:
        dv = np.ascontiguousarray(devices, dtype=np.int32)
        keep.append(dv)
        o.devices = _i(dv)
        o.n_devices = dv.size
    o.chunk_iters = int(chunk_iters)
    if poll is not None:
        cb = POLL_FN(lambda _arg: int(bool(poll())))
        keep.append(cb)
        o.poll = cb
    o.trace_liks = int(bool(trace_liks))
    return o


class Ctx:
    """ldsr_ctx: device list + reusable device-memory pools (keeps cudaMalloc out of repeated calls)."""

    def __init__(self, devices=None, n_devices=0):
        self.h = C.c_void_p()
        dv = None if devices is None else np.ascontiguousarray(devices, dtype=np.int32)
        err = C.create_string_buffer(512)
        rc = lib().ldsr_ctx_create(int(dv.size if dv is not None else n_devices), _i(dv), C.byref(self.h), err, 512)
        _check(rc, err)

    def trim(self):
        """Hand the cached device blocks back to the driver: (bytes released, bytes still held)."""
        kept = C.c_longlong(0)
        freed = lib().ldsr_ctx_trim(self.h, C.byref(kept))
        return int(freed), int(kept.value)

    def close(self):
        if self.h:
            lib().ldsr_ctx_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class EmOutputs:
    """numpy buffers behind an ldsr_em_result."""

    def __init__(self, pb, niter, want_liks=False, want_traj=True):
        nf, ng = pb.n_fits, pb.n_groups
        # the library writes every element of every output except the tail of a theta row beyond
        # its series' p + q + 6 (kept NaN here)
        same_width = bool(np.all(pb.p + pb.q + 6 == pb.stride))
        self.theta = np.empty((nf, pb.stride)) if same_width else np.full((nf, pb.stride), np.nan)
        self.lik = np.empty(nf)
        self.iters = np.empty(nf, dtype=np.int32)
        self.status = np.empty(nf, dtype=np.int32)
        self.best = np.empty(ng, dtype=np.int32)
        self.liks = np.empty((nf, niter)) if want_liks else None
        tot = int(pb.traj_ptr[-1])
        self.X, self.Y, self.V, self.J = ((np.empty(tot) for _ in range(4)) if want_traj else (None,) * 4)
        self.c = EmResult(_d(self.theta), _d(self.lik), _i(self.iters), _i(self.status),
                          _d(self.liks), _i(self.best), _d(self.X), _d(self.Y), _d(self.V), _d(self.J))

    def as_dict(self, pb):
        d = dict(theta=self.theta, lik=self.lik, iters=self.iters, status=self.status,
                 best=self.best, traj_ptr=pb.traj_ptr)
        if self.liks is not None:
            d["liks"] = self.liks
        if self.X is not None:
            d.update(X=self.X, Y=self.Y, V=self.V, J=self.J)
        return d


def em_batch(series, group_series, held, fit_group, theta0, niter=1000, tol=1e-5, n_devices=1,
             devices=None, chunk_iters=0, poll=None, want_liks=False, want_traj=True, ctx=None, variant=None):
    """ldsr_em_batch with host (numpy) buffers.  Same argument shapes as oracle.em_batch."""
    pb = PackedBatch(series, group_series, held, fit_group, theta0)
    out = EmOutputs(pb, niter, want_liks, want_traj)
    keep = []
    opt = _options(n_devices, devices, chunk_iters, poll, keep=keep, variant=variant)
    err = C.create_string_buffer(512)
    rc = lib().ldsr_em_batch(ctx.h if isinstance(ctx, Ctx) else ctx, C.byref(pb.c), int(niter), C.c_double(tol),
                             C.byref(opt), C.byref(out.c), err, 512)
    _check(rc, err)
    return out.as_dict(pb)


class Plan:
    """Device-resident batch (ldsr_plan_*): inputs are uploaded once, EM runs from HBM."""

    def __init__(self, series, group_series, held, fit_group, theta0, device=0):
        self.pb = PackedBatch(series, group_series, held, fit_group, theta0)
        self.h = C.c_void_p()
        err = C.create_string_buffer(512)
        rc = lib().ldsr_plan_create(C.byref(self.pb.c), int(device), C.byref(self.h), err, 512)
        _check(rc, err)
        self.niter = None

    def em(self, niter=1000, tol=1e-5, chunk_iters=0, stream=None, trace_liks=False, poll=None, variant=None):
        keep = []
        opt = _options(chunk_iters=chunk_iters, poll=poll, trace_liks=trace_liks, keep=keep, variant=variant)
        stats = (C.c_longlong * 8)()
        err = C.create_string_buffer(512)
        rc = lib().ldsr_plan_em(self.h, int(niter), C.c_double(tol), C.byref(opt),
                                C.c_void_p(stream or 0), stats, err, 512)
        _check(rc, err)
        self.niter = niter
        self.trace = bool(trace_liks)
        return dict(launches=stats[0], chunks=stats[1], esteps=stats[2], em_kernel_ns=stats[3],
                    kernel=("em_chunk_kernel", "em_split_kernel", "em_wide_kernel", "em_scan_kernel")[stats[4]],
                    shared_slots=stats[5])

    def set_theta0(self, theta0):
        th = np.ascontiguousarray(theta0, dtype=np.float64)
        assert th.shape == self.pb.theta0.shape
        err = C.create_string_buffer(512)
        _check(lib().ldsr_plan_set_theta0(self.h, _d(th), err, 512), err)

    def fetch(self, want_traj=True):
        out = EmOutputs(self.pb, self.niter, self.trace, want_traj)
        err = C.create_string_buffer(512)
        _check(lib().ldsr_plan_fetch(self.h, C.byref(out.c), err, 512), err)
        return out.as_dict(self.pb)

    def close(self):
        if self.h:
            lib().ldsr_plan_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _rows(flat, ptr):
    return [flat[ptr[i]:ptr[i + 1]] for i in range(len(ptr) - 1)]


def smoother_batch(series, group_series, held, fit_group, theta, stdlik=True, ctx=None):
    pb = PackedBatch(series, group_series, held, fit_group, theta)
    tot = int(pb.fit_ptr[-1])
    X, Y, V, J = (np.empty(tot) for _ in range(4))
    lik = np.empty(pb.n_fits)
    err = C.create_string_buffer(512)
    rc = lib().ldsr_smoother_batch(ctx, C.byref(pb.c), int(stdlik), _d(X), _d(Y), _d(V), _d(J), _d(lik), err, 512)
    _check(rc, err)
    return dict(X=_rows(X, pb.fit_ptr), Y=_rows(Y, pb.fit_ptr), V=_rows(V, pb.fit_ptr),
                J=_rows(J, pb.fit_ptr), lik=lik)


def mstep_batch(series, group_series, held, fit_group, X, V, J, theta_stride, ctx=None):
    nf = len(fit_group)
    pb = PackedBatch(series, group_series, held, fit_group, np.zeros((nf, theta_stride)))
    Xf, Vf, Jf = (np.ascontiguousarray(np.concatenate([np.ravel(r) for r in a]), dtype=np.float64)
                  for a in (X, V, J))
    assert Xf.size == pb.fit_ptr[-1]
    th = np.full((nf, theta_stride), np.nan)
    st = np.zeros(nf, dtype=np.int32)
    err = C.create_string_buffer(512)
    rc = lib().ldsr_mstep_batch(ctx, C.byref(pb.c), _d(Xf), _d(Vf), _d(Jf), _d(th), _i(st), err, 512)
    _check(rc, err)
    return dict(theta=th, status=st)


def propagate_batch(series, group_series, held, fit_group, theta, stdlik=True, ctx=None):
    pb = PackedBatch(series, group_series, held, fit_group, theta)
    tot = int(pb.fit_ptr[-1])
    X, Y, V = (np.empty(tot) for _ in range(3))
    lik = np.empty(pb.n_fits)
    err = C.create_string_buffer(512)
    rc = lib().ldsr_propagate_batch(ctx, C.byref(pb.c), int(stdlik), _d(X), _d(Y), _d(V), _d(lik), err, 512)
    _check(rc, err)
    return dict(X=_rows(X, pb.fit_ptr), Y=_rows(Y, pb.fit_ptr), V=_rows(V, pb.fit_ptr), lik=lik)


def rep_batch(theta, u, v, n, n_reps, z=None, seed=0, mu=0.0, exp_trans=True, p=None, q=None,
              want=("simX", "simY", "simQ"), ctx=None, r_seed=None):
    """ldsr_rep_batch; with r_seed the noise is what R draws after set.seed(r_seed) (ldsr_rep_batch_r)."""
    uf, pu = _colmajor(u)
    vf, qv = _colmajor(v)
    p = pu if p is None else p
    q = qv if q is None else q
    theta = np.ascontiguousarray(theta, dtype=np.float64)
    assert theta.size == p + q + 6
    zz = None
    if z is not None:
        zz = np.ascontiguousarray(z, dtype=np.float64)
        assert zz.size == n_reps * (1 + 2 * n)
    outs = {k: (np.empty((n_reps, n)) if k in want else None) for k in ("simX", "simY", "simQ")}
    err = C.create_string_buffer(512)
    if r_seed is not None and z is None:
        rc = lib().ldsr_rep_batch_r(ctx, _d(theta), _d(uf), _d(vf), int(n), int(p), int(q), int(n_reps),
                                    C.c_uint(int(r_seed) & 0xFFFFFFFF), C.c_double(mu), int(exp_trans),
                                    _d(outs["simX"]), _d(outs["simY"]), _d(outs["simQ"]), err, 512)
    else:
        rc = lib().ldsr_rep_batch(ctx, _d(theta), _d(uf), _d(vf), int(n), int(p), int(q), int(n_reps), _d(zz),
                                  C.c_ulonglong(seed), C.c_double(mu), int(exp_trans), _d(outs["simX"]),
                                  _d(outs["simY"]), _d(outs["simQ"]), err, 512)
    _check(rc, err)
    res = {k: v for k, v in outs.items() if v is not None}
    res["device_ms"] = float(lib().ldsr_last_device_ms())  # CUDA-event time of the replicate kernels
    return res


def posterior_rep_batch(series, group_series, held, fit_group, theta, n_reps, z=None, seed=0, mu=None, transform="log",
                        lams=None, want=("simX", "simY", "simQ"), ctx=None):
    """ldsr_posterior_rep_batch: n_reps replicates of every fit conditioned on its group's y (forward filtering,
    backward sampling).  Batch arguments as smoother_batch; theta [n_fits, stride] holds one model per fit.
    z (optional): 2 * n_reps * sum(T) standard normals in the ABI's layout; mu, lams: per fit (lams with
    transform="boxcox" only).  Returns, per requested output, a list over fits of [n_reps, T_f] arrays (views of
    one replicate-major buffer), and the kernels' device time."""
    pb = PackedBatch(series, group_series, held, fit_group, theta)
    nf = pb.n_fits
    tot = int(pb.fit_ptr[-1]) * int(n_reps)
    zz = None
    if z is not None:
        zz = np.ascontiguousarray(z, dtype=np.float64).ravel()
        if zz.size != 2 * tot:
            raise ValueError("z must hold 2 * n_reps * sum(T) = %d values" % (2 * tot))
    code = TRANSFORMS[transform] if isinstance(transform, str) else int(transform)
    mu_a = None if mu is None else np.ascontiguousarray(np.broadcast_to(np.asarray(mu, dtype=np.float64), (nf,)))
    lam_a = None if lams is None else np.ascontiguousarray(np.broadcast_to(np.asarray(lams, dtype=np.float64), (nf,)))
    outs = {k: (np.empty(tot) if k in want else None) for k in ("simX", "simY", "simQ")}
    err = C.create_string_buffer(512)
    rc = lib().ldsr_posterior_rep_batch(ctx.h if isinstance(ctx, Ctx) else ctx, C.byref(pb.c), int(n_reps), _d(zz),
                                        C.c_ulonglong(int(seed)), _d(mu_a), code, _d(lam_a), _d(outs["simX"]),
                                        _d(outs["simY"]), _d(outs["simQ"]), err, 512)
    _check(rc, err)
    ptr = pb.fit_ptr * int(n_reps)
    T = np.diff(pb.fit_ptr)
    res = {k: [o[ptr[f]:ptr[f + 1]].reshape(int(n_reps), int(T[f])) for f in range(nf)]
           for k, o in outs.items() if o is not None}
    res["device_ms"] = float(lib().ldsr_last_device_ms())
    return res


WINDOW_STATS = ("wmin", "wmin_at", "wmax", "wmax_at")
RUN_STATS = ("run_len", "run_at", "deficit", "deficit_at", "n_runs")


def posterior_stats_batch(series, group_series, held, fit_group, theta, n_reps, z=None, seed=0, mu=None,
                          transform="log", lams=None, windows=(10,), threshold=None, ranges=None, want=None, ctx=None):
    """ldsr_posterior_stats_batch: the drought statistics of posterior_rep_batch's replicates (same arguments, the
    same draws), reduced on the device.  windows: up to 4 moving-mean lengths in 1..64; threshold: per fit, on the Q
    scale (None: no run statistics); ranges: [n_fits, 2] step ranges [lo, hi) (None: whole series).  want: the
    outputs to return (default: all that the spec defines).  Returns window outputs shaped [n_windows, n_fits,
    n_reps], run outputs [n_fits, n_reps] (steps as int32, -1 where undefined), and the device time."""
    pb = PackedBatch(series, group_series, held, fit_group, theta)
    nf, n_reps = pb.n_fits, int(n_reps)
    zz = None
    if z is not None:
        zz = np.ascontiguousarray(z, dtype=np.float64).ravel()
        if zz.size != 2 * int(pb.fit_ptr[-1]) * n_reps:
            raise ValueError("z must hold 2 * n_reps * sum(T) = %d values" % (2 * int(pb.fit_ptr[-1]) * n_reps))
    code = TRANSFORMS[transform] if isinstance(transform, str) else int(transform)
    mu_a = None if mu is None else np.ascontiguousarray(np.broadcast_to(np.asarray(mu, dtype=np.float64), (nf,)))
    lam_a = None if lams is None else np.ascontiguousarray(np.broadcast_to(np.asarray(lams, dtype=np.float64), (nf,)))
    win = np.ascontiguousarray(np.atleast_1d(np.asarray(windows if windows is not None else (), dtype=np.int32)))
    thr = None if threshold is None else np.ascontiguousarray(
        np.broadcast_to(np.asarray(threshold, dtype=np.float64), (nf,)))
    rng = None if ranges is None else np.ascontiguousarray(np.broadcast_to(np.asarray(ranges, dtype=np.int32),
                                                                           (nf, 2)))
    if want is None:
        want = WINDOW_STATS + (RUN_STATS if thr is not None else ())
    nw = win.size
    outs = {}
    for k in WINDOW_STATS:
        if k in want:
            outs[k] = np.empty((nw, nf, n_reps), dtype=np.int32 if k.endswith("_at") else np.float64)
    for k in RUN_STATS:
        if k in want:
            outs[k] = np.empty((nf, n_reps), dtype=np.float64 if k == "deficit" else np.int32)
    spec = StatsSpec(nw, _i(win) if nw else None, _d(thr), _i(rng))
    out = StatsOut(*(_d(outs.get(k)) if k in ("wmin", "wmax", "deficit") else _i(outs.get(k))
                     for k, _ in StatsOut._fields_))
    err = C.create_string_buffer(512)
    rc = lib().ldsr_posterior_stats_batch(ctx.h if isinstance(ctx, Ctx) else ctx, C.byref(pb.c), n_reps, _d(zz),
                                          C.c_ulonglong(int(seed)), _d(mu_a), code, _d(lam_a), C.byref(spec),
                                          C.byref(out), err, 512)
    _check(rc, err)
    outs["device_ms"] = float(lib().ldsr_last_device_ms())
    return outs


class RRandom:
    """R's default generators after set.seed(seed) (ldsr_r_rng_*): runif / rnorm with R's state
    semantics, so that a seeded reference run (make_init, R/LDS_reconstruction.R:14-30) can be
    reproduced from outside R.  Host-side and sequential: meant for initial values, not bulk noise."""

    def __init__(self, seed):
        self.h = C.c_void_p()
        err = C.create_string_buffer(256)
        _check(lib().ldsr_r_rng_create(C.c_uint(int(seed) & 0xFFFFFFFF), C.byref(self.h), err, 256), err)

    def runif(self, n=1, a=0.0, b=1.0):
        out = np.empty(int(n))
        err = C.create_string_buffer(256)
        _check(lib().ldsr_r_rng_unif(self.h, int(n), C.c_double(a), C.c_double(b), _d(out), err, 256), err)
        return out

    def uniform(self, low=0.0, high=1.0, size=None):
        """numpy-Generator spelling of runif, so that api.make_init(p, q, n, RRandom(seed)) draws what
        `set.seed(seed); replicate(n, make_init(p, q))` draws."""
        r = self.runif(1 if size is None else size, low, high)
        return float(r[0]) if size is None else r

    def sample_int(self, n, size=None):
        """sample.int(n, size) without replacement (1-based)."""
        size = n if size is None else size
        out = np.empty(int(size), dtype=np.int32)
        err = C.create_string_buffer(256)
        _check(lib().ldsr_r_rng_sample(self.h, int(n), int(size), _i(out), err, 256), err)
        return out

    def choice(self, a, size, replace=False):
        """numpy-Generator spelling of R's sample(a, size): api.make_Z(obs, ..., rng=RRandom(seed)) makes the
        folds `set.seed(seed); make_Z(obs, ...)` makes.  Like R, a single number a >= 1 means 1:a."""
        if replace:
            raise ValueError("only sampling without replacement is needed by the reference (R/utils.R:96,98)")
        a = np.atleast_1d(np.asarray(a))
        if a.size == 1 and a[0] >= 1:
            return self.sample_int(int(a[0]), size)
        return a[self.sample_int(a.size, size) - 1]

    def rnorm(self, n=1, mean=0.0, sd=1.0):
        out = np.empty(int(n))
        err = C.create_string_buffer(256)
        _check(lib().ldsr_r_rng_norm(self.h, int(n), _d(out), err, 256), err)
        return mean + sd * out  # rnorm.c: mu + sigma * norm_rand()

    def close(self):
        if self.h:
            lib().ldsr_r_rng_destroy(self.h)
            self.h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def r_rnorm_device(seed, n, device=0):
    """set.seed(seed); rnorm(n), generated on the GPU."""
    out = np.empty(int(n))
    err = C.create_string_buffer(256)
    _check(lib().ldsr_r_rnorm_device(int(device), C.c_uint(int(seed) & 0xFFFFFFFF), C.c_longlong(int(n)), _d(out),
                                     err, 256), err)
    return out


def measure_fp64_peak(device=0):
    """Measured DFMA rate of the device in TFLOP/s (the FP64 roofline denominator)."""
    t = C.c_double()
    err = C.create_string_buffer(512)
    _check(lib().ldsr_measure_fp64_peak(int(device), C.byref(t), err, 512), err)
    return t.value


def shard_groups(series, group_series, held, fit_group, theta0, n_shards):
    """ldsr_shard_groups: the group -> device partition of ldsr_em_batch (host logic only)."""
    pb = PackedBatch(series, group_series, held, fit_group, theta0)
    out = np.empty(pb.n_groups, dtype=np.int32)
    err = C.create_string_buffer(512)
    _check(lib().ldsr_shard_groups(C.byref(pb.c), int(n_shards), _i(out), err, 512), err)
    return out


def smoother_d(d, y, u, v, theta, stdlik=True, method=1, chunk=0, device=0, want=("X", "V", "Y")):
    """ldsr_smoother_d_batch: Kalman/RTS smoother for state dimension d (1..4), sequential
    (method=0) or associative scan over time (method=1).  y [T]; u [p,T] | None; v [q,T] | None;
    theta [n_fits, len] flat (A d*d | B d*p | C d | D q | Q d*d | R | mu1 d | V1 d*d)."""
    y = np.ascontiguousarray(y, dtype=np.float64).ravel()
    T = y.size
    uf = None if u is None else np.ascontiguousarray(np.asarray(u, dtype=np.float64).T)
    vf = None if v is None else np.ascontiguousarray(np.asarray(v, dtype=np.float64).T)
    p = 0 if uf is None else uf.shape[1]
    q = 0 if vf is None else vf.shape[1]
    th = np.atleast_2d(np.ascontiguousarray(theta, dtype=np.float64))
    nf = th.shape[0]
    X = np.empty((nf, T, d)) if "X" in want else None
    V = np.empty((nf, T, d, d)) if "V" in want else None
    Y = np.empty((nf, T)) if "Y" in want else None
    lik = np.empty(nf)
    ms = C.c_double()
    err = C.create_string_buffer(512)
    rc = lib().ldsr_smoother_d_batch(int(device), int(d), T, p, q, _d(y), _d(uf), _d(vf), nf, _d(th), th.shape[1],
                                     int(bool(stdlik)), int(method), int(chunk), _d(X), _d(V), _d(Y), _d(lik),
                                     C.byref(ms), err, 512)
    _check(rc, err)
    return dict(X=X, V=V, Y=Y, lik=lik, kernel_ms=ms.value)


METRIC_NAMES = ("R2", "RE", "CE", "nRMSE", "KGE")


def cv_metrics(sim, obs, Z, exp_trans=False, device=0):
    """ldsr_cv_metrics_batch: calculate_metrics (R/utils.R:56-70) for every fold on the device.
    sim [n_folds, n]; obs [n]; Z: list of 1-based hold-out index vectors.  Returns [n_folds, 5]."""
    sim = np.ascontiguousarray(sim, dtype=np.float64)
    obs = np.ascontiguousarray(obs, dtype=np.float64)
    nf, n = sim.shape
    zp = np.zeros(nf + 1, dtype=np.int32)
    zp[1:] = np.cumsum([len(z) for z in Z])
    zi = np.ascontiguousarray(np.concatenate([np.asarray(z, dtype=np.int32) for z in Z]), dtype=np.int32)
    out = np.empty((nf, 5))
    err = C.create_string_buffer(512)
    _check(lib().ldsr_cv_metrics_batch(int(device), int(n), int(nf), _d(sim), _d(obs), _i(zp), _i(zi),
                                       int(bool(exp_trans)), _d(out), err, 512), err)
    return out


def _ptr(lengths):
    out = np.zeros(len(lengths) + 1, dtype=np.int32)
    out[1:] = np.cumsum(lengths)
    return out


def cv_metrics_stations(sims, obss, Zs, exp_trans=False, device=0):
    """ldsr_cv_metrics_stations: cv_metrics for several stations of different lengths in one launch.
    sims[s] [n_folds_s, n_s]; obss[s] [n_s]; Zs[s]: station s's folds, 1-based into obss[s].
    Returns one [n_folds_s, 5] array per station."""
    sims = [np.atleast_2d(np.asarray(a, dtype=np.float64)) for a in sims]
    obss = [np.asarray(a, dtype=np.float64).ravel() for a in obss]
    if not (len(sims) == len(obss) == len(Zs)):
        raise ValueError("one sim matrix, target and fold list per station")
    n = np.asarray([o.size for o in obss], dtype=np.int32)
    for s, (a, z) in enumerate(zip(sims, Zs)):
        if a.shape != (len(z), n[s]):
            raise ValueError("station %d: sim must be [%d folds, %d]" % (s, len(z), n[s]))
    fp = _ptr([len(z) for z in Zs])
    folds = [np.asarray(z, dtype=np.int32).ravel() for zs in Zs for z in zs]
    zp = _ptr([z.size for z in folds])
    zi = np.ascontiguousarray(np.concatenate(folds + [np.zeros(1, dtype=np.int32)]))
    sim = np.ascontiguousarray(np.concatenate([a.ravel() for a in sims]))
    obs = np.ascontiguousarray(np.concatenate(obss))
    out = np.empty((int(fp[-1]), 5))
    err = C.create_string_buffer(512)
    _check(lib().ldsr_cv_metrics_stations(int(device), len(obss), _i(n), _i(fp), _d(sim), _d(obs), _i(zp), _i(zi),
                                          int(bool(exp_trans)), _d(out), err, 512), err)
    return [out[fp[s]:fp[s + 1]] for s in range(len(obss))]


REC_COLUMNS = ("X", "Xl", "Xu", "Q", "Ql", "Qu")
TRANSFORMS = {"none": 0, "log": 1, "boxcox": 2}


def construct_rec(X, V, Y, C_, R_, mu, transform="log", lam=0.0, device=0):
    """ldsr_construct_rec_batch: construct_rec (R/LDS_reconstruction.R:190-212) for every ensemble member
    and the ensemble mean of X and Q.  X, V, Y: [n, T]; C_, R_: [n].  Returns (out [n, 6, T], mean [2, T])."""
    X, V, Y = (np.ascontiguousarray(np.atleast_2d(a), dtype=np.float64) for a in (X, V, Y))
    n, T = X.shape
    Cv = np.ascontiguousarray(np.broadcast_to(np.asarray(C_, dtype=np.float64).ravel(), (n,)))
    Rv = np.ascontiguousarray(np.broadcast_to(np.asarray(R_, dtype=np.float64).ravel(), (n,)))
    out = np.empty((n, 6, T))
    mean = np.empty((2, T))
    err = C.create_string_buffer(512)
    _check(lib().ldsr_construct_rec_batch(int(device), int(n), int(T), _d(X), _d(V), _d(Y), _d(Cv), _d(Rv),
                                          C.c_double(mu), int(TRANSFORMS[transform]), C.c_double(lam), _d(out),
                                          _d(mean), err, 512), err)
    return out, mean


def construct_rec_stations(Xs, Vs, Ys, Cs, Rs, mus, transform="log", lams=None, device=0):
    """ldsr_construct_rec_stations: construct_rec for the members of several stations of different lengths in
    one launch.  Xs[s], Vs[s], Ys[s]: [n_s, T_s]; Cs[s], Rs[s]: [n_s]; mus[s], lams[s]: station s's mean and
    Box-Cox lambda.  Returns one (out [n_s, 6, T_s], mean [2, T_s]) pair per station."""
    S = len(Xs)
    Xs, Vs, Ys = ([np.atleast_2d(np.asarray(a, dtype=np.float64)) for a in arrs] for arrs in (Xs, Vs, Ys))
    T = np.asarray([x.shape[1] for x in Xs], dtype=np.int32)
    nm = [x.shape[0] for x in Xs]
    for s in range(S):
        if Vs[s].shape != Xs[s].shape or Ys[s].shape != Xs[s].shape:
            raise ValueError("station %d: X, V and Y must have the same shape" % s)
    mp = _ptr(nm)
    X, V, Y = (np.ascontiguousarray(np.concatenate([a.ravel() for a in arrs])) for arrs in (Xs, Vs, Ys))
    Cv, Rv = (np.ascontiguousarray(np.concatenate([np.broadcast_to(np.asarray(c, dtype=np.float64).ravel(), (k,))
                                                   for c, k in zip(arrs, nm)])) for arrs in (Cs, Rs))
    mu = np.ascontiguousarray(mus, dtype=np.float64)
    lam = np.ascontiguousarray(np.zeros(S) if lams is None else [0.0 if l is None else l for l in lams],
                               dtype=np.float64)
    if mu.shape != (S,) or lam.shape != (S,):
        raise ValueError("one mu and one lambda per station")
    rows = np.concatenate([[0], np.cumsum(np.asarray(nm) * T)])
    years = np.concatenate([[0], np.cumsum(T)])
    out = np.empty(6 * int(rows[-1]))
    mean = np.empty(2 * int(years[-1]))
    err = C.create_string_buffer(512)
    _check(lib().ldsr_construct_rec_stations(int(device), S, _i(T), _i(mp), _d(X), _d(V), _d(Y), _d(Cv), _d(Rv),
                                             _d(mu), _d(lam), int(TRANSFORMS[transform]), _d(out), _d(mean), err, 512),
           err)
    return [(out[6 * rows[s]:6 * rows[s + 1]].reshape(nm[s], 6, T[s]), mean[2 * years[s]:2 * years[s + 1]].reshape(2, T[s]))
            for s in range(S)]


OBJECTIVES = {"penalized_likelihood": 0, "negLogLik": 1, "ssqTrain": 2}


def objective_batch(series, group_series, held, fit_group, theta, kind, lam=1.0, ctx=None):
    """ldsr_objective_batch: the objective functions of the reference's experimental learners
    (R/LDS_GA.R:28-44, 136-147) for a whole population of parameter vectors in one call."""
    pb = PackedBatch(series, group_series, held, fit_group, theta)
    out = np.empty(pb.c.n_fits)
    err = C.create_string_buffer(512)
    _check(lib().ldsr_objective_batch(ctx.h if isinstance(ctx, Ctx) else ctx, C.byref(pb.c), int(OBJECTIVES[kind]),
                                      C.c_double(lam), _d(out), err, 512), err)
    return out
