/*
 * ldsr_b200.h -- C ABI of the B200-native batched EM engine for ldsr's LDS model.
 *
 * Model (reference: vignettes/ldsr.Rmd:25-33, src/EM.cpp:20 -- scalar state, scalar output):
 *     x[t+1] = A x[t] + B u[t] + w[t],  w ~ N(0,Q)
 *     y[t]   = C x[t] + D v[t] + e[t],  e ~ N(0,R)
 *
 * This library replaces, as ONE batched call each, what the reference does one fit at a time
 * through its Rcpp `.Call` entry points (src/RcppExports.cpp:133-136) fanned out by R's
 * foreach (R/LDS_reconstruction.R:46, :242, :373-381):
 *
 *     reference entry point (file:line)                     replaced by
 *     ----------------------------------------------------  -------------------------------
 *     _ldsr_LDS_EM          src/RcppExports.cpp:40-53       ldsr_em_batch / ldsr_plan_em
 *       + LDS_EM_restart    R/LDS_reconstruction.R:42-62      (restart fan-out + selection)
 *       + one_lds_cv/cvLDS  R/LDS_reconstruction.R:270-285,     (hold-out folds = groups)
 *                             :372-382
 *     _ldsr_Kalman_smoother src/RcppExports.cpp:11-23       ldsr_smoother_batch
 *     _ldsr_Mstep           src/RcppExports.cpp:26-37       ldsr_mstep_batch
 *     _ldsr_propagate       src/RcppExports.cpp:56-68       ldsr_propagate_batch
 *     one_LDS_rep / LDS_rep R/stochastics.R:18-63           ldsr_rep_batch
 *
 * Conventions
 *   - All numerics are IEEE FP64 on the GPU.  There is NO CPU fallback: without a CUDA device
 *     every compute entry point returns LDSR_ERR_CUDA.
 *   - theta is flat, in the reference's own vector order (R/LDS_GA.R:6-16):
 *         [A, B_1..B_p, C, D_1..D_q, Q, R, mu1, V1]          length p+q+6
 *   - u is p x T, v is q x T, both COLUMN-major exactly as R stores them (the p-vector of one
 *     time step is contiguous: u[t*p + j]); y has T entries with NaN / NA_real_ = missing.
 *     +-Inf in y is rejected (LDSR_ERR_ARG): the reference treats it as observed in the filter
 *     and as missing in the likelihood (EM.cpp:61 vs :113), which is garbage either way.
 *   - u == NULL (v == NULL) replaces the reference's `matrix(0)` one-column sentinel
 *     (EM.cpp:50,71,157,189; R/LDS_reconstruction.R:131-136): the input term is dropped and
 *     B (D) is returned as zeros.  p (q) still gives the length of B (D) inside theta.
 *   - Every function returns an LDSR_* code; on error a message is written to errbuf (if given).
 *     Nothing is thrown across the ABI, nothing is retained after return except through an
 *     explicit ldsr_plan / ldsr_ctx handle.  The caller owns every buffer it passes.
 *   - Thread-safety: a ctx/plan must be used from one thread at a time.  Worker threads (one per
 *     GPU) are internal and never call back into the host language; the optional poll callback
 *     runs on the CALLING thread (so an R shim can run R_CheckUserInterrupt there).
 */
#ifndef LDSR_B200_H
#define LDSR_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define LDSR_ABI_VERSION 1

/* return codes */
#define LDSR_OK 0
#define LDSR_ERR_ARG 1         /* bad argument (message says which) */
#define LDSR_ERR_CUDA 2        /* CUDA runtime / no device / out of memory */
#define LDSR_ERR_INTERRUPTED 3 /* poll callback asked to stop */
#define LDSR_ERR_UNSUPPORTED 4 /* p or q beyond LDSR_MAX_PQ */

/* per-fit status written to ldsr_em_result.status */
#define LDSR_FIT_OK 0
#define LDSR_FIT_SINGULAR 1  /* Gram block (u u' or v v' over the fit's steps) not invertible:
                                the reference's arma::inv would throw (EM.cpp:166,198) */
#define LDSR_FIT_NONFINITE 2 /* final log-likelihood is NaN/Inf (fit ran to niter) */

#define LDSR_MAX_PQ 32 /* largest supported nrow(u), nrow(v) */
#define LDSR_MAX_STATE_DIM 4 /* ldsr_smoother_d_batch: largest state dimension */

/* ---- problem description (all HOST pointers) --------------------------------------------- */
typedef struct {
    /* series: one (y,u,v) triple.  LDS_reconstruction/cvLDS with a list of u/v (ensemble) or a
     * multi-station job has several. */
    int n_series;
    const int *T;             /* [n_series] time steps (>= 2)                               */
    const int *p;             /* [n_series] length of B                                      */
    const int *q;             /* [n_series] length of D                                      */
    const double *const *y;   /* [n_series] -> T doubles, NaN = missing                      */
    const double *const *u;   /* [n_series] -> p*T doubles column-major, or NULL             */
    const double *const *v;   /* [n_series] -> q*T doubles column-major, or NULL             */
    /* groups: one (series, hold-out fold).  The fits of a group compete in the
     * LDS_EM_restart selection (R/LDS_reconstruction.R:50-58).  held_idx lists the 0-based
     * time steps forced to missing for the group (`y[instPeriod][z] <- NA`, :274), CSR. */
    int n_groups;
    const int *group_series;  /* [n_groups]                                                  */
    const int *held_ptr;      /* [n_groups+1], may be NULL when no group holds anything out  */
    const int *held_idx;      /* [held_ptr[n_groups]]                                        */
    /* fits: one EM run from one initial theta.  Fits of one group must be contiguous and
     * groups must appear in increasing order (fit_group non-decreasing). */
    int n_fits;
    const int *fit_group;     /* [n_fits]                                                    */
    const double *theta0;     /* [n_fits * theta_stride] flat thetas                         */
    int theta_stride;         /* >= max(p+q+6) over series                                   */
} ldsr_batch;

/* ---- EM results (HOST pointers; any pointer may be NULL = not wanted) ------------------- */
typedef struct {
    double *theta;   /* [n_fits * theta_stride] theta the LAST E-step ran with (EM.cpp:276)  */
    double *lik;     /* [n_fits] final standardised log-likelihood (NaN if status==SINGULAR) */
    int *iters;      /* [n_fits] number of E-steps = length(liks) of the reference           */
    int *status;     /* [n_fits] LDSR_FIT_*                                                  */
    double *liks;    /* [n_fits * niter] likelihood trace, NaN-padded                        */
    int *best;       /* [n_groups] selected fit (index into the fit table), -1 if none       */
    /* smoothed trajectories of each group's selected fit (fit$X, $Y, $V, $J of the winner),
     * row g starts at traj_ptr[g] where traj_ptr is the exclusive prefix sum of T[series(g)].
     * For groups with best == -1 the rows are NaN. */
    double *X, *Y, *V, *J;
} ldsr_em_result;

typedef int (*ldsr_poll_fn)(void *arg); /* return nonzero to abort; called between chunks */

typedef struct {
    int n_devices;       /* 0 = all visible devices (never more than n_groups)               */
    const int *devices;  /* [n_devices] CUDA ordinals, NULL = 0..n_devices-1                 */
    int chunk_iters;     /* EM iterations per kernel launch between compactions; 0 = 100,
                            the reference's interrupt-poll cadence (EM.cpp:261)             */
    ldsr_poll_fn poll;   /* may be NULL                                                      */
    void *poll_arg;
    int variant;         /* EM kernel: 0 = auto (time-split kernel when its shared-memory plan
                            fits -- the wide-input one for input widths >= 5 -- else the
                            lane-per-fit kernel); 1 = lane-per-fit kernel with checkpoints in global
                            memory; 2 = lane-per-fit kernel; 3 = time-split kernel, 4 = wide-input
                            time-split kernel, 5 = small-batch scan kernel (one CTA per fit; auto for
                            up to 1200 fits of width <= 4, 900 of width 5..10), or LDSR_ERR_UNSUPPORTED;
                            6 = auto without the scan kernel (what a sharded call gives its workers when
                            the whole batch is above that range).  DESIGN.md section 4. */
    int trace_liks;      /* ldsr_plan_em only: record the likelihood trace so that
                            ldsr_plan_fetch can return liks (ldsr_em_batch infers it from
                            out->liks)                                                       */
} ldsr_options;

/* ---- context: owns per-device streams and reusable device/pinned arenas ------------------ */
typedef struct ldsr_ctx ldsr_ctx;
int ldsr_ctx_create(int n_devices, const int *devices, ldsr_ctx **out, char *errbuf, int errlen);
void ldsr_ctx_destroy(ldsr_ctx *ctx);
/* The arenas are caches: blocks are kept for reuse between calls and handed back to the driver only
   when an allocation fails, on ldsr_ctx_destroy, or here.  Returns the device bytes released (blocks
   in use by a live plan are kept); cached_bytes, if not NULL, receives what the context still holds. */
long long ldsr_ctx_trim(ldsr_ctx *ctx, long long *cached_bytes);
int ldsr_device_count(void); /* 0 when there is no usable CUDA device */
int ldsr_abi_version(void);

/* ---- the hot path: batched LDS_EM + restart selection ---------------------------------- */
/* Host buffers in, host buffers out; shards groups across the ctx's devices (one worker
 * thread + stream per device, no collective).  ctx may be NULL (a temporary one is made). */
int ldsr_em_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int niter, double tol,
                  const ldsr_options *opt, ldsr_em_result *out, char *errbuf, int errlen);

/* Device-resident form: a plan holds the packed batch in HBM on ONE device. */
typedef struct ldsr_plan ldsr_plan;
int ldsr_plan_create(const ldsr_batch *batch, int device, ldsr_plan **out, char *errbuf, int errlen);
/* Runs EM for every fit from the plan's resident theta0 on `stream` (a cudaStream_t, NULL =
 * the plan's own stream); blocks until the results are resident in HBM.  Launch statistics
 * are returned through the optional long long[8] `stats`:
 * {kernel launches issued, EM chunks (= em_chunk_kernel launches), total E-steps executed (all
 *  fits), summed device time of the EM kernel launches in ns (CUDA events on `stream`),
 *  which EM kernel ran: 0 lane-per-fit, 1 time-split, 2 wide-input time-split, 3 small-batch scan;
 *  CTAs of the co-resident grid that shared the tasks by iterations (time-split kernel, batches of one to four
 *  waves; 0 = one CTA per task); 0, 0}. */
int ldsr_plan_em(ldsr_plan *plan, int niter, double tol, const ldsr_options *opt, void *stream,
                 long long *stats, char *errbuf, int errlen);
int ldsr_plan_set_theta0(ldsr_plan *plan, const double *theta0_host, char *errbuf, int errlen);
int ldsr_plan_fetch(ldsr_plan *plan, ldsr_em_result *out, char *errbuf, int errlen);
void ldsr_plan_destroy(ldsr_plan *plan);

/* ---- single-step entry points (the reference's other .Call functions, batched) ---------- */
/* Kalman_smoother for every fit's theta0 on its group's (held-out) y.  X,Y,V,J are
 * [sum over fits of T] with fit f's row at fit_ptr[f] (prefix sum of T[series(f)]);
 * stdlik as in EM.cpp:22,124. */
int ldsr_smoother_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int stdlik, double *X, double *Y,
                        double *V, double *J, double *lik, char *errbuf, int errlen);
/* Mstep: X,V,J rows (same layout as above) -> theta_out [n_fits*theta_stride], status. */
int ldsr_mstep_batch(ldsr_ctx *ctx, const ldsr_batch *batch, const double *X, const double *V,
                     const double *J, double *theta_out, int *status, char *errbuf, int errlen);
/* propagate (EM.cpp:295-356): open-loop X,Y,V rows and lik for every fit's theta0. */
int ldsr_propagate_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int stdlik, double *X, double *Y,
                         double *V, double *lik, char *errbuf, int errlen);

/* LDS_rep (R/stochastics.R:18-63): n_reps stochastic replicates of ONE model over n steps.
 * Noise: if z != NULL it holds n_reps*(1+2n) standard-normal draws in the reference's draw order
 * per replicate (x1, then n state draws, then n observation draws) -- this is the exact-parity
 * path; else draws come from a counter-based generator keyed by (seed, replicate, index).
 * Outputs are [n_reps*n] replicate-major (the reference's rbindlist order); any may be NULL. */
int ldsr_rep_batch(ldsr_ctx *ctx, const double *theta, const double *u, const double *v, int n,
                   int p, int q, int n_reps, const double *z, unsigned long long seed, double mu,
                   int exp_trans, double *simX, double *simY, double *simQ, char *errbuf,
                   int errlen);

/* The same, with the noise the reference itself would draw: equal to `set.seed(r_seed);
 * LDS_rep(theta, u, v, years, num.reps = n_reps, mu, exp.trans)` under R's default generators
 * (Mersenne-Twister + Inversion, one stream across the replicates, R/stochastics.R:23-26,60-61).
 * The n_reps*(1+2n) normals are generated on the device (r_rng.cuh) and never cross PCIe. */
int ldsr_rep_batch_r(ldsr_ctx *ctx, const double *theta, const double *u, const double *v, int n,
                     int p, int q, int n_reps, unsigned int r_seed, double mu, int exp_trans,
                     double *simX, double *simY, double *simQ, char *errbuf, int errlen);

/* Replicates conditioned on the observed record (beyond the reference): draws of whole trajectories from the
 * smoothing distribution p(x_0..T-1 | y, theta) by forward filtering, backward sampling.  Unlike LDS_rep's
 * open-loop replicates they pass through the observed flows, and their year-wise spread is the reconstruction's
 * band.  Every fit's theta0 row is one model, conditioned on its group's y with the group's held-out steps
 * removed; the filter is Kalman_smoother's (mu1, V1 the prior of x_0, u with one step of lag, v without,
 * u == NULL drops B u and v == NULL drops D v).  Per replicate, for t = T-1 down to 0:
 *     x_t = m_t + J_t x_{t+1} + s_t zeta_t     (J_t = Vu_t A / Vp_{t+1}, m_t = Xu_t - J_t Xp_{t+1},
 *                                               s_t = sqrt(Vu_t Q / Vp_{t+1}); at t = T-1: J = 0, m = Xu, s = sqrt(Vu))
 *     simX_t = x_t
 *     simY_t = y_t (bit for bit) at observed steps, else C x_t + D v_t + sqrt(R) eps_t
 *     simQ_t = back-transform(simY_t + mu): transform 0 none, 1 exp, 2 inverse Box-Cox (lambda; 0 means exp)
 * simY is on the centred, transformed scale.  With zeta = eps = 0, simX is the smoother's X and simY its Y at
 * unobserved steps.  Outputs follow the caller's fit order: with fit_ptr the exclusive prefix sum of T over the
 * fits (ldsr_smoother_batch's rows), fit f's replicate r starts at n_reps*fit_ptr[f] + r*T_f; any output may be
 * NULL.  z (optional) holds fit f's replicate r at 2*(n_reps*fit_ptr[f] + r*T_f): T_f state draws zeta_t, then
 * T_f observation draws eps_t (present but unused at observed steps).  Without z the draws come from a
 * counter-based generator keyed by (seed, fit index, replicate, step): a replicate's draws do not depend on
 * n_reps or on the other fits.  mu [n_fits] may be NULL (0); lambda [n_fits] is read with transform 2 only.
 * One device (ctx device 0); arguments are checked before a device is touched. */
int ldsr_posterior_rep_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int n_reps, const double *z,
                             unsigned long long seed, const double *mu, int transform, const double *lambda,
                             double *simX, double *simY, double *simQ, char *errbuf, int errlen);

/* Device time in ms (CUDA events around the kernels, summed) of the last ldsr_rep_batch / ldsr_rep_batch_r /
 * ldsr_posterior_rep_batch call made by the calling thread: the measurement hook of bench.py's config-4 record. */
double ldsr_last_device_ms(void);

/* ---- the reference's random numbers (R's default generators after set.seed) ---------------
 * The reference draws its restarts' initial values with runif (make_init, R/LDS_reconstruction.R:
 * 14-30) and its replicates with rnorm; a caller outside R reproduces a seeded reference run by
 * drawing from this generator instead.  ldsr_r_rng_* is a sequential host generator (initial values
 * are a few thousand draws; no device needed): create = set.seed(seed), unif = runif(n, a, b),
 * norm = rnorm(n), sample = sample.int(n, k); the state advances across calls exactly as R's does.  ldsr_r_rnorm_device is
 * `set.seed(seed); rnorm(n)` generated on the GPU into a host buffer (bulk draws). */
typedef struct ldsr_r_rng ldsr_r_rng;
int ldsr_r_rng_create(unsigned int seed, ldsr_r_rng **out, char *errbuf, int errlen);
int ldsr_r_rng_unif(ldsr_r_rng *rng, int n, double a, double b, double *out, char *errbuf, int errlen);
int ldsr_r_rng_norm(ldsr_r_rng *rng, int n, double *out, char *errbuf, int errlen);
/* sample.int(n, k) without replacement, 1-based (the folds of make_Z, R/utils.R:83-101; R >= 3.6
 * "Rejection" sampling) */
int ldsr_r_rng_sample(ldsr_r_rng *rng, int n, int k, int *out, char *errbuf, int errlen);
void ldsr_r_rng_destroy(ldsr_r_rng *rng);
int ldsr_r_rnorm_device(int device, unsigned int seed, long long n, double *out, char *errbuf, int errlen);

/* ---- multi-GPU sharding (pure host logic, no device needed) ------------------------------
 * The partition ldsr_em_batch uses: group g goes to shard group_shard[g] in 0..n_shards-1.
 * All fits of a group stay on one device, so restart selection is device-local and the host only
 * concatenates results -- there is no collective on the data path. */
int ldsr_shard_groups(const ldsr_batch *batch, int n_shards, int *group_shard, char *errbuf, int errlen);

/* ---- cross-validation skill metrics: the step right after the EM hot path in cvLDS -------------
 * Replaces `mapply(calculate_metrics, sim = Ycv, z = Z, MoreArgs = list(obs = target))`
 * (R/LDS_reconstruction.R:395) = calculate_metrics (R/utils.R:56-70) over NSE, RE, nRMSE, corr, KGE
 * of src/utils.cpp:13-97, for all folds in one launch (one warp per fold).
 *   sim [n_folds][n]: cross-validated output per fold; exp_trans != 0 applies exp() first
 *                     (transform = 'log', R/LDS_reconstruction.R:385-386)
 *   obs [n]: target, NaN allowed (dropped from the calibration part)
 *   z_ptr [n_folds+1], z_idx: CSR of each fold's hold-out indices, 1-BASED as in R
 *   out [n_folds][5]: R2, RE, CE, nRMSE, KGE (the column order of metrics.dist) */
int ldsr_cv_metrics_batch(int device, int n, int n_folds, const double *sim, const double *obs, const int *z_ptr,
                          const int *z_idx, int exp_trans, double *out, char *errbuf, int errlen);
/* The same for many stations in one launch (cvLDS over a set of gauges): station s has a target of n[s] >= 2
 * values and the folds fold_ptr[s] .. fold_ptr[s+1]-1 (fold_ptr[0] = 0, non-decreasing, fold_ptr[n_stations]
 * >= 1 folds in all).
 *   sim: the folds' rows concatenated in fold order, each n[station] long
 *   obs: the stations' targets concatenated in station order
 *   z_ptr [n_folds+1], z_idx: CSR of each fold's hold-out indices, 1-BASED into its OWN station's target
 *   out [n_folds][5] in fold order.
 * ldsr_cv_metrics_batch is the one-station case (same kernel, same bits). */
int ldsr_cv_metrics_stations(int device, int n_stations, const int *n, const int *fold_ptr, const double *sim,
                             const double *obs, const int *z_ptr, const int *z_idx, int exp_trans, double *out,
                             char *errbuf, int errlen);

/* ---- objectives of the experimental learners, for a whole population of parameter vectors ------
 * One value per fit (= per theta0 row of the batch, on its group's y with its hold-outs removed):
 *   kind 0  penalized_likelihood (R/LDS_GA.R:28-44): Kalman_smoother(stdlik = FALSE)$lik
 *           - lambda * sum_t (X_{t+1} - A X_t - B u_t)^2          -- the GA fitness of LDS_GA
 *   kind 1  negLogLik (R/LDS_GA.R:136-141): -propagate(theta,u,v,y)$lik   -- LDS_BFGS objective
 *   kind 2  ssqTrain  (R/LDS_GA.R:143-147): sum((y - propagate(...)$Y)^2, na.rm = TRUE)
 * The reference calls these once per candidate from GA::gaisl / optim; here a generation is one call. */
int ldsr_objective_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int kind, double lambda, double *values,
                         char *errbuf, int errlen);

/* ---- construct_rec: the step right after restart selection in LDS_reconstruction -------------
 * Replaces construct_rec (R/LDS_reconstruction.R:190-212; exp_ci and inv_boxcox of
 * R/utils.R:112-125) for all ensemble members at once, and the year-wise ensemble mean of X and Q
 * (R/LDS_reconstruction.R:247-248).
 *   X, V, Y [n][T]: smoothed state, its variance, smoothed output of every member (fit$X, fit$V, fit$Y)
 *   C, R [n]: each member's theta$C and theta$R;  mu: mean of the transformed observations
 *   transform 0 = none, 1 = log, 2 = boxcox with `lambda`
 *   out [n][6][T]: X, Xl, Xu, Q, Ql, Qu (the columns of `rec`);  mean [2][T] (may be NULL): mean X, mean Q
 * Deviation: boxcox with lambda == 0 uses exp_ci(Y + mu, sdY) like the log branch; the reference passes the
 * centred observations `y` there (R/LDS_reconstruction.R:205), which is not what its own log branch does. */
int ldsr_construct_rec_batch(int device, int n, int T, const double *X, const double *V, const double *Y,
                             const double *C, const double *R, double mu, int transform, double lambda, double *out,
                             double *mean, char *errbuf, int errlen);
/* The same for many stations in one launch (LDS_reconstruction over a set of gauges): station s has T[s] >= 1
 * years and the members member_ptr[s] .. member_ptr[s+1]-1 (member_ptr[0] = 0, at least one member each).
 *   X, V, Y: the members' rows concatenated in member order, each T[station] long
 *   C, R [n_members]: each member's theta$C and theta$R;  mu, lambda [n_stations]: per station (lambda is only
 *   read with transform 2 and may be NULL otherwise); transform is shared
 *   out: per member [6][T[station]], concatenated in member order
 *   mean (may be NULL): per station [2][T[s]] (mean X, mean Q over its members), concatenated in station order
 * ldsr_construct_rec_batch is the one-station case (same kernel, same bits). */
int ldsr_construct_rec_stations(int device, int n_stations, const int *T, const int *member_ptr, const double *X,
                                const double *V, const double *Y, const double *C, const double *R, const double *mu,
                                const double *lambda, int transform, double *out, double *mean, char *errbuf,
                                int errlen);

/* ---- general state dimension, long series (beyond the reference) ----------------------------
 * The reference is scalar-state only (src/EM.cpp:20 "matrix inversion is treated as /").
 * BASELINE.json's config 5 (d = 4, 20 proxies, T = 100 000) asks for the E-step of a d-dimensional
 * state, sequentially and as an associative scan over time.  Conventions are those of
 * Kalman_smoother (src/EM.cpp:22-131): (mu1,V1) is the predicted law of x_0, u enters with one step
 * of lag, v without, NaN in y = missing, innovations-form likelihood (divided by n_obs when stdlik).
 *   theta  [n_fits][theta_stride]: A d*d row-major | B d*p | C d | D q | Q d*d | R | mu1 d | V1 d*d
 *   u      [T][p] (an R p x T matrix, column-major) or NULL;  v [T][q] or NULL;  y [T]
 *   method 0 = sequential recursion (one thread per fit), 1 = associative scan (time cut into
 *            chunks of `chunk` steps, 0 = automatic)
 *   X [n_fits][T][d], V [n_fits][T][d][d], Y [n_fits][T] may be NULL (not copied back); lik [n_fits]
 *   kernel_ms (optional): device time of the kernels, CUDA events
 * One device; no CPU fallback (LDSR_ERR_CUDA without a device). */
int ldsr_smoother_d_batch(int device, int d, int T, int p, int q, const double *y, const double *u, const double *v,
                          int n_fits, const double *theta, int theta_stride, int stdlik, int method, int chunk,
                          double *X, double *V, double *Y, double *lik, double *kernel_ms, char *errbuf,
                          int errlen);

/* ---- measurement helper -------------------------------------------------------------------
 * FP64 roofline denominator: runs a register-resident DFMA kernel (8 independent chains per
 * thread, all SMs full) on `device` and returns the best-of-5 rate in TFLOP/s (FMA = 2 flops). */
int ldsr_measure_fp64_peak(int device, double *tflops, char *errbuf, int errlen);

#ifdef __cplusplus
}
#endif
#endif /* LDSR_B200_H */
