/*
 * ldsr_b200_shim.c -- R `.Call` glue between the ldsr package and libldsr_b200.so.
 *
 * NOT COMPILED IN THIS REPOSITORY'S BUILD: the build image has no R (no Rinternals.h).  It is
 * the file a maintainer drops into ldsr's src/ in place of src/EM.cpp + src/RcppExports.cpp
 * (see INTEGRATION.md).  Only the R C API is used: no Rcpp, no Armadillo.
 *
 * Entry points keep the reference's names and arities (src/RcppExports.cpp:133-136) so that
 * R/RcppExports.R keeps working unchanged:
 *     _ldsr_Kalman_smoother(y,u,v,theta,stdlik)   5
 *     _ldsr_Mstep(y,u,v,fit)                      4
 *     _ldsr_LDS_EM(y,u,v,theta0,niter,tol)        6
 *     _ldsr_propagate(theta,u,v,y,stdlik)         5
 * and add the batched ones used by the drop-in R wrappers in ldsr_b200.R:
 *     _ldsr_em_batch(series,group_series,held,fit_group,theta0,niter,tol,n_devices)   8
 *     _ldsr_rep_batch(theta,u,v,n,num_reps,seed,mu,exp_trans,z,r_seed)               10
 *     _ldsr_posterior_rep_batch(series,thetas,num_reps,z,seed,mu,transform,lambda)   8
 *     _ldsr_posterior_stats_batch(series,thetas,num_reps,z,seed,mu,transform,lambda,windows,threshold,range)   11
 *     _ldsr_posterior_yearly_batch(series,thetas,num_reps,z,seed,mu,transform,lambda,windows,lengths,threshold,range)   12
 *     _ldsr_posterior_quantile_batch(series,thetas,num_reps,z,seed,mu,transform,lambda,windows,levels,range)   11
 *     _ldsr_cv_metrics(Ycv,target,Z,exp_trans)                                        4
 *     _ldsr_construct_rec(X,V,Y,C,R,mu,transform,lambda)                              8
 *     _ldsr_cv_metrics_stations(Ycv,target,Z,exp_trans)   lists, one element per station    4
 *     _ldsr_construct_rec_stations(X,V,Y,C,R,mu,transform,lambda)   lists / per-station vectors   8
 *     _ldsr_objective(y,u,v,thetas,kind,lambda)   thetas: (2d+6) x n matrix, one column per candidate   6
 *     _ldsr_smoother_d(y,u,v,theta,stdlik,method)                                     6
 *     _ldsr_trim()                                release the session's cached device memory  0
 *       (state dimension d > 1: theta$A is d x d, B d x p, C 1 x d, D 1 x q, Q d x d, R, mu1 d, V1 d x d)
 *
 * The reference's `matrix(0)` sentinel (a 1x1 matrix, EM.cpp:50,71) is mapped to a NULL u/v
 * pointer here, so callers keep passing what they pass today.
 */
#include <R.h>
#include <Rinternals.h>
#include <R_ext/Rdynload.h>
#include <string.h>

#include "ldsr_b200.h"

/* One context per R session: its device and pinned arenas are reused by every call (a context per
 * call would pay cudaMalloc / cudaMallocHost each time).  Created on first use, released by
 * R_unload_ldsr or by ldsr_gpu_trim() from R. */
static ldsr_ctx *session_ctx = NULL;
static ldsr_ctx *ctx(void) {
    if (!session_ctx) {
        char err[256] = "";
        if (ldsr_ctx_create(0, NULL, &session_ctx, err, sizeof err) != LDSR_OK) Rf_error("ldsr_b200: %s", err);
    }
    return session_ctx;
}

static const char *TH_NAMES[] = {"A", "B", "C", "D", "Q", "R", "mu1", "V1", ""};

static SEXP list_get(SEXP list, const char *name) {
    SEXP names = Rf_getAttrib(list, R_NamesSymbol);
    for (R_xlen_t i = 0; i < XLENGTH(list); i++)
        if (strcmp(CHAR(STRING_ELT(names, i)), name) == 0) return VECTOR_ELT(list, i);
    Rf_error("ldsr: list element '%s' not found", name);
    return R_NilValue;
}
/* one-column matrix == the reference's "no input" sentinel */
static const double *input_ptr(SEXP m, int T, int *rows) {
    if (Rf_isNull(m) || Rf_ncols(m) == 1) {
        *rows = Rf_isNull(m) ? 1 : Rf_nrows(m);
        return NULL;
    }
    if (Rf_ncols(m) != T) Rf_error("ldsr: u/v must have %d columns", T);
    *rows = Rf_nrows(m);
    return REAL(m);
}
static void theta_to_flat(SEXP theta, int p, int q, double *out) {
    out[0] = REAL(list_get(theta, "A"))[0];
    memcpy(out + 1, REAL(list_get(theta, "B")), sizeof(double) * p);
    out[1 + p] = REAL(list_get(theta, "C"))[0];
    memcpy(out + 2 + p, REAL(list_get(theta, "D")), sizeof(double) * q);
    out[2 + p + q] = REAL(list_get(theta, "Q"))[0];
    out[3 + p + q] = REAL(list_get(theta, "R"))[0];
    out[4 + p + q] = REAL(list_get(theta, "mu1"))[0];
    out[5 + p + q] = REAL(list_get(theta, "V1"))[0];
}
static SEXP mat1(const double *x, int ncol) { /* 1 x ncol matrix */
    SEXP m = PROTECT(Rf_allocMatrix(REALSXP, 1, ncol));
    memcpy(REAL(m), x, sizeof(double) * ncol);
    UNPROTECT(1);
    return m;
}
static SEXP flat_to_theta(const double *th, int p, int q) {
    SEXP out = PROTECT(Rf_mkNamed(VECSXP, TH_NAMES));
    SET_VECTOR_ELT(out, 0, mat1(th, 1));
    SET_VECTOR_ELT(out, 1, mat1(th + 1, p));
    SET_VECTOR_ELT(out, 2, mat1(th + 1 + p, 1));
    SET_VECTOR_ELT(out, 3, mat1(th + 2 + p, q));
    for (int k = 0; k < 4; k++) SET_VECTOR_ELT(out, 4 + k, mat1(th + 2 + p + q + k, 1));
    UNPROTECT(1);
    return out;
}

/* interrupt poll on R's main thread: R_CheckUserInterrupt longjmps, so run it under
 * R_ToplevelExec and translate to a flag (the library then returns LDSR_ERR_INTERRUPTED). */
static void chk_intr(void *dummy) { (void)dummy; R_CheckUserInterrupt(); }
static int poll_interrupt(void *arg) { (void)arg; return R_ToplevelExec(chk_intr, NULL) == FALSE; }

/* batch of exactly one series / group / fit */
typedef struct {
    ldsr_batch b;
    int T, p, q, zero;
    const double *y, *u, *v;
    double *theta0;
} one_fit;
static void one_fit_init(one_fit *f, SEXP y, SEXP u, SEXP v, SEXP theta) {
    memset(f, 0, sizeof *f);
    f->T = Rf_ncols(y);
    f->y = REAL(y);
    f->u = input_ptr(u, f->T, &f->p);
    f->v = input_ptr(v, f->T, &f->q);
    f->theta0 = (double *)R_alloc(f->p + f->q + 6, sizeof(double));
    if (!Rf_isNull(theta)) theta_to_flat(theta, f->p, f->q, f->theta0);
    f->b.n_series = f->b.n_groups = f->b.n_fits = 1;
    f->b.T = &f->T; f->b.p = &f->p; f->b.q = &f->q;
    f->b.y = &f->y; f->b.u = &f->u; f->b.v = &f->v;
    f->b.group_series = &f->zero; f->b.fit_group = &f->zero;
    f->b.theta0 = f->theta0; f->b.theta_stride = f->p + f->q + 6;
}
static void check(int rc, const char *err) {
    if (rc == LDSR_ERR_INTERRUPTED) Rf_onintr();
    if (rc != LDSR_OK) Rf_error("ldsr_b200: %s", err);
}
static SEXP fit_list(const double *X, const double *Y, const double *V, const double *J, double lik, int T) {
    const char *nm[] = {"X", "Y", "V", "J", "lik", ""};
    SEXP out = PROTECT(Rf_mkNamed(VECSXP, nm));
    SET_VECTOR_ELT(out, 0, mat1(X, T));
    SET_VECTOR_ELT(out, 1, mat1(Y, T));
    SET_VECTOR_ELT(out, 2, mat1(V, T));
    SET_VECTOR_ELT(out, 3, mat1(J, T));
    SET_VECTOR_ELT(out, 4, Rf_ScalarReal(lik));
    UNPROTECT(1);
    return out;
}

/* replaces src/RcppExports.cpp:11-23 */
SEXP _ldsr_Kalman_smoother(SEXP y, SEXP u, SEXP v, SEXP theta, SEXP stdlik) {
    one_fit f; char err[512] = "";
    one_fit_init(&f, y, u, v, theta);
    double *buf = (double *)R_alloc(4 * (size_t)f.T, sizeof(double)), lik;
    check(ldsr_smoother_batch(ctx(), &f.b, Rf_asLogical(stdlik), buf, buf + f.T, buf + 2 * f.T, buf + 3 * f.T, &lik,
                              err, sizeof err), err);
    return fit_list(buf, buf + f.T, buf + 2 * f.T, buf + 3 * f.T, lik, f.T);
}

/* replaces src/RcppExports.cpp:26-37 */
SEXP _ldsr_Mstep(SEXP y, SEXP u, SEXP v, SEXP fit) {
    one_fit f; char err[512] = "";
    one_fit_init(&f, y, u, v, R_NilValue);
    int status = 0;
    double *th = (double *)R_alloc(f.p + f.q + 6, sizeof(double));
    check(ldsr_mstep_batch(ctx(), &f.b, REAL(list_get(fit, "X")), REAL(list_get(fit, "V")), REAL(list_get(fit, "J")),
                           th, &status, err, sizeof err), err);
    if (status == LDSR_FIT_SINGULAR) Rf_error("inv(): matrix is singular");
    SEXP out = PROTECT(flat_to_theta(th, f.p, f.q));
    UNPROTECT(1);
    return out;
}

/* replaces src/RcppExports.cpp:40-53 */
SEXP _ldsr_LDS_EM(SEXP y, SEXP u, SEXP v, SEXP theta0, SEXP niterS, SEXP tolS) {
    one_fit f; char err[512] = "";
    one_fit_init(&f, y, u, v, theta0);
    const int niter = Rf_asInteger(niterS), nth = f.p + f.q + 6;
    double *buf = (double *)R_alloc(4 * (size_t)f.T + nth + niter, sizeof(double));
    double *th = buf + 4 * f.T, *liks = th + nth, lik;
    int iters = 0, status = 0, best = 0;
    ldsr_em_result r; memset(&r, 0, sizeof r);
    r.theta = th; r.lik = &lik; r.iters = &iters; r.status = &status; r.liks = liks; r.best = &best;
    r.X = buf; r.Y = buf + f.T; r.V = buf + 2 * f.T; r.J = buf + 3 * f.T;
    ldsr_options opt; memset(&opt, 0, sizeof opt);
    opt.n_devices = 1; opt.poll = poll_interrupt;
    check(ldsr_em_batch(ctx(), &f.b, niter, Rf_asReal(tolS), &opt, &r, err, sizeof err), err);
    if (status == LDSR_FIT_SINGULAR) Rf_error("inv(): matrix is singular");
    const char *nm[] = {"theta", "fit", "liks", "lik", ""};
    SEXP out = PROTECT(Rf_mkNamed(VECSXP, nm));
    SET_VECTOR_ELT(out, 0, flat_to_theta(th, f.p, f.q));
    SET_VECTOR_ELT(out, 1, fit_list(r.X, r.Y, r.V, r.J, lik, f.T));
    SEXP lk = PROTECT(Rf_allocVector(REALSXP, iters));
    memcpy(REAL(lk), liks, sizeof(double) * iters);
    SET_VECTOR_ELT(out, 2, lk);
    SET_VECTOR_ELT(out, 3, Rf_ScalarReal(lik));
    UNPROTECT(2);
    return out;
}

/* replaces src/RcppExports.cpp:56-68 */
SEXP _ldsr_propagate(SEXP theta, SEXP u, SEXP v, SEXP y, SEXP stdlik) {
    one_fit f; char err[512] = "";
    one_fit_init(&f, y, u, v, theta);
    double *buf = (double *)R_alloc(3 * (size_t)f.T, sizeof(double)), lik;
    check(ldsr_propagate_batch(ctx(), &f.b, Rf_asLogical(stdlik), buf, buf + f.T, buf + 2 * f.T, &lik, err, sizeof err),
          err);
    const char *nm[] = {"X", "Y", "V", "lik", ""};
    SEXP out = PROTECT(Rf_mkNamed(VECSXP, nm));
    SET_VECTOR_ELT(out, 0, mat1(buf, f.T));
    SET_VECTOR_ELT(out, 1, mat1(buf + f.T, f.T));
    SET_VECTOR_ELT(out, 2, mat1(buf + 2 * f.T, f.T));
    SET_VECTOR_ELT(out, 3, Rf_ScalarReal(lik));
    UNPROTECT(1);
    return out;
}

/* The batched fan-out that replaces foreach %dopar% LDS_EM (R/LDS_reconstruction.R:46,242,373).
 *   series       list of list(y = 1xT matrix, u = matrix, v = matrix)
 *   group_series integer, 1-based series index of each group
 *   held         list of integer vectors: 1-based time steps set to NA for the group
 *   fit_group    integer, 1-based, non-decreasing
 *   theta0       numeric matrix  stride x n_fits (one flat theta per COLUMN, R/LDS_GA.R:6-16 order)
 * Returns list(theta [stride x n_fits], lik, iters, status, best (1-based, NA if none), X,Y,V,J =
 * lists of per-group vectors). */
SEXP _ldsr_em_batch(SEXP series, SEXP group_series, SEXP held, SEXP fit_group, SEXP theta0, SEXP niterS, SEXP tolS,
                    SEXP ndevS) {
    const int ns = (int)XLENGTH(series), ng = (int)XLENGTH(group_series), nf = (int)XLENGTH(fit_group);
    int *T = (int *)R_alloc(ns, sizeof(int)), *p = (int *)R_alloc(ns, sizeof(int)), *q = (int *)R_alloc(ns, sizeof(int));
    const double **y = (const double **)R_alloc(ns, sizeof(double *));
    const double **u = (const double **)R_alloc(ns, sizeof(double *));
    const double **v = (const double **)R_alloc(ns, sizeof(double *));
    for (int s = 0; s < ns; s++) {
        SEXP e = VECTOR_ELT(series, s);
        T[s] = Rf_ncols(list_get(e, "y"));
        y[s] = REAL(list_get(e, "y"));
        u[s] = input_ptr(list_get(e, "u"), T[s], &p[s]);
        v[s] = input_ptr(list_get(e, "v"), T[s], &q[s]);
    }
    int *gs = (int *)R_alloc(ng, sizeof(int)), *hp = (int *)R_alloc(ng + 1, sizeof(int));
    size_t nheld = 0, tot = 0;
    for (int g = 0; g < ng; g++) nheld += XLENGTH(VECTOR_ELT(held, g));
    int *hi = (int *)R_alloc(nheld + 1, sizeof(int));
    long long *tp = (long long *)R_alloc(ng + 1, sizeof(long long));
    hp[0] = 0; tp[0] = 0;
    for (int g = 0; g < ng; g++) {
        gs[g] = INTEGER(group_series)[g] - 1;
        SEXP h = VECTOR_ELT(held, g);
        for (R_xlen_t k = 0; k < XLENGTH(h); k++) hi[hp[g] + k] = INTEGER(h)[k] - 1;
        hp[g + 1] = hp[g] + (int)XLENGTH(h);
        tp[g + 1] = tp[g] + T[gs[g]];
    }
    tot = (size_t)tp[ng];
    int *fg = (int *)R_alloc(nf, sizeof(int));
    for (int f = 0; f < nf; f++) fg[f] = INTEGER(fit_group)[f] - 1;
    ldsr_batch b; memset(&b, 0, sizeof b);
    b.n_series = ns; b.T = T; b.p = p; b.q = q; b.y = y; b.u = u; b.v = v;
    b.n_groups = ng; b.group_series = gs; b.held_ptr = hp; b.held_idx = hi;
    b.n_fits = nf; b.fit_group = fg; b.theta0 = REAL(theta0); b.theta_stride = Rf_nrows(theta0);

    const char *nm[] = {"theta", "lik", "iters", "status", "best", "X", "Y", "V", "J", ""};
    SEXP out = PROTECT(Rf_mkNamed(VECSXP, nm));
    SEXP th = PROTECT(Rf_allocMatrix(REALSXP, b.theta_stride, nf));
    SEXP lik = PROTECT(Rf_allocVector(REALSXP, nf)), it = PROTECT(Rf_allocVector(INTSXP, nf));
    SEXP st = PROTECT(Rf_allocVector(INTSXP, nf)), best = PROTECT(Rf_allocVector(INTSXP, ng));
    double *traj = (double *)R_alloc(4 * tot, sizeof(double));
    ldsr_em_result r; memset(&r, 0, sizeof r);
    r.theta = REAL(th); r.lik = REAL(lik); r.iters = INTEGER(it); r.status = INTEGER(st); r.best = INTEGER(best);
    r.X = traj; r.Y = traj + tot; r.V = traj + 2 * tot; r.J = traj + 3 * tot;
    ldsr_options opt; memset(&opt, 0, sizeof opt);
    opt.n_devices = Rf_asInteger(ndevS); opt.poll = poll_interrupt;
    char err[512] = "";
    check(ldsr_em_batch(ctx(), &b, Rf_asInteger(niterS), Rf_asReal(tolS), &opt, &r, err, sizeof err), err);
    for (int g = 0; g < ng; g++) INTEGER(best)[g] = INTEGER(best)[g] < 0 ? NA_INTEGER : INTEGER(best)[g] + 1;
    SET_VECTOR_ELT(out, 0, th); SET_VECTOR_ELT(out, 1, lik); SET_VECTOR_ELT(out, 2, it);
    SET_VECTOR_ELT(out, 3, st); SET_VECTOR_ELT(out, 4, best);
    for (int a = 0; a < 4; a++) {
        SEXP lst = PROTECT(Rf_allocVector(VECSXP, ng));
        for (int g = 0; g < ng; g++) SET_VECTOR_ELT(lst, g, mat1(traj + a * tot + tp[g], T[gs[g]]));
        SET_VECTOR_ELT(out, 5 + a, lst);
        UNPROTECT(1);
    }
    UNPROTECT(6);
    return out;
}

/* LDS_rep (R/stochastics.R:58-63) on the device generator.  Returns a 3-column matrix
 * (simX, simY, simQ), rows replicate-major like rbindlist(lapply(...)). */
SEXP _ldsr_rep_batch(SEXP theta, SEXP u, SEXP v, SEXP nS, SEXP repsS, SEXP seedS, SEXP muS, SEXP expS, SEXP zS,
                     SEXP rseedS) {
    const int n = Rf_asInteger(nS), reps = Rf_asInteger(repsS);
    int p = 0, q = 0;
    const double *up = Rf_isNull(u) ? NULL : input_ptr(u, n, &p), *vp = Rf_isNull(u) || Rf_isNull(v) ? NULL : input_ptr(v, n, &q);
    if (!up) p = 0;
    if (!vp) q = 0;
    double *th = (double *)R_alloc(p + q + 6, sizeof(double));
    th[0] = REAL(list_get(theta, "A"))[0];
    memcpy(th + 1, REAL(list_get(theta, "B")), sizeof(double) * p);
    th[1 + p] = REAL(list_get(theta, "C"))[0];
    memcpy(th + 2 + p, REAL(list_get(theta, "D")), sizeof(double) * q);
    th[2 + p + q] = REAL(list_get(theta, "Q"))[0]; th[3 + p + q] = REAL(list_get(theta, "R"))[0];
    th[4 + p + q] = REAL(list_get(theta, "mu1"))[0]; th[5 + p + q] = REAL(list_get(theta, "V1"))[0];
    SEXP out = PROTECT(Rf_allocMatrix(REALSXP, n * reps, 3));
    double *o = REAL(out);
    char err[512] = "";
    /* z: num_reps*(1+2n) standard normals drawn by R in one_LDS_rep's order (R/stochastics.R:23-26), or NULL */
    const double *z = Rf_isNull(zS) ? NULL : REAL(zS);
    if (z && XLENGTH(zS) != (R_xlen_t)reps * (1 + 2 * (R_xlen_t)n)) Rf_error("ldsr: z must hold num.reps*(1+2n) draws");
    if (!z && !Rf_isNull(rseedS)) /* the stream of set.seed(r_seed), generated on the device (r_rng.cuh) */
        check(ldsr_rep_batch_r(ctx(), th, up, vp, n, p, q, reps, (unsigned int)Rf_asInteger(rseedS), Rf_asReal(muS),
                               Rf_asLogical(expS), o, o + (size_t)n * reps, o + 2 * (size_t)n * reps, err, sizeof err),
              err);
    else
    check(ldsr_rep_batch(ctx(), th, up, vp, n, p, q, reps, z, (unsigned long long)Rf_asReal(seedS), Rf_asReal(muS),
                         Rf_asLogical(expS), o, o + (size_t)n * reps, o + 2 * (size_t)n * reps, err, sizeof err), err);
    UNPROTECT(1);
    return out;
}

/* Replicates conditioned on the observed record (LDS_rep_posterior in ldsr_b200.R): series is a list of
 * list(y, u, v), one per ensemble member, each its own group and fit; thetas a stride x n matrix (one column per
 * member, the flat order of R/LDS_GA.R:6-16); mu and lambda per member (lambda NULL unless transform = 2).
 * Returns a 3-column matrix (simX, simY, simQ): member by member, replicate by replicate, T rows each. */
SEXP _ldsr_posterior_rep_batch(SEXP series, SEXP thetas, SEXP repsS, SEXP zS, SEXP seedS, SEXP muS, SEXP transformS,
                               SEXP lambdaS) {
    const int ns = (int)XLENGTH(series), reps = Rf_asInteger(repsS);
    int *T = (int *)R_alloc(ns, sizeof(int)), *p = (int *)R_alloc(ns, sizeof(int)), *q = (int *)R_alloc(ns, sizeof(int));
    int *idx = (int *)R_alloc(ns, sizeof(int));
    const double **y = (const double **)R_alloc(ns, sizeof(double *));
    const double **u = (const double **)R_alloc(ns, sizeof(double *));
    const double **v = (const double **)R_alloc(ns, sizeof(double *));
    R_xlen_t tot = 0;
    for (int s = 0; s < ns; s++) {
        SEXP e = VECTOR_ELT(series, s);
        T[s] = Rf_ncols(list_get(e, "y"));
        y[s] = REAL(list_get(e, "y"));
        u[s] = input_ptr(list_get(e, "u"), T[s], &p[s]);
        v[s] = input_ptr(list_get(e, "v"), T[s], &q[s]);
        idx[s] = s;
        tot += (R_xlen_t)reps * T[s];
    }
    if (Rf_ncols(thetas) != ns) Rf_error("ldsr: thetas must have one column per series");
    if (XLENGTH(muS) != ns) Rf_error("ldsr: mu must have one value per series");
    const double *z = Rf_isNull(zS) ? NULL : REAL(zS);
    if (z && XLENGTH(zS) != 2 * tot) Rf_error("ldsr: z must hold 2 * num.reps * sum(T) draws");
    const double *lam = Rf_isNull(lambdaS) ? NULL : REAL(lambdaS);
    if (lam && XLENGTH(lambdaS) != ns) Rf_error("ldsr: lambda must have one value per series");
    ldsr_batch b; memset(&b, 0, sizeof b);
    b.n_series = ns; b.T = T; b.p = p; b.q = q; b.y = y; b.u = u; b.v = v;
    b.n_groups = ns; b.group_series = idx;
    b.n_fits = ns; b.fit_group = idx; b.theta0 = REAL(thetas); b.theta_stride = Rf_nrows(thetas);
    SEXP out = PROTECT(Rf_allocMatrix(REALSXP, tot, 3));
    double *o = REAL(out);
    char err[512] = "";
    check(ldsr_posterior_rep_batch(ctx(), &b, reps, z, (unsigned long long)Rf_asReal(seedS), REAL(muS),
                                   Rf_asInteger(transformS), lam, o, o + tot, o + 2 * tot, err, sizeof err),
          err);
    UNPROTECT(1);
    return out;
}

/* Drought statistics of the same replicates, reduced on the device (LDS_rep_posterior_stats in ldsr_b200.R):
 * arguments as _ldsr_posterior_rep_batch, then windows (integer, up to 4 lengths of 1..64), threshold (one per
 * series, Q scale, or NULL) and range (a 2 x n integer matrix of 0-based [lo, hi) per series, or NULL).  Returns
 * list(wmin, wmin_at, wmax, wmax_at) as (num_reps * n) x n_windows matrices and, with a threshold, run_len, run_at,
 * deficit, deficit_at, n_runs as vectors of num_reps * n: member by member, replicate by replicate; steps 0-based,
 * -1 where undefined. */
SEXP _ldsr_posterior_stats_batch(SEXP series, SEXP thetas, SEXP repsS, SEXP zS, SEXP seedS, SEXP muS,
                                 SEXP transformS, SEXP lambdaS, SEXP windowsS, SEXP thresholdS, SEXP rangeS) {
    const int ns = (int)XLENGTH(series), reps = Rf_asInteger(repsS), nw = (int)XLENGTH(windowsS);
    int *T = (int *)R_alloc(ns, sizeof(int)), *p = (int *)R_alloc(ns, sizeof(int)), *q = (int *)R_alloc(ns, sizeof(int));
    int *idx = (int *)R_alloc(ns, sizeof(int));
    const double **y = (const double **)R_alloc(ns, sizeof(double *));
    const double **u = (const double **)R_alloc(ns, sizeof(double *));
    const double **v = (const double **)R_alloc(ns, sizeof(double *));
    R_xlen_t tot = 0;
    for (int s = 0; s < ns; s++) {
        SEXP e = VECTOR_ELT(series, s);
        T[s] = Rf_ncols(list_get(e, "y"));
        y[s] = REAL(list_get(e, "y"));
        u[s] = input_ptr(list_get(e, "u"), T[s], &p[s]);
        v[s] = input_ptr(list_get(e, "v"), T[s], &q[s]);
        idx[s] = s;
        tot += (R_xlen_t)reps * T[s];
    }
    if (Rf_ncols(thetas) != ns) Rf_error("ldsr: thetas must have one column per series");
    if (XLENGTH(muS) != ns) Rf_error("ldsr: mu must have one value per series");
    const double *z = Rf_isNull(zS) ? NULL : REAL(zS);
    if (z && XLENGTH(zS) != 2 * tot) Rf_error("ldsr: z must hold 2 * num.reps * sum(T) draws");
    const double *lam = Rf_isNull(lambdaS) ? NULL : REAL(lambdaS);
    if (lam && XLENGTH(lambdaS) != ns) Rf_error("ldsr: lambda must have one value per series");
    const double *thr = Rf_isNull(thresholdS) ? NULL : REAL(thresholdS);
    if (thr && XLENGTH(thresholdS) != ns) Rf_error("ldsr: threshold must have one value per series");
    const int *range = Rf_isNull(rangeS) ? NULL : INTEGER(rangeS);
    if (range && XLENGTH(rangeS) != 2 * (R_xlen_t)ns) Rf_error("ldsr: range must hold 2 values per series");
    ldsr_batch b; memset(&b, 0, sizeof b);
    b.n_series = ns; b.T = T; b.p = p; b.q = q; b.y = y; b.u = u; b.v = v;
    b.n_groups = ns; b.group_series = idx;
    b.n_fits = ns; b.fit_group = idx; b.theta0 = REAL(thetas); b.theta_stride = Rf_nrows(thetas);
    const R_xlen_t rows = (R_xlen_t)reps * ns;
    ldsr_stats_spec spec = {nw, INTEGER(windowsS), thr, range};
    ldsr_stats_out so; memset(&so, 0, sizeof so);
    const int n_out = thr ? 9 : 4;
    SEXP out = PROTECT(Rf_allocVector(VECSXP, n_out));
    for (int k = 0; k < n_out; k++) {
        const int is_real = k == 0 || k == 2 || k == 6;
        SEXP a = k < 4 ? Rf_allocMatrix(is_real ? REALSXP : INTSXP, rows, nw)
                       : Rf_allocVector(is_real ? REALSXP : INTSXP, rows);
        SET_VECTOR_ELT(out, k, a);
    }
    so.wmin = REAL(VECTOR_ELT(out, 0)); so.wmin_at = INTEGER(VECTOR_ELT(out, 1));
    so.wmax = REAL(VECTOR_ELT(out, 2)); so.wmax_at = INTEGER(VECTOR_ELT(out, 3));
    if (thr) {
        so.run_len = INTEGER(VECTOR_ELT(out, 4)); so.run_at = INTEGER(VECTOR_ELT(out, 5));
        so.deficit = REAL(VECTOR_ELT(out, 6)); so.deficit_at = INTEGER(VECTOR_ELT(out, 7));
        so.n_runs = INTEGER(VECTOR_ELT(out, 8));
    }
    char err[512] = "";
    check(ldsr_posterior_stats_batch(ctx(), &b, reps, z, (unsigned long long)Rf_asReal(seedS), REAL(muS),
                                     Rf_asInteger(transformS), lam, &spec, &so, err, sizeof err),
          err);
    UNPROTECT(1);
    return out;
}

/* Year-by-year drought counts of the same replicates, reduced across replicates on the device
 * (LDS_rep_posterior_yearly in ldsr_b200.R): arguments as _ldsr_posterior_rep_batch, then windows and lengths
 * (integer, up to 4 of 1..64 each), threshold (one per series, Q scale, required) and range (a 2 x n integer matrix
 * of 0-based [lo, hi) per series, or NULL).  Returns list(below, in_run, wbelow, nonfinite): below and nonfinite
 * as integer vectors of sum(T) (series by series, step by step), in_run and wbelow as sum(T) x n_lengths /
 * n_windows matrices; counts of replicates, -1 where undefined. */
SEXP _ldsr_posterior_yearly_batch(SEXP series, SEXP thetas, SEXP repsS, SEXP zS, SEXP seedS, SEXP muS,
                                  SEXP transformS, SEXP lambdaS, SEXP windowsS, SEXP lengthsS, SEXP thresholdS,
                                  SEXP rangeS) {
    const int ns = (int)XLENGTH(series), reps = Rf_asInteger(repsS);
    const int nw = (int)XLENGTH(windowsS), nl = (int)XLENGTH(lengthsS);
    int *T = (int *)R_alloc(ns, sizeof(int)), *p = (int *)R_alloc(ns, sizeof(int)), *q = (int *)R_alloc(ns, sizeof(int));
    int *idx = (int *)R_alloc(ns, sizeof(int));
    const double **y = (const double **)R_alloc(ns, sizeof(double *));
    const double **u = (const double **)R_alloc(ns, sizeof(double *));
    const double **v = (const double **)R_alloc(ns, sizeof(double *));
    R_xlen_t tot = 0, steps = 0;
    for (int s = 0; s < ns; s++) {
        SEXP e = VECTOR_ELT(series, s);
        T[s] = Rf_ncols(list_get(e, "y"));
        y[s] = REAL(list_get(e, "y"));
        u[s] = input_ptr(list_get(e, "u"), T[s], &p[s]);
        v[s] = input_ptr(list_get(e, "v"), T[s], &q[s]);
        idx[s] = s;
        tot += (R_xlen_t)reps * T[s];
        steps += T[s];
    }
    if (Rf_ncols(thetas) != ns) Rf_error("ldsr: thetas must have one column per series");
    if (XLENGTH(muS) != ns) Rf_error("ldsr: mu must have one value per series");
    const double *z = Rf_isNull(zS) ? NULL : REAL(zS);
    if (z && XLENGTH(zS) != 2 * tot) Rf_error("ldsr: z must hold 2 * num.reps * sum(T) draws");
    const double *lam = Rf_isNull(lambdaS) ? NULL : REAL(lambdaS);
    if (lam && XLENGTH(lambdaS) != ns) Rf_error("ldsr: lambda must have one value per series");
    if (Rf_isNull(thresholdS) || XLENGTH(thresholdS) != ns) Rf_error("ldsr: threshold must have one value per series");
    const int *range = Rf_isNull(rangeS) ? NULL : INTEGER(rangeS);
    if (range && XLENGTH(rangeS) != 2 * (R_xlen_t)ns) Rf_error("ldsr: range must hold 2 values per series");
    ldsr_batch b; memset(&b, 0, sizeof b);
    b.n_series = ns; b.T = T; b.p = p; b.q = q; b.y = y; b.u = u; b.v = v;
    b.n_groups = ns; b.group_series = idx;
    b.n_fits = ns; b.fit_group = idx; b.theta0 = REAL(thetas); b.theta_stride = Rf_nrows(thetas);
    ldsr_yearly_spec spec = {nw, INTEGER(windowsS), nl, INTEGER(lengthsS), REAL(thresholdS), range};
    SEXP out = PROTECT(Rf_allocVector(VECSXP, 4));
    SET_VECTOR_ELT(out, 0, Rf_allocVector(INTSXP, steps));
    SET_VECTOR_ELT(out, 1, Rf_allocMatrix(INTSXP, steps, nl));
    SET_VECTOR_ELT(out, 2, Rf_allocMatrix(INTSXP, steps, nw));
    SET_VECTOR_ELT(out, 3, Rf_allocVector(INTSXP, steps));
    ldsr_yearly_out yo = {INTEGER(VECTOR_ELT(out, 0)), INTEGER(VECTOR_ELT(out, 1)), INTEGER(VECTOR_ELT(out, 2)),
                          INTEGER(VECTOR_ELT(out, 3))};
    char err[512] = "";
    check(ldsr_posterior_yearly_batch(ctx(), &b, reps, z, (unsigned long long)Rf_asReal(seedS), REAL(muS),
                                      Rf_asInteger(transformS), lam, &spec, &yo, err, sizeof err),
          err);
    UNPROTECT(1);
    return out;
}

/* Per-year quantiles of w-year mean flows over the same replicates, selected on the device
 * (LDS_rep_posterior_quantiles in ldsr_b200.R): arguments as _ldsr_posterior_rep_batch, then windows (integer, 1 to
 * 4 of 1..64), levels (double, 1 to 8 in [0, 1], strictly increasing) and range (a 2 x n integer matrix of 0-based
 * [lo, hi) per series, or NULL).  Returns list(q, nonfinite, passes): q as a sum(T) x (n_levels n_windows) matrix
 * (series by series, step by step; window k's level l in column k n_levels + l; NaN where undefined), nonfinite as a sum(T) x n_windows integer matrix (-1 where
 * undefined), passes the sampler runs. */
SEXP _ldsr_posterior_quantile_batch(SEXP series, SEXP thetas, SEXP repsS, SEXP zS, SEXP seedS, SEXP muS,
                                    SEXP transformS, SEXP lambdaS, SEXP windowsS, SEXP levelsS, SEXP rangeS) {
    const int ns = (int)XLENGTH(series), reps = Rf_asInteger(repsS);
    const int nw = (int)XLENGTH(windowsS), nl = (int)XLENGTH(levelsS);
    int *T = (int *)R_alloc(ns, sizeof(int)), *p = (int *)R_alloc(ns, sizeof(int)), *q = (int *)R_alloc(ns, sizeof(int));
    int *idx = (int *)R_alloc(ns, sizeof(int));
    const double **y = (const double **)R_alloc(ns, sizeof(double *));
    const double **u = (const double **)R_alloc(ns, sizeof(double *));
    const double **v = (const double **)R_alloc(ns, sizeof(double *));
    R_xlen_t tot = 0, steps = 0;
    for (int s = 0; s < ns; s++) {
        SEXP e = VECTOR_ELT(series, s);
        T[s] = Rf_ncols(list_get(e, "y"));
        y[s] = REAL(list_get(e, "y"));
        u[s] = input_ptr(list_get(e, "u"), T[s], &p[s]);
        v[s] = input_ptr(list_get(e, "v"), T[s], &q[s]);
        idx[s] = s;
        tot += (R_xlen_t)reps * T[s];
        steps += T[s];
    }
    if (Rf_ncols(thetas) != ns) Rf_error("ldsr: thetas must have one column per series");
    if (XLENGTH(muS) != ns) Rf_error("ldsr: mu must have one value per series");
    const double *z = Rf_isNull(zS) ? NULL : REAL(zS);
    if (z && XLENGTH(zS) != 2 * tot) Rf_error("ldsr: z must hold 2 * num.reps * sum(T) draws");
    const double *lam = Rf_isNull(lambdaS) ? NULL : REAL(lambdaS);
    if (lam && XLENGTH(lambdaS) != ns) Rf_error("ldsr: lambda must have one value per series");
    const int *range = Rf_isNull(rangeS) ? NULL : INTEGER(rangeS);
    if (range && XLENGTH(rangeS) != 2 * (R_xlen_t)ns) Rf_error("ldsr: range must hold 2 values per series");
    ldsr_batch b; memset(&b, 0, sizeof b);
    b.n_series = ns; b.T = T; b.p = p; b.q = q; b.y = y; b.u = u; b.v = v;
    b.n_groups = ns; b.group_series = idx;
    b.n_fits = ns; b.fit_group = idx; b.theta0 = REAL(thetas); b.theta_stride = Rf_nrows(thetas);
    ldsr_quant_spec spec = {nw, INTEGER(windowsS), nl, REAL(levelsS), range};
    SEXP out = PROTECT(Rf_allocVector(VECSXP, 3));
    SET_VECTOR_ELT(out, 0, Rf_allocMatrix(REALSXP, steps, nl * nw));
    SET_VECTOR_ELT(out, 1, Rf_allocMatrix(INTSXP, steps, nw));
    SET_VECTOR_ELT(out, 2, Rf_allocVector(INTSXP, 1));
    ldsr_quant_out qo = {REAL(VECTOR_ELT(out, 0)), INTEGER(VECTOR_ELT(out, 1)), INTEGER(VECTOR_ELT(out, 2))};
    char err[512] = "";
    check(ldsr_posterior_quantile_batch(ctx(), &b, reps, z, (unsigned long long)Rf_asReal(seedS), REAL(muS),
                                        Rf_asInteger(transformS), lam, &spec, &qo, err, sizeof err),
          err);
    UNPROTECT(1);
    return out;
}

/* same shape as src/RcppExports.cpp:132-148 */
/* mapply(calculate_metrics, sim = Ycv, z = Z, MoreArgs = list(obs = target)) in one call
 * (R/LDS_reconstruction.R:395): Ycv is an n x n_folds matrix, Z a list of integer vectors. */
SEXP _ldsr_cv_metrics(SEXP Ycv, SEXP target, SEXP Z, SEXP expS) {
    char err[512] = "";
    const int n = Rf_nrows(Ycv), nf = Rf_ncols(Ycv);
    if ((int)XLENGTH(Z) != nf) Rf_error("ldsr: one fold per column of Ycv");
    int *zp = (int *)R_alloc((size_t)nf + 1, sizeof(int)), tot = 0;
    zp[0] = 0;
    for (int f = 0; f < nf; f++) {
        tot += (int)XLENGTH(VECTOR_ELT(Z, f));
        zp[f + 1] = tot;
    }
    int *zi = (int *)R_alloc((size_t)(tot > 0 ? tot : 1), sizeof(int));
    for (int f = 0; f < nf; f++)
        memcpy(zi + zp[f], INTEGER(VECTOR_ELT(Z, f)), sizeof(int) * (size_t)(zp[f + 1] - zp[f]));
    SEXP out = PROTECT(Rf_allocMatrix(REALSXP, 5, nf)); /* 5 x n_folds, like mapply's result */
    check(ldsr_cv_metrics_batch(0, n, nf, REAL(Ycv), REAL(target), zp, zi, Rf_asLogical(expS), REAL(out), err,
                                sizeof err),
          err);
    UNPROTECT(1);
    return out;
}

/* construct_rec for all ensemble members + the ensemble mean (R/LDS_reconstruction.R:190-212, 247-248).
 * X, V, Y: T x n matrices (one column per member).  Returns list(rec = T x 6 x n array, mean = T x 2). */
SEXP _ldsr_construct_rec(SEXP X, SEXP V, SEXP Y, SEXP C, SEXP R, SEXP muS, SEXP trS, SEXP lamS) {
    char err[512] = "";
    const int T = Rf_nrows(X), n = Rf_ncols(X);
    const char *nm[] = {"rec", "mean", ""};
    SEXP out = PROTECT(Rf_mkNamed(VECSXP, nm));
    SEXP rec = PROTECT(Rf_allocVector(REALSXP, (R_xlen_t)T * 6 * n)); /* [member][column][year], year fastest */
    SEXP mean = PROTECT(Rf_allocMatrix(REALSXP, T, 2));
    check(ldsr_construct_rec_batch(0, n, T, REAL(X), REAL(V), REAL(Y), REAL(C), REAL(R), Rf_asReal(muS),
                                   Rf_asInteger(trS), Rf_asReal(lamS), REAL(rec), REAL(mean), err, sizeof err),
          err);
    SET_VECTOR_ELT(out, 0, rec);
    SET_VECTOR_ELT(out, 1, mean);
    UNPROTECT(3);
    return out;
}

/* _ldsr_cv_metrics for many stations in one device call (ldsr_cv_metrics_stations).  Ycv: list of n_s x n_folds_s
 * matrices; target: list of numeric vectors (n_s); Z: list of lists of integer vectors (1-based into the station's
 * target).  Returns a list of 5 x n_folds_s matrices. */
SEXP _ldsr_cv_metrics_stations(SEXP Ycv, SEXP target, SEXP Z, SEXP expS) {
    char err[512] = "";
    const int S = (int)XLENGTH(Ycv);
    if ((int)XLENGTH(target) != S || (int)XLENGTH(Z) != S) Rf_error("ldsr: one Ycv, target and Z per station");
    int *n = (int *)R_alloc((size_t)S, sizeof(int)), *fp = (int *)R_alloc((size_t)S + 1, sizeof(int));
    R_xlen_t n_sim = 0, n_obs = 0, n_idx = 0;
    fp[0] = 0;
    for (int s = 0; s < S; s++) {
        SEXP Y = VECTOR_ELT(Ycv, s), zs = VECTOR_ELT(Z, s);
        n[s] = (int)XLENGTH(VECTOR_ELT(target, s));
        if (Rf_nrows(Y) != n[s] || Rf_ncols(Y) != (int)XLENGTH(zs))
            Rf_error("ldsr: station %d: Ycv must be length(target) x length(Z)", s + 1);
        fp[s + 1] = fp[s] + (int)XLENGTH(zs);
        n_sim += XLENGTH(Y);
        n_obs += n[s];
        for (R_xlen_t f = 0; f < XLENGTH(zs); f++) n_idx += XLENGTH(VECTOR_ELT(zs, f));
    }
    const int nf = fp[S];
    double *sim = (double *)R_alloc((size_t)(n_sim > 0 ? n_sim : 1), sizeof(double));
    double *obs = (double *)R_alloc((size_t)(n_obs > 0 ? n_obs : 1), sizeof(double));
    int *zp = (int *)R_alloc((size_t)nf + 1, sizeof(int)), *zi = (int *)R_alloc((size_t)(n_idx > 0 ? n_idx : 1), sizeof(int));
    double *ps = sim, *po = obs;
    int f = 0;
    zp[0] = 0;
    for (int s = 0; s < S; s++) {
        SEXP zs = VECTOR_ELT(Z, s);
        memcpy(ps, REAL(VECTOR_ELT(Ycv, s)), sizeof(double) * (size_t)XLENGTH(VECTOR_ELT(Ycv, s)));
        ps += XLENGTH(VECTOR_ELT(Ycv, s));
        memcpy(po, REAL(VECTOR_ELT(target, s)), sizeof(double) * (size_t)n[s]);
        po += n[s];
        for (R_xlen_t k = 0; k < XLENGTH(zs); k++, f++) {
            const int len = (int)XLENGTH(VECTOR_ELT(zs, k));
            memcpy(zi + zp[f], INTEGER(VECTOR_ELT(zs, k)), sizeof(int) * (size_t)len);
            zp[f + 1] = zp[f] + len;
        }
    }
    double *o = (double *)R_alloc((size_t)nf * 5, sizeof(double));
    check(ldsr_cv_metrics_stations(0, S, n, fp, sim, obs, zp, zi, Rf_asLogical(expS), o, err, sizeof err), err);
    SEXP out = PROTECT(Rf_allocVector(VECSXP, S));
    for (int s = 0; s < S; s++) { /* 5 x n_folds_s, like mapply's result */
        SEXP m = PROTECT(Rf_allocMatrix(REALSXP, 5, fp[s + 1] - fp[s]));
        memcpy(REAL(m), o + (size_t)fp[s] * 5, sizeof(double) * 5 * (size_t)(fp[s + 1] - fp[s]));
        SET_VECTOR_ELT(out, s, m);
        UNPROTECT(1);
    }
    UNPROTECT(1);
    return out;
}

/* _ldsr_construct_rec for many stations in one device call (ldsr_construct_rec_stations).  X, V, Y: lists of
 * T_s x n_s matrices (one column per member); C, R: lists of numeric vectors (n_s); mu, lambda: numeric vectors
 * (one value per station).  Returns a list of list(rec = T_s x 6 x n_s array, mean = T_s x 2). */
SEXP _ldsr_construct_rec_stations(SEXP X, SEXP V, SEXP Y, SEXP C, SEXP R, SEXP muS, SEXP trS, SEXP lamS) {
    char err[512] = "";
    const int S = (int)XLENGTH(X);
    if ((int)XLENGTH(V) != S || (int)XLENGTH(Y) != S || (int)XLENGTH(C) != S || (int)XLENGTH(R) != S ||
        (int)XLENGTH(muS) != S || (int)XLENGTH(lamS) != S)
        Rf_error("ldsr: one X, V, Y, C, R, mu and lambda per station");
    int *T = (int *)R_alloc((size_t)S, sizeof(int)), *mp = (int *)R_alloc((size_t)S + 1, sizeof(int));
    R_xlen_t rows = 0, years = 0;
    mp[0] = 0;
    for (int s = 0; s < S; s++) {
        T[s] = Rf_nrows(VECTOR_ELT(X, s));
        mp[s + 1] = mp[s] + Rf_ncols(VECTOR_ELT(X, s));
        if (XLENGTH(VECTOR_ELT(V, s)) != XLENGTH(VECTOR_ELT(X, s)) || XLENGTH(VECTOR_ELT(Y, s)) != XLENGTH(VECTOR_ELT(X, s)) ||
            (int)XLENGTH(VECTOR_ELT(C, s)) != mp[s + 1] - mp[s] || (int)XLENGTH(VECTOR_ELT(R, s)) != mp[s + 1] - mp[s])
            Rf_error("ldsr: station %d: X, V, Y must be T x n and C, R of length n", s + 1);
        rows += XLENGTH(VECTOR_ELT(X, s));
        years += T[s];
    }
    const size_t nr = (size_t)(rows > 0 ? rows : 1);
    double *x = (double *)R_alloc(nr, sizeof(double)), *v = (double *)R_alloc(nr, sizeof(double));
    double *y = (double *)R_alloc(nr, sizeof(double));
    double *c = (double *)R_alloc((size_t)mp[S] + 1, sizeof(double)), *r = (double *)R_alloc((size_t)mp[S] + 1, sizeof(double));
    for (int s = 0, off = 0; s < S; s++) {
        const size_t len = (size_t)XLENGTH(VECTOR_ELT(X, s));
        memcpy(x + off, REAL(VECTOR_ELT(X, s)), sizeof(double) * len);
        memcpy(v + off, REAL(VECTOR_ELT(V, s)), sizeof(double) * len);
        memcpy(y + off, REAL(VECTOR_ELT(Y, s)), sizeof(double) * len);
        memcpy(c + mp[s], REAL(VECTOR_ELT(C, s)), sizeof(double) * (size_t)(mp[s + 1] - mp[s]));
        memcpy(r + mp[s], REAL(VECTOR_ELT(R, s)), sizeof(double) * (size_t)(mp[s + 1] - mp[s]));
        off += (int)len;
    }
    double *rec = (double *)R_alloc(6 * nr, sizeof(double)), *mean = (double *)R_alloc(2 * (size_t)years + 1, sizeof(double));
    check(ldsr_construct_rec_stations(0, S, T, mp, x, v, y, c, r, REAL(muS), REAL(lamS), Rf_asInteger(trS), rec, mean, err,
                                      sizeof err),
          err);
    const char *nm[] = {"rec", "mean", ""};
    SEXP out = PROTECT(Rf_allocVector(VECSXP, S));
    double *pr = rec, *pm = mean;
    for (int s = 0; s < S; s++) {
        const size_t n6 = 6 * (size_t)XLENGTH(VECTOR_ELT(X, s));
        SEXP one = PROTECT(Rf_mkNamed(VECSXP, nm));
        SEXP a = PROTECT(Rf_allocVector(REALSXP, (R_xlen_t)n6)); /* [member][column][year], year fastest */
        SEXP m = PROTECT(Rf_allocMatrix(REALSXP, T[s], 2));
        memcpy(REAL(a), pr, sizeof(double) * n6);
        memcpy(REAL(m), pm, sizeof(double) * 2 * (size_t)T[s]);
        pr += n6;
        pm += 2 * (size_t)T[s];
        SET_VECTOR_ELT(one, 0, a);
        SET_VECTOR_ELT(one, 1, m);
        SET_VECTOR_ELT(out, s, one);
        UNPROTECT(3);
    }
    UNPROTECT(1);
    return out;
}

/* penalized_likelihood / negLogLik / ssqTrain (R/LDS_GA.R:28-44, 136-147) for a population of
 * parameter vectors (the columns of `thetas`, in vec_to_list order, R/LDS_GA.R:6-16) in one call. */
SEXP _ldsr_objective(SEXP y, SEXP u, SEXP v, SEXP thetas, SEXP kindS, SEXP lamS) {
    char err[512] = "";
    const int T = Rf_ncols(y), n = Rf_ncols(thetas), stride = Rf_nrows(thetas);
    int p = 0, q = 0;
    const double *up = input_ptr(u, T, &p), *vp = input_ptr(v, T, &q);
    const double *yp = REAL(y);
    int Ts = T, zero = 0, *fg = (int *)R_alloc((size_t)n, sizeof(int));
    for (int i = 0; i < n; i++) fg[i] = 0;
    ldsr_batch b;
    memset(&b, 0, sizeof b);
    b.n_series = 1; b.n_groups = 1; b.n_fits = n; b.theta_stride = stride;
    b.T = &Ts; b.p = &p; b.q = &q; b.y = &yp; b.u = &up; b.v = &vp;
    b.group_series = &zero; b.fit_group = fg; b.theta0 = REAL(thetas);
    SEXP out = PROTECT(Rf_allocVector(REALSXP, n));
    check(ldsr_objective_batch(ctx(), &b, Rf_asInteger(kindS), Rf_asReal(lamS), REAL(out), err, sizeof err), err);
    UNPROTECT(1);
    return out;
}

/* General state dimension (beyond the reference): theta holds R matrices, which are column-major;
 * the ABI wants row-major blocks. */
static void put_rowmajor(SEXP m, int rows, int cols, double *out) {
    if (Rf_nrows(m) * Rf_ncols(m) != rows * cols) Rf_error("ldsr: theta block has the wrong size");
    const double *x = REAL(m);
    for (int i = 0; i < rows; i++)
        for (int j = 0; j < cols; j++) out[i * cols + j] = x[j * rows + i];
}
SEXP _ldsr_smoother_d(SEXP y, SEXP u, SEXP v, SEXP theta, SEXP stdlik, SEXP methodS) {
    char err[512] = "";
    const int T = Rf_ncols(y);
    int p = 0, q = 0;
    const double *up = input_ptr(u, T, &p), *vp = input_ptr(v, T, &q);
    if (!up) p = 0;
    if (!vp) q = 0;
    const int d = Rf_nrows(list_get(theta, "A"));
    const int tl = 2 * d * d + d * p + d + q + 1 + d + d * d;
    double *th = (double *)R_alloc((size_t)tl, sizeof(double)), *o = th;
    put_rowmajor(list_get(theta, "A"), d, d, o); o += d * d;
    if (p) { put_rowmajor(list_get(theta, "B"), d, p, o); o += d * p; }
    put_rowmajor(list_get(theta, "C"), 1, d, o); o += d;
    if (q) { put_rowmajor(list_get(theta, "D"), 1, q, o); o += q; }
    put_rowmajor(list_get(theta, "Q"), d, d, o); o += d * d;
    *o++ = REAL(list_get(theta, "R"))[0];
    put_rowmajor(list_get(theta, "mu1"), d, 1, o); o += d;
    put_rowmajor(list_get(theta, "V1"), d, d, o);
    double *X = (double *)R_alloc((size_t)T * d, sizeof(double));
    double *V = (double *)R_alloc((size_t)T * d * d, sizeof(double));
    double *Y = (double *)R_alloc((size_t)T, sizeof(double)), lik;
    check(ldsr_smoother_d_batch(0, d, T, p, q, REAL(y), up, vp, 1, th, tl, Rf_asLogical(stdlik), Rf_asInteger(methodS), 0,
                                X, V, Y, &lik, NULL, err, sizeof err),
          err);
    const char *nm[] = {"X", "Y", "V", "lik", ""};
    SEXP out = PROTECT(Rf_mkNamed(VECSXP, nm));
    SEXP Xm = PROTECT(Rf_allocMatrix(REALSXP, d, T)); /* d x T: X[t][i] is already column-major */
    memcpy(REAL(Xm), X, sizeof(double) * (size_t)T * d);
    SEXP Vm = PROTECT(Rf_allocMatrix(REALSXP, d * d, T)); /* column t = vec(V_t) (symmetric) */
    memcpy(REAL(Vm), V, sizeof(double) * (size_t)T * d * d);
    SET_VECTOR_ELT(out, 0, Xm);
    SET_VECTOR_ELT(out, 1, mat1(Y, T));
    SET_VECTOR_ELT(out, 2, Vm);
    SET_VECTOR_ELT(out, 3, Rf_ScalarReal(lik));
    UNPROTECT(3);
    return out;
}

/* bytes of cached device memory handed back to the driver */
SEXP _ldsr_trim(void) { return Rf_ScalarReal(session_ctx ? (double)ldsr_ctx_trim(session_ctx, NULL) : 0.0); }

static const R_CallMethodDef CallEntries[] = {
    {"_ldsr_Kalman_smoother", (DL_FUNC)&_ldsr_Kalman_smoother, 5},
    {"_ldsr_Mstep", (DL_FUNC)&_ldsr_Mstep, 4},
    {"_ldsr_LDS_EM", (DL_FUNC)&_ldsr_LDS_EM, 6},
    {"_ldsr_propagate", (DL_FUNC)&_ldsr_propagate, 5},
    {"_ldsr_em_batch", (DL_FUNC)&_ldsr_em_batch, 8},
    {"_ldsr_rep_batch", (DL_FUNC)&_ldsr_rep_batch, 10},
    {"_ldsr_posterior_rep_batch", (DL_FUNC)&_ldsr_posterior_rep_batch, 8},
    {"_ldsr_posterior_stats_batch", (DL_FUNC)&_ldsr_posterior_stats_batch, 11},
    {"_ldsr_posterior_yearly_batch", (DL_FUNC)&_ldsr_posterior_yearly_batch, 12},
    {"_ldsr_posterior_quantile_batch", (DL_FUNC)&_ldsr_posterior_quantile_batch, 11},
    {"_ldsr_smoother_d", (DL_FUNC)&_ldsr_smoother_d, 6},
    {"_ldsr_cv_metrics", (DL_FUNC)&_ldsr_cv_metrics, 4},
    {"_ldsr_construct_rec", (DL_FUNC)&_ldsr_construct_rec, 8},
    {"_ldsr_cv_metrics_stations", (DL_FUNC)&_ldsr_cv_metrics_stations, 4},
    {"_ldsr_construct_rec_stations", (DL_FUNC)&_ldsr_construct_rec_stations, 8},
    {"_ldsr_objective", (DL_FUNC)&_ldsr_objective, 6},
    {"_ldsr_trim", (DL_FUNC)&_ldsr_trim, 0},
    {NULL, NULL, 0}};

void R_init_ldsr(DllInfo *dll) {
    R_registerRoutines(dll, NULL, CallEntries, NULL, NULL);
    R_useDynamicSymbols(dll, FALSE);
}

void R_unload_ldsr(DllInfo *dll) {
    (void)dll;
    if (session_ctx) ldsr_ctx_destroy(session_ctx);
    session_ctx = NULL;
}
