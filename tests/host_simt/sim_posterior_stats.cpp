// sim_posterior_stats.cpp -- TEST INFRASTRUCTURE: the statistics mode of posterior_rep_kernel
// (ldsr_b200/csrc/aux_kernels.cuh, posterior_rep_kernel<REP_TT, true>) compiled for the CPU and run by the coroutine
// emulator of host_simt.h after smoother_kernel's coefficient mode, with the set-up of sim_em.cpp (through
// sim_posterior.cpp).
//
//   g++ -O1 -g -std=c++17 -DLDSR_HOST_SIM -shared -fPIC sim_posterior_stats.cpp -o libldsr_hostsim_stats.so
//
// Built and driven by tests/test_posterior_stats_host.py; never linked into the product.
#include "sim_posterior.cpp"

namespace {

// As ldsr_posterior_stats_batch runs it: the coefficient pass, then ONE launch of the statistics mode over every
// (fit, 32 replicates) block with caller noise (one series here, so fit f's rows start at f T).
template <int PQ> int run_stats(int T, int p, int q, const double *y, const double *u, const double *v, int ng,
                                const int *held_ptr, const int *held_idx, int nf, const int *fit_group,
                                const double *theta, int n_reps, const double *z, const double *mu, int transform,
                                const double *lam, int n_win, const int *win, const double *thr, const int *range,
                                int order, double *wmin, int *wmin_at, double *wmax, int *wmax_at, int *run_len,
                                int *run_at, double *deficit, int *deficit_at, int *n_runs) {
    constexpr int TL = 2 * PQ + 6;
    const int stride = p + q + 6;
    Prep Pr;
    prepare<PQ>(T, p, q, y, u, v, ng, held_ptr, held_idx, Pr);
    std::vector<double> th((size_t)nf * TL), m((size_t)nf * T), o((size_t)nf * T), s((size_t)nf * T),
        J((size_t)nf * T), par((size_t)4 * nf);
    std::vector<long long> job_row(nf), fit_ptr(nf + 1), f_mask_off(nf);
    std::vector<int> job_theta(nf);
    for (int f = 0; f < nf; f++) {
        pad_theta<PQ>(theta + (size_t)f * stride, p, q, u != nullptr, v != nullptr, &th[(size_t)f * TL]);
        job_row[f] = fit_ptr[f] = (long long)f * T;
        job_theta[f] = f;
        f_mask_off[f] = Pr.g_mask_off[fit_group[f]];
        par[4 * f] = theta[(size_t)f * stride + 1 + p];
        par[4 * f + 1] = std::sqrt(theta[(size_t)f * stride + 3 + p + q]);
        par[4 * f + 2] = mu[f];
        par[4 * f + 3] = transform == 2 ? lam[f] : 0.0;
    }
    fit_ptr[nf] = (long long)nf * T;
    SmootherParams sp;
    std::memset(&sp, 0, sizeof sp);
    sp.series = &Pr.S;
    sp.blobs = Pr.blob.data();
    sp.g_series = Pr.g_series.data();
    sp.masks = Pr.masks.data();
    sp.g_mask_off = Pr.g_mask_off.data();
    sp.g_nobs = Pr.g_nobs.data();
    sp.n_jobs = nf;
    sp.job_group = fit_group;
    sp.job_theta = job_theta.data();
    sp.job_row = job_row.data();
    sp.theta = th.data();
    sp.X = m.data();
    sp.Y = o.data();
    sp.V = s.data();
    sp.J = J.data();
    hostsim::launch((nf + 63) / 64, 64, 0, order, [&] { smoother_kernel<PQ, true>(sp); });
    PostRepParams pp;
    std::memset(&pp, 0, sizeof pp);
    pp.m = m.data();
    pp.o = o.data();
    pp.s = s.data();
    pp.J = J.data();
    pp.fit_ptr = fit_ptr.data();
    pp.par = par.data();
    pp.masks = Pr.masks.data();
    pp.f_mask_off = f_mask_off.data();
    pp.z = z;
    pp.n_reps = n_reps;
    pp.wpf = (n_reps + 31) / 32;
    pp.n_blk = (long long)nf * pp.wpf;
    pp.transform = transform;
    pp.n_win = n_win;
    int longest = 0;
    for (int k = 0; k < n_win; k++) {
        pp.win[k] = win[k];
        longest = std::max(longest, win[k]);
    }
    for (pp.ring = n_win > 0 ? 1 : 0; pp.ring > 0 && pp.ring < longest;) pp.ring *= 2;
    pp.n_rows = (long long)nf * n_reps;
    pp.range = range;
    pp.thr = thr;
    pp.wmin = wmin;
    pp.wmin_at = wmin_at;
    pp.wmax = wmax;
    pp.wmax_at = wmax_at;
    pp.run_len = run_len;
    pp.run_at = run_at;
    pp.deficit = deficit;
    pp.deficit_at = deficit_at;
    pp.n_runs = n_runs;
    hostsim::launch((int)((pp.n_blk + REP_WARPS - 1) / REP_WARPS), REP_WARPS * 32,
                    posterior_stats_smem_bytes<REP_TT>(true, pp.ring), order,
                    [&] { posterior_rep_kernel<REP_TT, true>(pp); });
    return 0;
}

} // namespace

// The statistics mode with caller noise, padded to width 3, 5 or 16; arguments as hostsim_posterior_rep's, then the
// statistics spec (range [n_fits][2], thr [n_fits] or NULL) and the outputs of ldsr_posterior_stats_batch (any NULL).
extern "C" int hostsim_posterior_stats(int T, int p, int q, const double *y, const double *u, const double *v,
                                       int n_groups, const int *held_ptr, const int *held_idx, int n_fits,
                                       const int *fit_group, const double *theta, int n_reps, const double *z,
                                       const double *mu, int transform, const double *lam, int n_win, const int *win,
                                       const double *thr, const int *range, int order, double *wmin, int *wmin_at,
                                       double *wmax, int *wmax_at, int *run_len, int *run_at, double *deficit,
                                       int *deficit_at, int *n_runs) {
    const int need = std::max(1, std::max(u ? p : 0, v ? q : 0));
#define LDSR_STATS(W)                                                                                              \
    return run_stats<W>(T, p, q, y, u, v, n_groups, held_ptr, held_idx, n_fits, fit_group, theta, n_reps, z, mu,   \
                        transform, lam, n_win, win, thr, range, order, wmin, wmin_at, wmax, wmax_at, run_len,      \
                        run_at, deficit, deficit_at, n_runs)
    if (need <= 3) LDSR_STATS(3);
    if (need <= 5) LDSR_STATS(5);
    if (need <= 16) LDSR_STATS(16);
#undef LDSR_STATS
    return 13;
}
