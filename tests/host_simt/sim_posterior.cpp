// sim_posterior.cpp -- TEST INFRASTRUCTURE: smoother_kernel's coefficient mode and posterior_rep_kernel
// (ldsr_b200/csrc/aux_kernels.cuh) compiled for the CPU and run by the coroutine emulator of host_simt.h, with the
// set-up of sim_em.cpp (prepare, pad_theta).
//
//   g++ -O1 -g -std=c++17 -DLDSR_HOST_SIM -shared -fPIC sim_posterior.cpp -o libldsr_hostsim_post.so
//
// Built and driven by tests/test_posterior_rep_host.py; never linked into the product.
#include "sim_em.cpp"

namespace {

// Conditioned replicates: smoother_kernel's coefficient mode, then posterior_rep_kernel with caller noise, as
// ldsr_posterior_rep_batch runs them (one series here, so fit f's rows start at f T).  chunk_blk > 0 cuts the
// sampler into launches of that many (fit, 32 replicates) blocks, each writing from its own output offset.
template <int PQ> int run_posterior(int T, int p, int q, const double *y, const double *u, const double *v, int ng,
                                    const int *held_ptr, const int *held_idx, int nf, const int *fit_group,
                                    const double *theta, int n_reps, const double *z, const double *mu, int transform,
                                    const double *lam, int order, int chunk_blk, double *simX, double *simY,
                                    double *simQ) {
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
    const int wpf = (n_reps + 31) / 32;
    const long long n_blk = (long long)nf * wpf;
    const long long per = chunk_blk > 0 ? chunk_blk : n_blk;
    for (long long b0 = 0; b0 < n_blk; b0 += per) {
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
        pp.n_reps = n_reps;
        pp.wpf = wpf;
        pp.blk0 = b0;
        pp.n_blk = std::min(per, n_blk - b0);
        const int f0 = (int)(b0 / wpf), r0 = (int)(b0 % wpf) * 32;
        pp.out0 = (long long)n_reps * fit_ptr[f0] + (long long)r0 * T;
        pp.z = z + 2 * pp.out0;
        pp.transform = transform;
        pp.simX = simX ? simX + pp.out0 : nullptr;
        pp.simY = simY ? simY + pp.out0 : nullptr;
        pp.simQ = simQ ? simQ + pp.out0 : nullptr;
        hostsim::launch((int)((pp.n_blk + REP_WARPS - 1) / REP_WARPS), REP_WARPS * 32, posterior_smem_bytes<REP_TT>(true), order,
                        [&] { posterior_rep_kernel<REP_TT>(pp); });
    }
    return 0;
}

} // namespace

// smoother_kernel's coefficient mode and posterior_rep_kernel in caller-noise mode, padded to width 3, 5 or 16; one
// series, fits as hostsim_step's jobs.  Outputs ([n_fits][n_reps][T], fit-major) may be NULL.
extern "C" int hostsim_posterior_rep(int T, int p, int q, const double *y, const double *u, const double *v,
                                     int n_groups, const int *held_ptr, const int *held_idx, int n_fits,
                                     const int *fit_group, const double *theta, int n_reps, const double *z,
                                     const double *mu, int transform, const double *lam, int order, int chunk_blk,
                                     double *simX, double *simY, double *simQ) {
    const int need = std::max(1, std::max(u ? p : 0, v ? q : 0));
#define LDSR_POST(W)                                                                                              \
    return run_posterior<W>(T, p, q, y, u, v, n_groups, held_ptr, held_idx, n_fits, fit_group, theta, n_reps, z, mu, \
                            transform, lam, order, chunk_blk, simX, simY, simQ)
    if (need <= 3) LDSR_POST(3);
    if (need <= 5) LDSR_POST(5);
    if (need <= 16) LDSR_POST(16);
#undef LDSR_POST
    return 13;
}
