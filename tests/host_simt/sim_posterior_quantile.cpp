// sim_posterior_quantile.cpp -- TEST INFRASTRUCTURE: the quantile selection of ldsr_posterior_quantile_batch
// (ldsr_b200/csrc/aux_kernels.cuh: posterior_rep_kernel<REP_TT, POST_QUANT> and the quant_* kernels) compiled for the
// CPU and run by the coroutine emulator of host_simt.h after smoother_kernel's coefficient mode, with the set-up of
// sim_em.cpp (through sim_posterior.cpp).
//
//   g++ -O1 -g -std=c++17 -DLDSR_HOST_SIM -shared -fPIC sim_posterior_quantile.cpp -o libldsr_hostsim_quant.so
//
// Built and driven by tests/test_posterior_quantile_host.py; never linked into the product.
#include "sim_posterior.cpp"

namespace {

// As ldsr_posterior_quantile_batch runs it: the coefficient pass, the range pass, quant_init_kernel<>, then plan /
// selection pass / bracket kernel until no bracket is left, and quant_out_kernel<>; caller noise, one series (fit f's
// rows start at f T).  nb_log2 and cap are the bins and the collect cap; stats[0] counts the sampler passes,
// stats[1] the histogram brackets and stats[2] the collected brackets over all passes.
template <int PQ> int run_quant(int T, int p, int q, const double *y, const double *u, const double *v, int ng,
                                const int *held_ptr, const int *held_idx, int nf, const int *fit_group,
                                const double *theta, int n_reps, const double *z, const double *mu, int transform,
                                const double *lam, int n_win, const int *win, int n_lev, const double *lev,
                                const int *range, int nb_log2, int cap, int order, double *qout, int *nonfinite,
                                long long *stats) {
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
    for (pp.ring = 1; pp.ring < longest;) pp.ring *= 2;
    pp.range = range;
    const long long ns = fit_ptr[nf], n_slots = n_win * ns;
    pp.n_steps = ns;
    pp.n_lev = n_lev;
    QuantParams Q;
    std::memset(&Q, 0, sizeof Q);
    Q.n_slots = n_slots;
    Q.n_steps = ns;
    Q.n_lev = n_lev;
    Q.nb_log2 = nb_log2;
    Q.cap = cap;
    Q.n_reps = n_reps;
    for (int l = 0; l < n_lev; l++) Q.lev[l] = lev[l];
    std::vector<int> n0((size_t)n_slots, -1), slot_nbr((size_t)n_slots), slot_br((size_t)n_slots * n_lev);
    for (int k = 0; k < n_win; k++)
        for (int f = 0; f < nf; f++)
            for (int t = range[2 * f]; t <= range[2 * f + 1] - win[k]; t++) n0[(size_t)(k * ns + fit_ptr[f] + t)] = 0;
    std::vector<unsigned long long> kmin((size_t)n_slots, ~0ull), kmax((size_t)n_slots, 0ull), ctr(4, ~0ull), seg;
    std::vector<QuantLevel> lv((size_t)n_slots * n_lev);
    std::vector<QuantBracket> br((size_t)n_slots * n_lev);
    std::vector<unsigned> hist;
    pp.q_n = n0.data();
    pp.q_min = kmin.data();
    pp.q_max = kmax.data();
    pp.q_slot_nbr = slot_nbr.data();
    pp.q_slot_br = slot_br.data();
    pp.q_br = br.data();
    Q.n = n0.data();
    Q.kmin = kmin.data();
    Q.kmax = kmax.data();
    Q.lv = lv.data();
    Q.br = br.data();
    Q.slot_nbr = slot_nbr.data();
    Q.slot_br = slot_br.data();
    Q.ctr = ctr.data();
    Q.q = qout;
    Q.nonfinite = nonfinite;
    const unsigned slot_grid = (unsigned)((n_slots + 255) / 256);
    auto sampler = [&] {
        hostsim::launch((int)((pp.n_blk + REP_WARPS - 1) / REP_WARPS), REP_WARPS * 32,
                        posterior_stats_smem_bytes<REP_TT>(true, pp.ring), order,
                        [&] { posterior_rep_kernel<REP_TT, POST_QUANT>(pp); });
        stats[0]++;
    };
    pp.qpass = QUANT_RANGE;
    sampler();
    hostsim::launch(slot_grid, 256, 0, order, [&] { quant_init_kernel<>(Q); });
    for (;;) {
        ctr[0] = ctr[1] = ctr[2] = 0;
        hostsim::launch(slot_grid, 256, 0, order, [&] { quant_plan_kernel<>(Q); });
        if (ctr[3] != ~0ull) return 20; // two passes disagreed
        if (ctr[0] == 0) break;
        if (stats[0] >= 2 + (64 + nb_log2 - 1) / nb_log2) return 21; // did not settle
        hist.assign((size_t)ctr[1] << nb_log2, 0u);
        seg.assign(std::max<size_t>(ctr[2], 1), 0ull);
        stats[1] += (long long)ctr[1];
        stats[2] += (long long)(ctr[0] - ctr[1]);
        pp.qpass = QUANT_SELECT;
        Q.hist = pp.q_hist = hist.data();
        Q.seg = pp.q_seg = seg.data();
        sampler();
        Q.n_br = (long long)ctr[0]; // two CTAs walk every bracket (one CTA per bracket costs a CTA's stacks each)
        hostsim::launch(2, QUANT_THREADS, 0, order, [&] { quant_bracket_kernel<>(Q); });
    }
    hostsim::launch(slot_grid, 256, 0, order, [&] { quant_out_kernel<>(Q); });
    return 0;
}

} // namespace

// The quantile selection with caller noise, padded to width 3, 5 or 16; arguments as hostsim_posterior_rep's, then
// the spec (windows, levels, range [n_fits][2]), the bins (log2) and collect cap, the schedule, the outputs of
// ldsr_posterior_quantile_batch (q [n_win][n_lev][n_fits T], nonfinite [n_win][n_fits T]) and stats[3].
extern "C" int hostsim_posterior_quantile(int T, int p, int q, const double *y, const double *u, const double *v,
                                          int n_groups, const int *held_ptr, const int *held_idx, int n_fits,
                                          const int *fit_group, const double *theta, int n_reps, const double *z,
                                          const double *mu, int transform, const double *lam, int n_win,
                                          const int *win, int n_lev, const double *lev, const int *range, int nb_log2,
                                          int cap, int order, double *qout, int *nonfinite, long long *stats) {
    const int need = std::max(1, std::max(u ? p : 0, v ? q : 0));
#define LDSR_QUANT(W)                                                                                              \
    return run_quant<W>(T, p, q, y, u, v, n_groups, held_ptr, held_idx, n_fits, fit_group, theta, n_reps, z, mu,   \
                        transform, lam, n_win, win, n_lev, lev, range, nb_log2, cap, order, qout, nonfinite, stats)
    if (need <= 3) LDSR_QUANT(3);
    if (need <= 5) LDSR_QUANT(5);
    if (need <= 16) LDSR_QUANT(16);
#undef LDSR_QUANT
    return 13;
}
