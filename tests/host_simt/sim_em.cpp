// sim_em.cpp -- TEST INFRASTRUCTURE: the EM kernels' and the single-step kernels' SOURCE (ldsr_b200/csrc/*.cuh)
// compiled for the CPU and run by the coroutine emulator of host_simt.h on one series.  The host side here
// re-states what plan_build / setup_kernel / compact_kernel prepare (blob, masks, Gram constants, task list) with
// plain loops, so the comparison with the oracle also covers those conventions.
//
//   g++ -O1 -g -std=c++17 -DLDSR_HOST_SIM -shared -fPIC sim_em.cpp -o libldsr_hostsim.so
//
// Built and driven by tests/test_host_simt.py; never linked into the product.
#include "host_simt.h"

#include "../../ldsr_b200/csrc/em_split_kernel.cuh"
#ifdef LDSR_HAVE_WIDE
#include "../../ldsr_b200/csrc/em_wide_kernel.cuh"
#endif
#ifdef LDSR_HAVE_SCAN
#include "../../ldsr_b200/csrc/em_scan_kernel.cuh"
#endif
#include "../../ldsr_b200/csrc/aux_kernels.cuh"

#include <vector>

using namespace ldsr;

namespace {

// inverse of a symmetric positive definite n x n matrix (row-major, ld = n) by Gauss-Jordan
bool invert(std::vector<double> &a, int n) {
    std::vector<double> inv((size_t)n * n, 0.0);
    for (int i = 0; i < n; i++) inv[(size_t)i * n + i] = 1.0;
    for (int c = 0; c < n; c++) {
        int piv = c;
        for (int r = c + 1; r < n; r++)
            if (std::fabs(a[(size_t)r * n + c]) > std::fabs(a[(size_t)piv * n + c])) piv = r;
        if (!(std::fabs(a[(size_t)piv * n + c]) > 0.0)) return false;
        for (int k = 0; k < n; k++) {
            std::swap(a[(size_t)c * n + k], a[(size_t)piv * n + k]);
            std::swap(inv[(size_t)c * n + k], inv[(size_t)piv * n + k]);
        }
        const double d = 1.0 / a[(size_t)c * n + c];
        for (int k = 0; k < n; k++) {
            a[(size_t)c * n + k] *= d;
            inv[(size_t)c * n + k] *= d;
        }
        for (int r = 0; r < n; r++) {
            if (r == c) continue;
            const double f = a[(size_t)r * n + c];
            if (f == 0.0) continue;
            for (int k = 0; k < n; k++) {
                a[(size_t)r * n + k] -= f * a[(size_t)c * n + k];
                inv[(size_t)r * n + k] -= f * inv[(size_t)c * n + k];
            }
        }
    }
    a = inv;
    return true;
}

// Gram block of `rows` ([T][PQ], first n_real columns real) over the steps with keep[t], inverted and
// embedded in PQ x PQ (zero outside the real block)
bool gram_inverse(const double *rows, int T_end, int PQ, int n_real, const std::vector<char> &keep,
                  std::vector<double> &out) {
    std::vector<double> g((size_t)n_real * n_real, 0.0);
    for (int t = 0; t < T_end; t++) {
        if (!keep[t]) continue;
        for (int a = 0; a < n_real; a++)
            for (int b = 0; b < n_real; b++) g[(size_t)a * n_real + b] += rows[(size_t)t * PQ + a] * rows[(size_t)t * PQ + b];
    }
    const bool ok = n_real == 0 || invert(g, n_real);
    out.assign((size_t)PQ * PQ, 0.0);
    if (ok)
        for (int a = 0; a < n_real; a++)
            for (int b = 0; b < n_real; b++) out[(size_t)a * PQ + b] = g[(size_t)a * n_real + b];
    return ok;
}

struct Job {
    int kind, T, p, q, n_groups, n_fits, niter, chunk, order, grid_cap;
    const double *y, *u, *v;
    const int *held_ptr, *held_idx, *fit_group;
    const double *theta0;
    double tol;
    double *theta_out, *lik_out;
    int *iters_out;
    double *traj_out = nullptr; // optional [4][n_fits][T]: X, Y, V, J of every fit's final theta (scan kernel, EMIT mode)
};

#ifdef LDSR_HAVE_WIDE
template <int PQ> int launch_wide_hostsim(const EmParams &ep, const SeriesDev &S, const double *y, size_t blob_sm,
                                          int grid, int order) {
#ifndef LDSR_WIDE_NW
#define LDSR_WIDE_NW 8
#endif
    constexpr int NW = LDSR_WIDE_NW, MSEG = 8, UW = 32;
    int nu = 0, nm = 0;
    wide_count_units(y, S.T, MSEG, UW, &nu, &nm);
    WideParams wp;
    wp.em = ep;
    wp.max_units = nu;
    wp.max_msteps = nm;
    wp.max_T = S.T;
    const size_t wblob = wide_blob_smem((size_t)S.blob_doubles * 8, S.T);
    (void)blob_sm;
    wp.blob_smem = (int)wblob;
    wp.cost_u = UW * 17 / 2;
    wp.cost_m = MSEG * 90;
    const size_t smem = wblob + wide_smem_bytes(PQ, NW, S.T, nu, nm);
    hostsim::launch(grid, NW * 32, smem, order, [&] { em_wide_kernel<PQ, NW, MSEG, UW>(wp); });
    return 0;
}
#endif

// What plan_build and setup_kernel prepare for one series and its groups: the blob, the window Gram blocks of u,
// the series constant (TuuInv over t < T - 1, then its singular flag), and per group the observed-step mask, the
// Gram constants and the status.
struct Prep {
    SeriesDev S;
    std::vector<double> blob, uwin, sconst, gconst;
    std::vector<unsigned> masks;
    std::vector<long long> g_mask_off;
    std::vector<int> g_status, g_series, g_nobs;
    bool tuu_singular = false;
};

template <int PQ> void prepare(int T, int p, int q, const double *y, const double *u, const double *v, int ng,
                               const int *held_ptr, const int *held_idx, Prep &P) {
    constexpr int UW = 32;
    // ---- blob (plan_build)
    SeriesDev &S = P.S;
    std::memset(&S, 0, sizeof S);
    S.T = T;
    S.p = p;
    S.q = q;
    S.has_u = u != nullptr;
    S.has_v = v != nullptr;
    S.same_uv = (u && v && p == q && std::memcmp(u, v, sizeof(double) * (size_t)p * T) == 0) || (!u && !v);
    const int Ty = (T + 1) & ~1, nuv = T * PQ;
    S.y_off = 0;
    S.u_off = Ty;
    S.v_off = S.same_uv ? S.u_off : ((S.u_off + nuv + 1) & ~1);
    S.blob_doubles = ((S.v_off + nuv) + 1) & ~1;
    std::vector<double> &blob = P.blob;
    blob.assign((size_t)S.blob_doubles, 0.0);
    for (int t = 0; t < T; t++) {
        blob[t] = y[t];
        if (u)
            for (int j = 0; j < p; j++) blob[S.u_off + (size_t)t * PQ + j] = u[(size_t)t * p + j];
        if (v && !S.same_uv)
            for (int j = 0; j < q; j++) blob[S.v_off + (size_t)t * PQ + j] = v[(size_t)t * q + j];
    }
    const int nwin = (T + UW - 1) / UW;
    P.uwin.assign((size_t)nwin * PQ * PQ, 0.0);
    if (u)
        for (int t = 0; t < T; t++)
            for (int a = 0; a < p; a++)
                for (int c = 0; c < p; c++)
                    P.uwin[(size_t)(t / UW) * PQ * PQ + a * PQ + c] += u[(size_t)t * p + a] * u[(size_t)t * p + c];
    // ---- series constant: TuuInv over t < T-1
    {
        std::vector<char> keep(T, 1);
        P.tuu_singular = !gram_inverse(blob.data() + S.u_off, T - 1, PQ, u ? p : 0, keep, P.sconst);
        P.sconst.push_back(P.tuu_singular ? 1.0 : 0.0);
    }
    // ---- groups: masks + constants (setup_kernel, merge_status_kernel)
    const int nwords = (T + 31) / 32;
    P.masks.assign((size_t)ng * nwords, 0u);
    P.g_mask_off.assign(ng, 0);
    P.gconst.assign((size_t)ng * gconst_stride(PQ), 0.0);
    P.g_status.assign(ng, 0);
    P.g_series.assign(ng, 0);
    P.g_nobs.assign(ng, 0);
    for (int g = 0; g < ng; g++) {
        P.g_mask_off[g] = (long long)g * nwords;
        std::vector<char> keep(T, 0);
        for (int t = 0; t < T; t++) keep[t] = std::isfinite(y[t]) ? 1 : 0;
        if (held_ptr)
            for (int k = held_ptr[g]; k < held_ptr[g + 1]; k++) keep[held_idx[k]] = 0;
        for (int t = 0; t < T; t++)
            if (keep[t]) P.masks[(size_t)g * nwords + (t >> 5)] |= 1u << (t & 31);
        double *gc = P.gconst.data() + (size_t)g * gconst_stride(PQ);
        const double *vr = blob.data() + S.v_off;
        std::vector<double> svv_inv;
        if (!gram_inverse(vr, T, PQ, v ? q : 0, keep, svv_inv) || P.tuu_singular) P.g_status[g] = 1;
        double Syy = 0.0, n_obs = 0.0;
        std::vector<double> Syv(PQ, 0.0);
        for (int t = 0; t < T; t++) {
            if (!keep[t]) continue;
            Syy += y[t] * y[t];
            n_obs += 1.0;
            for (int a = 0; a < PQ; a++) Syv[a] += y[t] * vr[(size_t)t * PQ + a];
        }
        gc[0] = Syy;
        gc[1] = n_obs;
        P.g_nobs[g] = (int)n_obs;
        for (int a = 0; a < PQ; a++) {
            gc[2 + a] = Syv[a];
            double acc = 0.0;
            for (int b = 0; b < PQ; b++) acc += svv_inv[(size_t)a * PQ + b] * Syv[b];
            gc[2 + PQ + a] = acc;
        }
        for (int e = 0; e < PQ * PQ; e++) gc[2 + 2 * PQ + e] = svv_inv[e];
    }
}

// a caller theta (p, q) in the device layout (PQ, PQ) and back (ldsr_abi.cu: pad_theta, unpad_theta)
template <int PQ> void pad_theta(const double *src, int p, int q, bool has_u, bool has_v, double *dst) {
    std::fill(dst, dst + 2 * PQ + 6, 0.0);
    dst[0] = src[0];
    if (has_u)
        for (int j = 0; j < p; j++) dst[1 + j] = src[1 + j];
    dst[1 + PQ] = src[1 + p];
    if (has_v)
        for (int j = 0; j < q; j++) dst[2 + PQ + j] = src[2 + p + j];
    for (int k = 0; k < 4; k++) dst[2 + 2 * PQ + k] = src[2 + p + q + k];
}
template <int PQ> void unpad_theta(const double *src, int p, int q, bool has_u, bool has_v, double *dst) {
    dst[0] = src[0];
    for (int j = 0; j < p; j++) dst[1 + j] = has_u ? src[1 + j] : 0.0;
    dst[1 + p] = src[1 + PQ];
    for (int j = 0; j < q; j++) dst[2 + p + j] = has_v ? src[2 + PQ + j] : 0.0;
    for (int k = 0; k < 4; k++) dst[2 + p + q + k] = src[2 + 2 * PQ + k];
}

template <int PQ> int run(const Job &J) {
    constexpr int NW = 4, MSEG = 4, UW = 32;
    const int T = J.T, p = J.p, q = J.q, ng = J.n_groups, nf = J.n_fits;
    constexpr int TL = 2 * PQ + 6;
    Prep Pr;
    prepare<PQ>(T, p, q, J.y, J.u, J.v, ng, J.held_ptr, J.held_idx, Pr);
    if (Pr.tuu_singular) return 10;
    SeriesDev &S = Pr.S;
    S.fit_begin = 0;
    S.fit_end = nf;
    std::vector<double> &blob = Pr.blob, &uwin = Pr.uwin, &sconst = Pr.sconst, &gconst = Pr.gconst;
    std::vector<unsigned> &masks = Pr.masks;
    std::vector<long long> &g_mask_off = Pr.g_mask_off;
    std::vector<int> &g_status = Pr.g_status, &g_series = Pr.g_series;
    // ---- fits
    std::vector<double> theta((size_t)nf * TL, 0.0), l1(nf, 0.0), l2(nf, 0.0), lik(nf, std::nan(""));
    std::vector<int> ne(nf, 0), done(nf, 0), f_group(J.fit_group, J.fit_group + nf), f_user(nf);
    const int stride = p + q + 6;
    for (int f = 0; f < nf; f++) {
        f_user[f] = f;
        pad_theta<PQ>(J.theta0 + (size_t)f * stride, p, q, J.u != nullptr, J.v != nullptr, &theta[(size_t)f * TL]);
    }
    std::vector<int> active(nf, 0);
    std::vector<int4> tasks(nf + 2);
    int n_tasks = 0;

    EmParams ep;
    std::memset(&ep, 0, sizeof ep);
    ep.series = &S;
    ep.blobs = blob.data();
    ep.sconst = sconst.data();
    ep.uwin = uwin.data();
    ep.g_series = g_series.data();
    ep.masks = masks.data();
    ep.g_mask_off = g_mask_off.data();
    ep.gconst = gconst.data();
    ep.g_status = g_status.data();
    ep.f_group = f_group.data();
    ep.theta = theta.data();
    ep.l1 = l1.data();
    ep.l2 = l2.data();
    ep.lik = lik.data();
    ep.ne = ne.data();
    ep.done = done.data();
    ep.liks = nullptr;
    ep.f_user = f_user.data();
    ep.active = active.data();
    ep.tasks = tasks.data();
    ep.n_tasks = &n_tasks;
    ep.niter = J.niter;
    ep.chunk = J.chunk;
    ep.tol = J.tol;
    const size_t blob_sm = ((size_t)S.blob_doubles * 8 + 127) & ~size_t(127);
    const int max_units = split_units_upper_bound(J.y, T, MSEG, UW);
    const int max_uunits = (T + UW - 1) / UW;

    const int max_chunks = (J.niter + J.chunk - 1) / J.chunk;
    std::vector<int> share_flags, share_ctl, share_order;
    for (int c = 0; c < max_chunks; c++) {
        // compact_kernel: live fits in order, 32 (or 128) per CTA
        const int per = J.kind == 2 ? 32 * 4 : (J.kind == 5 ? 1 : 32);
        int nl = 0;
        for (int f = 0; f < nf; f++)
            if (!done[f]) active[nl++] = f;
        if (nl == 0) break;
        n_tasks = (nl + per - 1) / per;
        if ((int)tasks.size() < n_tasks) return 11;
        for (int i = 0; i < n_tasks; i++) tasks[i] = make_int4(0, i * per, std::min(per, nl - i * per), 0);
        int grid = n_tasks;
        if (J.grid_cap > 0) grid = std::min(grid, J.grid_cap);
        if (J.kind == 3) {
            SplitParams sp;
            // grid_cap < 0: -grid_cap CTAs share the tasks by iterations (hand-over flags); the emulator runs one CTA
            // at a time, the highest first, so the part of a task that must run first always has
            const bool share = J.grid_cap < 0;
            if (share) {
                grid = -J.grid_cap;
                share_flags.resize(std::max<size_t>(share_flags.size(), (size_t)n_tasks), 0);
            }
            sp.flags = share ? share_flags.data() : nullptr;
            sp.epoch = c + 1;
            sp.ctl = nullptr;
            sp.order = nullptr;
            sp.n_sm = grid / 2;
            if (share && grid % 2 == 0 && n_tasks <= grid) { // what compact_kernel prepares for the ranked assignment
                share_ctl.assign(SHARE_CTL_LEN, 0);
                share_order.resize(n_tasks);
                auto key = [&](int t) { // the task's least advanced fit
                    int k = 0x7fffffff;
                    for (int i = 0; i < tasks[t].z; i++) k = std::min(k, ne[active[tasks[t].y + i]]);
                    return k;
                };
                for (int t = 0; t < n_tasks; t++) {
                    int rank = 0;
                    const int mine = key(t);
                    for (int j = 0; j < n_tasks; j++) rank += (key(j) > mine) || (key(j) == mine && j < t);
                    share_order[rank] = t;
                }
                sp.ctl = share_ctl.data();
                sp.order = share_order.data();
            }
            sp.em = ep;
            sp.max_units = max_units;
            sp.max_uunits = max_uunits;
            sp.blob_smem = (int)blob_sm;
            sp.cost_u = UW * 22;
            sp.cost_m = MSEG * 168;
            const size_t smem = blob_sm + split_smem_bytes(PQ, NW, max_units, max_uunits);
            hostsim::launch(grid, NW * 32, smem, J.order, [&] { em_split_kernel<PQ, NW, 2, MSEG, UW>(sp); }, share);
        } else if (J.kind == 2) {
            constexpr int SEG = 8, W = 4;
            ep.max_seg = (T + SEG - 1) / SEG;
            ep.ckpt_smem_off = (int)blob_sm;
            ep.mode = 2;
            const size_t smem = blob_sm + (size_t)W * ep.max_seg * 64 * sizeof(double);
            hostsim::launch(grid, W * 32, smem, J.order, [&] { em_chunk_kernel<PQ, SEG, W, 2>(ep); });
        }
#ifdef LDSR_HAVE_WIDE
        else if (J.kind == 4) {
            const int rc = launch_wide_hostsim<PQ>(ep, S, J.y, blob_sm, grid, J.order);
            if (rc) return rc;
        }
#endif
#ifdef LDSR_HAVE_SCAN
        else if (J.kind == 5) {
            // 4 steps per thread (what plan_em chooses); orders >= 8 run the 2-steps-per-thread build
            const int L = (T <= 2 * 32 * SCAN_MAX_WARPS && J.order >= 8) ? 2 : 4;
            const int nwarps = (T + 32 * L - 1) / (32 * L);
            if (nwarps > SCAN_MAX_WARPS) return 14;
            if constexpr (PQ <= 4) {
                if (L == 2)
                    hostsim::launch(grid, nwarps * 32, 0, J.order, [&] { em_scan_kernel<PQ, 2>(ep); });
                else
                    hostsim::launch(grid, nwarps * 32, 0, J.order, [&] { em_scan_kernel<PQ, 4>(ep); });
            } else { // wide inputs: two steps per thread, v == u
                if (!S.same_uv || T > 2 * 32 * SCAN_MAX_WARPS) return 15;
                const int nw2 = (T + 63) / 64;
                hostsim::launch(grid, nw2 * 32, 0, J.order, [&] { em_scan_kernel<PQ, 2>(ep); });
            }
        }
#endif
        else
            return 12;
    }
#ifdef LDSR_HAVE_SCAN
    if (J.traj_out) { // the E-step once more, writing the trajectories: one job per fit
        if (J.kind != 5) return 16;
        std::vector<int> job_theta(nf);
        std::vector<long long> job_row(nf);
        for (int f = 0; f < nf; f++) {
            job_theta[f] = f;
            job_row[f] = (long long)f * T;
        }
        if (nf > 1) job_theta[nf - 1] = -1; // a group without a winner: NaN rows
        EmParams tp = ep;
        tp.n_jobs = nf;
        tp.job_group = f_group.data();
        tp.job_theta = job_theta.data();
        tp.job_row = job_row.data();
        tp.tX = J.traj_out;
        tp.tY = J.traj_out + (size_t)nf * T;
        tp.tV = J.traj_out + (size_t)2 * nf * T;
        tp.tJ = J.traj_out + (size_t)3 * nf * T;
        const int grid = J.grid_cap > 0 ? std::min(nf, J.grid_cap) : nf;
        if constexpr (PQ <= 4) {
            const int L = (T <= 2 * 32 * SCAN_MAX_WARPS && J.order >= 8) ? 2 : 4;
            const int nwarps = (T + 32 * L - 1) / (32 * L);
            if (L == 2)
                hostsim::launch(grid, nwarps * 32, 0, J.order, [&] { em_scan_kernel<PQ, 2, true>(tp); });
            else
                hostsim::launch(grid, nwarps * 32, 0, J.order, [&] { em_scan_kernel<PQ, 4, true>(tp); });
        } else {
            if (!S.same_uv || T > 2 * 32 * SCAN_MAX_WARPS) return 15;
            hostsim::launch(grid, ((T + 63) / 64) * 32, 0, J.order, [&] { em_scan_kernel<PQ, 2, true>(tp); });
        }
    }
#endif
    for (int f = 0; f < nf; f++) {
        unpad_theta<PQ>(&theta[(size_t)f * TL], p, q, J.u != nullptr, J.v != nullptr, J.theta_out + (size_t)f * stride);
        J.lik_out[f] = lik[f];
        J.iters_out[f] = ne[f];
    }
    return 0;
}

// The single-step kernels (aux_kernels.cuh) on one series: kind 0 = smoother_kernel, 1 = propagate_kernel, 2 =
// mstep_kernel.  One job per row of X, Y, V, J ([n_jobs][T]); the M-step reads X, V, J and writes theta_out.
struct StepJob {
    int kind, T, p, q, n_groups, n_jobs, stdlik, order;
    const double *y, *u, *v;
    const int *held_ptr, *held_idx, *job_group, *job_theta;
    const double *theta;
    double *X, *Y, *V, *J, *lik, *aux, *theta_out;
    int *status;
};

template <int PQ> int run_step(const StepJob &J) {
    constexpr int TL = 2 * PQ + 6;
    const int T = J.T, nj = J.n_jobs, stride = J.p + J.q + 6;
    Prep Pr;
    prepare<PQ>(T, J.p, J.q, J.y, J.u, J.v, J.n_groups, J.held_ptr, J.held_idx, Pr);
    std::vector<long long> job_row(nj);
    for (int j = 0; j < nj; j++) job_row[j] = (long long)j * T;
    std::vector<double> th((size_t)nj * TL, 0.0);
    const int block = 64, grid = (nj + block - 1) / block; // as kernels_inst.cu launches them
    if (J.kind == 2) {
        MstepParams mp;
        std::memset(&mp, 0, sizeof mp);
        mp.series = &Pr.S;
        mp.blobs = Pr.blob.data();
        mp.sconst = Pr.sconst.data();
        mp.g_series = Pr.g_series.data();
        mp.masks = Pr.masks.data();
        mp.g_mask_off = Pr.g_mask_off.data();
        mp.gconst = Pr.gconst.data();
        mp.g_status = Pr.g_status.data();
        mp.n_fits = nj;
        mp.f_group = J.job_group;
        mp.f_row = job_row.data();
        mp.X = J.X;
        mp.V = J.V;
        mp.J = J.J;
        mp.theta_out = th.data();
        mp.status = J.status;
        hostsim::launch(grid, block, 0, J.order, [&] { mstep_kernel<PQ>(mp); });
        for (int j = 0; j < nj; j++)
            unpad_theta<PQ>(&th[(size_t)j * TL], J.p, J.q, J.u != nullptr, J.v != nullptr, J.theta_out + (size_t)j * stride);
        return 0;
    }
    for (int j = 0; j < nj; j++)
        pad_theta<PQ>(J.theta + (size_t)j * stride, J.p, J.q, J.u != nullptr, J.v != nullptr, &th[(size_t)j * TL]);
    SmootherParams sp;
    std::memset(&sp, 0, sizeof sp);
    sp.series = &Pr.S;
    sp.blobs = Pr.blob.data();
    sp.g_series = Pr.g_series.data();
    sp.masks = Pr.masks.data();
    sp.g_mask_off = Pr.g_mask_off.data();
    sp.g_nobs = Pr.g_nobs.data();
    sp.n_jobs = nj;
    sp.job_group = J.job_group;
    sp.job_theta = J.job_theta;
    sp.job_row = job_row.data();
    sp.theta = th.data();
    sp.X = J.X;
    sp.Y = J.Y;
    sp.V = J.V;
    sp.J = J.J;
    sp.lik = J.lik;
    sp.stdlik = J.stdlik;
    sp.aux = J.aux;
    if (J.kind == 0)
        hostsim::launch(grid, block, 0, J.order, [&] { smoother_kernel<PQ>(sp); });
    else if (J.kind == 1)
        hostsim::launch(grid, block, 0, J.order, [&] { propagate_kernel<PQ>(sp); });
    else
        return 12;
    return 0;
}

// rep_kernel with caller noise z ([n_reps][1 + 2n]); what ldsr_rep_batch prepares (padded theta, u, v)
template <int PQ> int run_rep(int p, int q, const double *u, const double *v, int n, int n_reps, const double *z,
                              const double *theta, double mu, int exp_trans, int order, double *simX, double *simY,
                              double *simQ) {
    std::vector<double> th(2 * PQ + 6), up((size_t)n * PQ, 0.0), vp((size_t)n * PQ, 0.0);
    pad_theta<PQ>(theta, p, q, u != nullptr, v != nullptr, th.data());
    for (int t = 0; t < n; t++) {
        if (u)
            for (int j = 0; j < p; j++) up[(size_t)t * PQ + j] = u[(size_t)t * p + j];
        if (v)
            for (int j = 0; j < q; j++) vp[(size_t)t * PQ + j] = v[(size_t)t * q + j];
    }
    RepParams rp;
    std::memset(&rp, 0, sizeof rp);
    rp.theta = th.data();
    rp.u = up.data();
    rp.v = vp.data();
    rp.z = z;
    rp.n = n;
    rp.n_reps = n_reps;
    rp.mu = mu;
    rp.exp_trans = exp_trans;
    rp.simX = simX;
    rp.simY = simY;
    rp.simQ = simQ;
    const int per_cta = REP_WARPS * 32;
    hostsim::launch((n_reps + per_cta - 1) / per_cta, per_cta, rep_smem_bytes(z != nullptr), order,
                    [&] { rep_kernel<PQ>(rp); });
    return 0;
}

} // namespace

// kind: 2 = lane-per-fit kernel (MODE 2), 3 = time-split kernel, 4 = wide time-split kernel, 5 = scan kernel
// (one CTA per fit).
// One series; u, v are [T][p] / [T][q] (an R p x T matrix, column-major).  order: thread schedule of the
// emulator (0 forward, 1 reverse, >= 2 seeded shuffle).  grid_cap > 0 makes CTAs loop over tasks.
extern "C" int hostsim_em(int kind, int T, int p, int q, const double *y, const double *u, const double *v, int n_groups,
                          const int *held_ptr, const int *held_idx, int n_fits, const int *fit_group,
                          const double *theta0, int niter, double tol, int chunk, int order, int grid_cap,
                          double *theta_out, double *lik_out, int *iters_out) {
    Job J{kind, T, p, q, n_groups, n_fits, niter, chunk, order, grid_cap, y, u, v, held_ptr, held_idx, fit_group, theta0,
          tol, theta_out, lik_out, iters_out};
    const int need = std::max(u ? p : 1, v ? q : 1);
    if (need <= 3) return run<3>(J);
    if (need <= 10) return run<10>(J);
    return 13;
}

// hostsim_em for the scan kernel, followed by its trajectory mode on every fit's final theta (the last fit's job
// is marked "no winner"): traj_out is [4][n_fits][T] = X, Y, V, J.
extern "C" int hostsim_em_traj(int T, int p, int q, const double *y, const double *u, const double *v, int n_groups,
                               const int *held_ptr, const int *held_idx, int n_fits, const int *fit_group,
                               const double *theta0, int niter, double tol, int chunk, int order, int grid_cap,
                               double *theta_out, double *lik_out, int *iters_out, double *traj_out) {
    Job J{5, T, p, q, n_groups, n_fits, niter, chunk, order, grid_cap, y, u, v, held_ptr, held_idx, fit_group, theta0,
          tol, theta_out, lik_out, iters_out, traj_out};
    const int need = std::max(u ? p : 1, v ? q : 1);
    if (need <= 3) return run<3>(J);
    if (need <= 10) return run<10>(J);
    return 13;
}

// The single-step kernels, padded to width 3, 5 or 16 (steps per smoother block 8, 4, 1).  kind: 0 smoother, 1
// propagate, 2 M-step (see StepJob); theta is [n_jobs][p + q + 6]; job_theta[j] < 0 marks a job without theta
// (smoother only: NaN rows).
extern "C" int hostsim_step(int kind, int T, int p, int q, const double *y, const double *u, const double *v,
                            int n_groups, const int *held_ptr, const int *held_idx, int n_jobs, const int *job_group,
                            const int *job_theta, const double *theta, int stdlik, int order, double *X, double *Y,
                            double *V, double *J, double *lik, double *aux, double *theta_out, int *status) {
    StepJob sj{kind, T, p, q, n_groups, n_jobs, stdlik, order, y, u, v, held_ptr, held_idx, job_group, job_theta, theta,
               X, Y, V, J, lik, aux, theta_out, status};
    const int need = std::max(1, std::max(u ? p : 0, v ? q : 0));
    if (need <= 3) return run_step<3>(sj);
    if (need <= 5) return run_step<5>(sj);
    if (need <= 16) return run_step<16>(sj);
    return 13;
}

// rep_kernel in caller-noise mode; any of simX, simY, simQ may be NULL
extern "C" int hostsim_rep(int p, int q, const double *u, const double *v, int n, int n_reps, const double *z,
                           const double *theta, double mu, int exp_trans, int order, double *simX, double *simY,
                           double *simQ) {
    const int need = std::max(1, std::max(u ? p : 0, v ? q : 0));
    if (need <= 3) return run_rep<3>(p, q, u, v, n, n_reps, z, theta, mu, exp_trans, order, simX, simY, simQ);
    if (need <= 5) return run_rep<5>(p, q, u, v, n, n_reps, z, theta, mu, exp_trans, order, simX, simY, simQ);
    if (need <= 16) return run_rep<16>(p, q, u, v, n, n_reps, z, theta, mu, exp_trans, order, simX, simY, simQ);
    return 13;
}
