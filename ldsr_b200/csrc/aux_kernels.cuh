// aux_kernels.cuh -- set-up (hold-out masks, theta-independent Gram blocks), restart selection,
// and the single-step batched kernels (Kalman_smoother, Mstep, propagate, LDS_rep).
#pragma once
#include "lds_math.cuh"

namespace ldsr {

// ------------------------------------------------------------------------------------------
// Kalman_smoother for a list of jobs (EM.cpp:22-131), one lane per job, trajectories written to
// global rows (X,Y,V,J of length T each).  Used for the winners after EM and for
// ldsr_smoother_batch.  The filter pass parks Xu,Vu in the X,V rows; the backward pass then
// overwrites them in place.
// ------------------------------------------------------------------------------------------
struct SmootherParams {
    const SeriesDev *series;
    const double *blobs;
    const int *g_series;
    const unsigned *masks;
    const long long *g_mask_off;
    const int *g_nobs;
    int n_jobs;
    const int *job_group;     // [n_jobs]
    const int *job_theta;     // [n_jobs] row in theta (or -1: skip, rows become NaN)
    const long long *job_row; // [n_jobs] offset of the job's output rows, in doubles
    const double *theta;      // padded thetas
    double *X, *Y, *V, *J, *lik;
    int stdlik;
    // optional per-job scalar for the experimental learners' objectives (R/LDS_GA.R:28-44,136-147):
    // smoother: sum_t (X_{t+1} - A X_t - B u_t)^2 ; propagate: sum over observed t of (y_t - Y_t)^2
    double *aux;
};

// Input rows of a block of BK consecutive steps starting at t0, in registers (zeros past the end).
// Every lane of a warp reads the same addresses, so these are L1 broadcasts; issuing a block at a
// time, one block ahead of its use, keeps the L1/L2 latency out of the recursion.
template <int PQ, int BK>
__device__ __forceinline__ void load_rows(const double *__restrict__ rows, int t0, int T, double (&dst)[BK * PQ]) {
#pragma unroll
    for (int k = 0; k < BK; k++)
#pragma unroll
        for (int j = 0; j < PQ; j++) dst[k * PQ + j] = t0 + k >= 0 && t0 + k < T ? rows[(size_t)(t0 + k) * PQ + j] : 0.0;
}
template <int PQ> __device__ __forceinline__ double dot_regs(const double (&w)[PQ], const double *row) {
    double s = 0.0;
#pragma unroll
    for (int j = 0; j < PQ; j++) s = fma(w[j], row[j], s);
    return s;
}

// COEF: the forward pass alone, writing the backward-sampling coefficients of p(x_t | x_{t+1}, y_{0..t})
// instead of the smoothed rows (posterior_rep_kernel reads them): X <- m, Y <- o, V <- s, J <- J, with
// x_t = m_t + J_t x_{t+1} + s_t zeta_t, and o_t = y_t at observed steps, D v_t elsewhere.  J must be given.
template <int PQ, bool COEF = false> __global__ void smoother_kernel(const SmootherParams P) {
    const int job = blockIdx.x * blockDim.x + threadIdx.x;
    if (job >= P.n_jobs) return;
    const int grp = P.job_group[job];
    const SeriesDev S = P.series[P.g_series[grp]];
    const int T = S.T;
    const double *__restrict__ ys = P.blobs + S.blob_off + S.y_off;
    const double *__restrict__ us = P.blobs + S.blob_off + S.u_off;
    const double *__restrict__ vs = P.blobs + S.blob_off + S.v_off;
    const unsigned *__restrict__ mw = P.masks + P.g_mask_off[grp];
    // the four output rows of a job never overlap each other or the inputs
    double *__restrict__ X = P.X + P.job_row[job], *__restrict__ Y = P.Y + P.job_row[job],
                        *__restrict__ V = P.V + P.job_row[job],
                        *__restrict__ J = P.J ? P.J + P.job_row[job] : nullptr;
    if (P.job_theta[job] < 0) {
        const double nan = __longlong_as_double(0x7ff8000000000000ULL);
        for (int t = 0; t < T; t++) {
            X[t] = Y[t] = V[t] = nan;
            if (J) J[t] = nan;
        }
        if (P.lik) P.lik[job] = nan;
        return;
    }
    Theta<PQ> th;
    load_theta<PQ>(th, P.theta + (size_t)P.job_theta[job] * theta_pad_len<PQ>());
    const double A = th.A, A2 = th.A * th.A, Q = th.Q;
    // steps per block: about 24 input values in flight, always a divisor of the 32-step mask word
    constexpr int BK = PQ <= 3 ? 8 : (PQ <= 6 ? 4 : (PQ <= 12 ? 2 : 1));
    const bool same_uv = S.same_uv != 0;

    // ---- forward (EM.cpp:43-90); Xu, Vu are parked in the X, V rows
    double Xp = th.mu1, Vp = th.V1, acc = 0.0;
    {
        double ub[BK * PQ], un[BK * PQ];
        load_rows<PQ, BK>(us, 0, T, ub);
        for (int t0 = 0; t0 < T; t0 += BK) {
            load_rows<PQ, BK>(us, t0 + BK, T, un);
            const unsigned bits = mw[t0 >> 5] >> (t0 & 31);
#pragma unroll
            for (int k = 0; k < BK; k++) {
                const int t = t0 + k;
                if (t >= T) break;
                double Xu = Xp, Vu = Vp;
                const bool obs = (bits >> k) & 1u;
                if (obs) { // EM.cpp:61-68, 82-89
                    const double Dv = same_uv ? dot_regs<PQ>(th.D, &ub[k * PQ]) : dot_row<PQ>(th.D, vs + (size_t)t * PQ);
                    const double Sg = fma(th.C * Vp, th.C, th.R);
                    const double rS = 1.0 / Sg;
                    const double K = Vp * th.C * rS;
                    const double delta = ys[t] - fma(th.C, Xp, Dv);
                    Xu = fma(K, delta, Xp);
                    Vu = (1.0 - K * th.C) * Vp;
                    acc += delta * rS * delta + log(Sg);
                }
                const double Xn = fma(A, Xu, dot_regs<PQ>(th.B, &ub[k * PQ]));
                const double Vn = fma(A2, Vu, Q);
                if constexpr (COEF) {
                    // filtered form of the conditional variance, Vu Q / Vp_{t+1}: it equals V_t - J_t^2 V_{t+1}
                    // but cannot come out negative.  The last step has no successor: x ~ N(Xu, Vu).
                    const bool last = t == T - 1;
                    const double Jt = last ? 0.0 : Vu * A / Vn;
                    X[t] = last ? Xu : Xu - Jt * Xn;
                    V[t] = sqrt(last ? Vu : Vu * Q / Vn);
                    J[t] = Jt;
                    Y[t] = obs ? ys[t] : (same_uv ? dot_regs<PQ>(th.D, &ub[k * PQ]) : dot_row<PQ>(th.D, vs + (size_t)t * PQ));
                } else {
                    X[t] = Xu;
                    V[t] = Vu;
                }
                Xp = Xn;
                Vp = Vn;
            }
#pragma unroll
            for (int i = 0; i < BK * PQ; i++) ub[i] = un[i];
        }
    }
    if (P.lik) {
        const double n = (double)P.g_nobs[grp];
        double l = -0.5 * n * LOG_2PI - 0.5 * acc;
        P.lik[job] = P.stdlik ? l / n : l;
    }
    if constexpr (COEF) return;
    // ---- backward (EM.cpp:94-110)
    {
        const double VuT = V[T - 1];
        if (J) J[T - 1] = VuT * A * (1.0 / fma(A2, VuT, Q)); // EM.cpp:98
        Y[T - 1] = fma(th.C, X[T - 1], dot_row<PQ>(th.D, vs + (size_t)(T - 1) * PQ));
    }
    double Xs1 = X[T - 1], Vs1 = V[T - 1];
    double ssq = 0.0;
    // The filtered rows come back from L2 (several hundred cycles per access): they are read a
    // block at a time as well, one block ahead of the arithmetic.  Blocks are [lo, lo + BK), walked
    // downwards from the block that holds T - 2; step k of a block is lo + k.
    {
        double xb[BK], vb[BK], xn[BK], vn[BK], ub[BK * PQ], un[BK * PQ];
        int lo = ((T - 2) / BK) * BK;
#pragma unroll
        for (int k = 0; k < BK; k++) {
            xb[k] = lo + k <= T - 2 ? X[lo + k] : 0.0;
            vb[k] = lo + k <= T - 2 ? V[lo + k] : 0.0;
        }
        load_rows<PQ, BK>(us, lo, T, ub);
        for (; lo >= 0; lo -= BK) {
#pragma unroll
            for (int k = 0; k < BK; k++) {
                xn[k] = lo - BK + k >= 0 ? X[lo - BK + k] : 0.0;
                vn[k] = lo - BK + k >= 0 ? V[lo - BK + k] : 0.0;
            }
            load_rows<PQ, BK>(us, lo - BK, T, un);
#pragma unroll
            for (int k = BK - 1; k >= 0; k--) {
                const int t = lo + k;
                if (t > T - 2) continue;
                const double Xu = xb[k], Vu = vb[k];
                const double Bu = dot_regs<PQ>(th.B, &ub[k * PQ]);
                const double Xp1 = fma(A, Xu, Bu);
                const double Vp1 = fma(A2, Vu, Q);
                const double Jt = Vu * A * fast_rcp(Vp1); // off the loop-carried chain: overlaps across the block
                const double Xs = fma(Jt, Xs1 - Xp1, Xu);
                const double Vs = fma(Jt * (Vs1 - Vp1), Jt, Vu);
                X[t] = Xs;
                V[t] = Vs;
                if (J) J[t] = Jt;
                // v differs from u only for callers that pass two input sets: read in place then
                Y[t] = fma(th.C, Xs, same_uv ? dot_regs<PQ>(th.D, &ub[k * PQ]) : dot_row<PQ>(th.D, vs + (size_t)t * PQ));
                const double res = Xs1 - fma(A, Xs, Bu); // X_{t+1} - A X_t - B u_t   (R/LDS_GA.R:38)
                ssq = fma(res, res, ssq);
                Xs1 = Xs;
                Vs1 = Vs;
            }
#pragma unroll
            for (int k = 0; k < BK; k++) {
                xb[k] = xn[k];
                vb[k] = vn[k];
            }
#pragma unroll
            for (int i = 0; i < BK * PQ; i++) ub[i] = un[i];
        }
    }
    if (P.aux) P.aux[job] = ssq;
}

// ------------------------------------------------------------------------------------------
// Mstep (EM.cpp:139-229) from caller-supplied smoothed rows X,V,J: one lane per fit gathers the
// sums and calls the same mstep_from_stats the EM kernel uses.
// ------------------------------------------------------------------------------------------
struct MstepParams {
    const SeriesDev *series;
    const double *blobs;
    const double *sconst;
    const int *g_series;
    const unsigned *masks;
    const long long *g_mask_off;
    const double *gconst;
    const int *g_status;
    int n_fits;
    const int *f_group;
    const long long *f_row;
    const double *X, *V, *J;
    double *theta_out;
    int *status;
};

template <int PQ> __global__ void mstep_kernel(const MstepParams P) {
    const int f = blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= P.n_fits) return;
    const int grp = P.f_group[f];
    const SeriesDev S = P.series[P.g_series[grp]];
    const int T = S.T;
    const double *__restrict__ ys = P.blobs + S.blob_off + S.y_off;
    const double *__restrict__ us = P.blobs + S.blob_off + S.u_off;
    const double *__restrict__ vs = P.blobs + S.blob_off + S.v_off;
    const unsigned *__restrict__ mw = P.masks + P.g_mask_off[grp];
    const double *X = P.X + P.f_row[f], *V = P.V + P.f_row[f], *J = P.J + P.f_row[f];
    Stats<PQ> st;
    st.zero();
    for (int t = 0; t < T; t++) {
        const double Xs = X[t], Vs = V[t];
        if (t < T - 1) {
            st.Tx1x = fma(X[t + 1], Xs, st.Tx1x);
            st.Tx1xv = fma(V[t + 1], J[t], st.Tx1xv);
            st.Txx = fma(Xs, Xs, st.Txx);
            st.Txxv += Vs;
#pragma unroll
            for (int k = 0; k < PQ; k++) {
                st.Tx1u[k] = fma(X[t + 1], us[(size_t)t * PQ + k], st.Tx1u[k]);
                st.Tux[k] = fma(us[(size_t)t * PQ + k], Xs, st.Tux[k]);
            }
        }
        if ((mw[t >> 5] >> (t & 31)) & 1u) {
            st.Syx = fma(ys[t], Xs, st.Syx);
            st.Sxx = fma(Xs, Xs, st.Sxx);
            st.Sxxv += Vs;
#pragma unroll
            for (int k = 0; k < PQ; k++) st.Sxv[k] = fma(Xs, vs[(size_t)t * PQ + k], st.Sxv[k]);
        }
    }
    st.X0 = X[0];
    st.V0 = V[0];
    st.XT = X[T - 1];
    st.VT = V[T - 1];
    Theta<PQ> th;
    mstep_from_stats<PQ>(st, P.gconst + (size_t)grp * gconst_stride(PQ), P.sconst + S.sconst_off, T, th);
    store_theta<PQ>(th, P.theta_out + (size_t)f * theta_pad_len<PQ>());
    P.status[f] = P.g_status[grp];
}

// ------------------------------------------------------------------------------------------
// propagate (EM.cpp:295-356): open-loop prediction, one lane per job.
// ------------------------------------------------------------------------------------------
template <int PQ> __global__ void propagate_kernel(const SmootherParams P) {
    const int job = blockIdx.x * blockDim.x + threadIdx.x;
    if (job >= P.n_jobs) return;
    const int grp = P.job_group[job];
    const SeriesDev S = P.series[P.g_series[grp]];
    const int T = S.T;
    const double *__restrict__ ys = P.blobs + S.blob_off + S.y_off;
    const double *__restrict__ us = P.blobs + S.blob_off + S.u_off;
    const double *__restrict__ vs = P.blobs + S.blob_off + S.v_off;
    const unsigned *__restrict__ mw = P.masks + P.g_mask_off[grp];
    double *X = P.X + P.job_row[job], *Y = P.Y + P.job_row[job], *V = P.V + P.job_row[job];
    Theta<PQ> th;
    load_theta<PQ>(th, P.theta + (size_t)P.job_theta[job] * theta_pad_len<PQ>());
    const double A2 = th.A * th.A;
    double Xp = th.mu1, Vp = th.V1, acc = 0.0, ssq = 0.0;
    for (int t = 0; t < T; t++) {
        const double Yp = fma(th.C, Xp, dot_row<PQ>(th.D, vs + (size_t)t * PQ));
        X[t] = Xp;
        V[t] = Vp;
        Y[t] = Yp;
        if ((mw[t >> 5] >> (t & 31)) & 1u) {
            const double delta = ys[t] - Yp, Sg = fma(th.C * Vp, th.C, th.R);
            acc += delta / Sg * delta + log(Sg);
            ssq = fma(delta, delta, ssq); // ssqTrain (R/LDS_GA.R:143-147)
        }
        Xp = fma(th.A, Xp, dot_row<PQ>(th.B, us + (size_t)t * PQ));
        Vp = fma(A2, Vp, th.Q);
    }
    const double n = (double)P.g_nobs[grp];
    double l = -0.5 * n * LOG_2PI - 0.5 * acc;
    P.lik[job] = P.stdlik ? l / n : l;
    if (P.aux) P.aux[job] = ssq;
}

// ------------------------------------------------------------------------------------------
// LDS_rep (R/stochastics.R:18-63): one lane per replicate, one warp per 32 replicates, ONE pass for all
// requested outputs.  The noise is either read from z (n_reps x (1+2n), the reference's draw order) or
// generated from a counter-based generator (splitmix64 -> Box-Muller, both outputs of a pair used: the state
// and the observation draw of a step) keyed by (seed, replicate, step).
// Outputs are REPLICATE-MAJOR (the reference's rbindlist order) and every byte is written once: the warp
// simulates REP_TT steps into a [step][replicate] tile in shared memory (row stride 33: conflict-free both
// ways) and writes it out replicate by replicate, 128 contiguous bytes per half-warp; caller noise is read
// the same way (one instruction fetches the state draws and the observation draws of a replicate's tile).
// HBM traffic: 8 B per requested output and (replicate, step) + 16 B of noise when z is given.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long splitmix64(unsigned long long x) {
    x += 0x9E3779B97F4A7C15ULL;
    x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ULL;
    x = (x ^ (x >> 27)) * 0x94D049BB133111EBULL;
    return x ^ (x >> 31);
}
// two independent standard normals from counter (key, idx)
__device__ __forceinline__ void counter_normal_pair(unsigned long long key, unsigned long long idx, double &z0,
                                                    double &z1) {
    const unsigned long long a = splitmix64(key + 2 * idx), b = splitmix64(key + 2 * idx + 1);
    const double u1 = ((double)(a >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    const double u2 = ((double)(b >> 11) + 0.5) * (1.0 / 9007199254740992.0);
    double sn, cs;
    sincospi(2.0 * u2, &sn, &cs);
    const double r = sqrt(-2.0 * log(u1));
    z0 = r * cs;
    z1 = r * sn;
}
__device__ __forceinline__ unsigned long long counter_key(unsigned long long seed, unsigned long long rep) {
    return splitmix64(seed ^ splitmix64(rep * 0xD1342543DE82EF95ULL + 1));
}

constexpr int REP_TT = 16;     // steps per tile
constexpr int REP_WARPS = 4;   // warps per CTA
constexpr int REP_TILE = REP_TT * 33; // doubles per tile

struct RepParams {
    const double *theta; // padded, one model
    const double *u, *v; // [n][PQ] padded, time-major (zeros when absent)
    const double *z;     // optional noise [n_reps][1+2n], row 0 = replicate rep0
    unsigned long long seed;
    int n, n_reps;       // steps; replicates of THIS launch
    long long rep0;      // global index of the launch's first replicate (keys the generator)
    double mu;
    int exp_trans;
    double *simX, *simY, *simQ; // [n_reps][n] replicate-major, any may be null
};
__host__ __device__ inline size_t rep_smem_bytes(bool with_z) {
    return (size_t)REP_WARPS * (3 + (with_z ? 2 : 0)) * REP_TILE * sizeof(double);
}

template <int PQ> __global__ void __launch_bounds__(REP_WARPS * 32) rep_kernel(const RepParams P) {
    LDSR_DYN_SMEM(smem_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int n = P.n;
    const long long r0 = ((long long)blockIdx.x * REP_WARPS + warp) * 32; // first replicate of the warp
    if (r0 >= P.n_reps) return;
    const int n_rows = (int)(P.n_reps - r0 < 32 ? P.n_reps - r0 : 32);
    const bool have_z = P.z != nullptr;
    double *const tiles = reinterpret_cast<double *>(smem_raw) + (size_t)warp * (3 + (have_z ? 2 : 0)) * REP_TILE;
    double *const tX = tiles, *const tY = tiles + REP_TILE, *const tQ = tiles + 2 * REP_TILE;
    double *const tZq = tiles + 3 * REP_TILE, *const tZe = tiles + 4 * REP_TILE;
    Theta<PQ> th;
    load_theta<PQ>(th, P.theta);
    const double sQ = sqrt(th.Q), sR = sqrt(th.R), sV = sqrt(th.V1);
    const long long rep = r0 + lane; // my replicate (rows beyond n_rows compute garbage that is never stored)
    const size_t zstride = 1 + 2 * (size_t)n;
    const unsigned long long key = counter_key(P.seed, (unsigned long long)(P.rep0 + rep));
    double x;
    if (have_z) {
        x = (lane < n_rows ? P.z[(size_t)rep * zstride] : 0.0) * sV; // mean 0, not mu1 (stochastics.R:23)
    } else {
        double a, b;
        counter_normal_pair(key, 0, a, b);
        x = a * sV;
    }
    const int half = lane >> 4, hl = lane & 15; // half-warp and lane inside it
    for (int t0 = 0; t0 < n; t0 += REP_TT) {
        const int cnt = n - t0 < REP_TT ? n - t0 : REP_TT;
        if (have_z) { // state draws z[1 + t], observation draws z[1 + n + t]: lanes 0-15 / 16-31 of one instruction
            __syncwarp();
            for (int rr = 0; rr < n_rows; ++rr) {
                if (hl < cnt) {
                    const double val = P.z[(size_t)(r0 + rr) * zstride + 1 + (half ? n : 0) + t0 + hl];
                    (half ? tZe : tZq)[hl * 33 + rr] = val;
                }
            }
            __syncwarp();
        }
#pragma unroll 4
        for (int j = 0; j < cnt; ++j) { // only x chains from step to step: the draws of several steps overlap
            const int t = t0 + j;
            double zq, ze;
            if (have_z) {
                zq = tZq[j * 33 + lane];
                ze = tZe[j * 33 + lane];
            } else {
                counter_normal_pair(key, 1 + (unsigned long long)t, zq, ze);
            }
            const double y = fma(th.C, x, dot_row<PQ>(th.D, P.v + (size_t)t * PQ)) + ze * sR;
            tX[j * 33 + lane] = x;
            tY[j * 33 + lane] = y;
            tQ[j * 33 + lane] = P.exp_trans ? exp(y + P.mu) : y + P.mu;
            x = fma(th.A, x, dot_row<PQ>(th.B, P.u + (size_t)t * PQ)) + zq * sQ;
        }
        __syncwarp();
        // write the tile out: each half-warp one replicate row (up to 128 contiguous bytes) per instruction
        for (int rr = half; rr < n_rows; rr += 2) {
            if (hl < cnt) {
                const size_t o = (size_t)(r0 + rr) * n + t0 + hl;
                if (P.simX) P.simX[o] = tX[hl * 33 + rr];
                if (P.simY) P.simY[o] = tY[hl * 33 + rr];
                if (P.simQ) P.simQ[o] = tQ[hl * 33 + rr];
            }
        }
        __syncwarp();
    }
}

// ------------------------------------------------------------------------------------------
// Replicates conditioned on the observed record (forward filtering, backward sampling): draws of
// x_{0..T-1} from p(x | y, theta).  smoother_kernel's coefficient mode has written, per fit, the rows
// m, o, s, J; here one lane per replicate walks t = T-1 .. 0:
//     x_t = m_t + J_t x_{t+1} + s_t zeta_t                 (x_T = 0, J_{T-1} = 0)
//     y_t = o_t (the observation, bit for bit)              at observed steps
//     y_t = C x_t + o_t + sqrt(R) eps_t   (o_t = D v_t)    elsewhere
//     q_t = back-transform(y_t + mu): none / exp / inverse Box-Cox (construct_rec_kernel's)
// The warp layout is rep_kernel's: one warp per 32 replicates of ONE fit (fits of different T share a
// launch), outputs through [step][replicate] tiles of REP_TT steps written replicate-major, every
// byte once.  Tiles are aligned to REP_TT steps, so a tile's mask bits sit in one 32-bit word.
// Output order: fit f's replicate r starts at n_reps fit_ptr[f] + r T_f; caller noise z holds it at
// twice that offset, T_f state draws (zeta) then T_f observation draws (eps).  Without z, step t of
// (fit f, replicate r) takes the pair (zeta, eps) = counter_normal_pair(key(seed, f, r), t).
// The width of the inputs does not enter (D v is in o): one instantiation, compiled where it is
// launched (a template, so that the per-width units do not carry it).
// ------------------------------------------------------------------------------------------
struct PostRepParams {
    const double *m, *o, *s, *J;  // coefficient rows, fit f's T_f steps at fit_ptr[f]
    const long long *fit_ptr;     // [n_fits + 1]
    const double *par;            // [n_fits][4]: C, sqrt(R), mu, lambda
    const unsigned *masks;        // observed-step bits
    const long long *f_mask_off;  // [n_fits] the fit's group's first mask word
    const double *z;              // optional noise, indexed 2 (offset - out0)
    unsigned long long seed;
    int n_reps, wpf;              // replicates per fit, warps per fit
    long long blk0, n_blk;        // this launch's warps: (fit, 32 replicates) blocks blk0 .. blk0 + n_blk - 1
    long long out0;               // output offset of the launch's first element (outputs are written at - out0)
    int transform;                // 0 none, 1 log, 2 Box-Cox
    double *simX, *simY, *simQ;   // any may be null
};

__device__ __forceinline__ unsigned long long posterior_key(unsigned long long seed, int fit, long long rep) {
    return counter_key(counter_key(seed, (unsigned long long)fit), (unsigned long long)rep);
}

// shared memory per warp: the output tiles, the noise tiles (with z) and a [4][TT] coefficient tile
template <int TT> __host__ __device__ inline size_t posterior_smem_bytes(bool with_z) {
    return (size_t)REP_WARPS * ((3 + (with_z ? 2 : 0)) * TT * 33 + 4 * TT) * sizeof(double);
}

template <int TT> __global__ void __launch_bounds__(REP_WARPS * 32) posterior_rep_kernel(const PostRepParams P) {
    static_assert(32 % TT == 0 && TT <= 16, "a tile's mask bits sit in one word; a half-warp loads a tile row");
    LDSR_DYN_SMEM(smem_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long blk = (long long)blockIdx.x * REP_WARPS + warp;
    if (blk >= P.n_blk) return;
    const int f = (int)((P.blk0 + blk) / P.wpf);
    const int r0 = (int)((P.blk0 + blk) % P.wpf) * 32; // the warp's first replicate of fit f
    const int n_rows = P.n_reps - r0 < 32 ? P.n_reps - r0 : 32;
    const bool have_z = P.z != nullptr;
    constexpr int TILE = TT * 33;
    double *const tiles = reinterpret_cast<double *>(smem_raw) + (size_t)warp * ((3 + (have_z ? 2 : 0)) * TILE + 4 * TT);
    double *const tX = tiles, *const tY = tiles + TILE, *const tQ = tiles + 2 * TILE;
    double *const tZq = tiles + 3 * TILE, *const tZe = tiles + 4 * TILE;
    double *const tC = tiles + (3 + (have_z ? 2 : 0)) * TILE; // [m | s | o | J] of the tile's steps
    const long long fp = P.fit_ptr[f];
    const int T = (int)(P.fit_ptr[f + 1] - fp);
    const unsigned *__restrict__ mw = P.masks + P.f_mask_off[f];
    const double C = P.par[4 * f], sR = P.par[4 * f + 1], mu = P.par[4 * f + 2], lam = P.par[4 * f + 3];
    const double il = P.transform == 2 && lam != 0.0 ? 1.0 / lam : 0.0;
    const int tr = P.transform == 2 && lam == 0.0 ? 1 : P.transform;
    const long long base = (long long)P.n_reps * fp + (long long)r0 * T - P.out0; // row rr at base + rr T
    const unsigned long long key = posterior_key(P.seed, f, r0 + lane); // lanes >= n_rows: never stored
    const int half = lane >> 4, hl = lane & 15;
    // the coefficients of a tile: half-warp 0 loads m and o, half-warp 1 s and J (128 contiguous bytes each); the
    // next tile's are in flight while this one's chain runs, then read back from shared memory as broadcasts
    const double *__restrict__ ca = (half ? P.s : P.m) + fp, *__restrict__ cb = (half ? P.J : P.o) + fp;
    int lo = ((T - 1) / TT) * TT;
    double na = hl < T - lo ? ca[lo + hl] : 0.0, nb = hl < T - lo ? cb[lo + hl] : 0.0;
    double x1 = 0.0; // x_{t+1}
    for (; lo >= 0; lo -= TT) {
        const int cnt = T - lo < TT ? T - lo : TT;
        tC[half * TT + hl] = na;
        tC[(2 + half) * TT + hl] = nb;
        if (lo > 0) {
            na = ca[lo - TT + hl];
            nb = cb[lo - TT + hl];
        }
        const unsigned bits = mw[lo >> 5] >> (lo & 31);
        if (have_z) { // state draws at 2 row + t, observation draws at 2 row + T + t: lanes 0-15 / 16-31
            for (int rr = 0; rr < n_rows; ++rr) {
                if (hl < cnt) {
                    const double val = P.z[2 * (base + (long long)rr * T) + (half ? T : 0) + lo + hl];
                    (half ? tZe : tZq)[hl * 33 + rr] = val;
                }
            }
        }
        __syncwarp();
#pragma unroll 4
        for (int j = cnt - 1; j >= 0; j--) { // only x chains from step to step: the draws of several steps overlap
            double zq, ze;
            if (have_z) {
                zq = tZq[j * 33 + lane];
                ze = tZe[j * 33 + lane];
            } else {
                counter_normal_pair(key, (unsigned long long)(lo + j), zq, ze);
            }
            const double x = fma(tC[TT + j], zq, fma(tC[3 * TT + j], x1, tC[j]));
            const double y = (bits >> j) & 1u ? tC[2 * TT + j] : fma(sR, ze, fma(C, x, tC[2 * TT + j]));
            const double yq = y + mu;
            tX[j * 33 + lane] = x;
            tY[j * 33 + lane] = y;
            tQ[j * 33 + lane] = tr == 1 ? exp(yq) : (tr == 0 ? yq : pow(fma(yq, lam, 1.0), il));
            x1 = x;
        }
        __syncwarp();
        // each half-warp writes one replicate row of the tile (up to 128 contiguous bytes) per instruction
        for (int rr = half; rr < n_rows; rr += 2) {
            if (hl < cnt) {
                const long long off = base + (long long)rr * T + lo + hl;
                if (P.simX) P.simX[off] = tX[hl * 33 + rr];
                if (P.simY) P.simY[off] = tY[hl * 33 + rr];
                if (P.simQ) P.simQ[off] = tQ[hl * 33 + rr];
            }
        }
        __syncwarp();
    }
}

} // namespace ldsr
