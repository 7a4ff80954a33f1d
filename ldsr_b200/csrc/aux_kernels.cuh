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
constexpr int POST_MAX_WIN = 4;   // windows per statistics call (LDSR_STATS_MAX_WINDOWS)
constexpr int POST_MAX_RING = 64; // longest window (LDSR_STATS_MAX_WINDOW): the Q ring covers the last 64 steps

// Quantile mode (ldsr_posterior_quantile_batch): exact order statistics over replicates by radix selection on
// order-preserving 64-bit keys, one sampler pass per round.  A slot is (window k, row fit_ptr[f] + t), at
// k n_steps + fit_ptr[f] + t.  Each level of a slot keeps a bracket [lo, hi] of keys that holds its rank; the
// distinct brackets of a pass are histogrammed (more than `cap` values) or collected (at most `cap`).
constexpr int QUANT_MAX_LEV = 8;      // LDSR_QUANT_MAX_LEVELS
constexpr int QUANT_MAX_CAP = 2048;   // values a collected bracket may hold (shared-memory sort)
constexpr int QUANT_THREADS = 256;    // threads of the bracket kernel
constexpr int QUANT_RANGE = 0, QUANT_SELECT = 1; // PostRepParams::qpass
constexpr int QL_ACTIVE = 0, QL_DONE = 1, QL_NONE = 2; // QuantLevel::state (QL_NONE: no value, the output is NaN)
struct QuantBracket {
    unsigned long long lo, hi; // the keys it covers, both included
    long long base;            // its first bin (histogram) or first segment entry (collected)
    long long slot;
    int count;                 // values in [lo, hi], from the previous pass
    int shift;                 // histogram: bin = (key - lo) >> shift; -1: collected
    int cursor;                // collected: values appended so far (the self-check compares it with count)
};
struct QuantLevel {
    unsigned long long lo, hi, key; // the bracket that holds the rank; key: the answer once QL_DONE
    int rank, below, count, state;  // rank among the slot's values (1-based), values below lo, values in [lo, hi]
};
// order-preserving map of a double onto an unsigned key (-0 below +0, NaN never occurs: windows with a non-finite
// flow have no value) and back
__device__ __forceinline__ unsigned long long quant_key(double v) {
    const unsigned long long b = (unsigned long long)__double_as_longlong(v);
    return b ^ (b >> 63 ? ~0ull : 1ull << 63);
}
__device__ __forceinline__ double quant_value(unsigned long long k) {
    return __longlong_as_double((long long)(k ^ (k >> 63 ? 1ull << 63 : ~0ull)));
}

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
    // statistics mode (posterior_rep_kernel<TT, true>, one launch, blk0 = out0 = 0): per (fit, replicate) row
    // n_reps f + r, window k's outputs at k n_rows + row; any output may be null
    int n_win, win[POST_MAX_WIN]; // moving-mean window lengths, 1 .. POST_MAX_RING
    int ring;                     // Q ring slots per lane: a power of two >= every window (0 without windows)
    long long n_rows;             // n_fits n_reps
    const int *range;             // [n_fits][2]: the statistics range [lo, hi) of steps
    const double *thr;            // [n_fits] run threshold on the Q scale, or null (no run statistics)
    double *wmin, *wmax, *deficit;
    int *wmin_at, *wmax_at, *run_len, *run_at, *deficit_at, *n_runs;
    // yearly mode (posterior_rep_kernel<TT, POST_YEARLY>, one launch, blk0 = out0 = 0; win, n_win, ring, range and
    // thr as above, thr required): counts of replicates added at row fit_ptr[f] + t, length / window k's at
    // k n_steps + fit_ptr[f] + t; any output may be null
    int n_len, len[POST_MAX_WIN]; // run lengths L_k, 1 .. POST_MAX_RING
    int delay;                    // D = max L_k: step s is decided when the walk reaches s - D + 1 (0 without lengths)
    long long n_steps;            // fit_ptr[n_fits]
    int *y_below, *y_in_run, *y_wbelow, *y_nonfinite;
    // quantile mode (posterior_rep_kernel<TT, POST_QUANT>, one launch per pass, blk0 = out0 = 0; win, n_win, ring,
    // range and n_steps as above, n_win >= 1).  QUANT_RANGE adds, per slot, the values (q_n, which starts at 0 where
    // the slot has values and at -1 elsewhere) and their smallest and largest key.  QUANT_SELECT adds each value to
    // the histogram or the segment of the bracket of its slot that covers it, if any.
    int qpass, n_lev;
    int *q_n;
    unsigned long long *q_min, *q_max;
    const int *q_slot_nbr, *q_slot_br; // the slot's brackets: q_slot_br[slot n_lev + m], m < q_slot_nbr[slot]
    QuantBracket *q_br;
    unsigned *q_hist;
    unsigned long long *q_seg;
};

__device__ __forceinline__ unsigned long long posterior_key(unsigned long long seed, int fit, long long rep) {
    return counter_key(counter_key(seed, (unsigned long long)fit), (unsigned long long)rep);
}

// shared memory per warp: the output tiles, the noise tiles (with z) and a [4][TT] coefficient tile
template <int TT> __host__ __device__ inline size_t posterior_smem_bytes(bool with_z) {
    return (size_t)REP_WARPS * ((3 + (with_z ? 2 : 0)) * TT * 33 + 4 * TT) * sizeof(double);
}
// statistics and yearly modes: no output tiles; the noise tiles (with z), the coefficient tile and the lanes' Q rings
template <int TT> __host__ __device__ inline size_t posterior_stats_smem_bytes(bool with_z, int ring) {
    return (size_t)REP_WARPS * ((with_z ? 2 : 0) * TT * 33 + 4 * TT + 32 * ring) * sizeof(double);
}

// The modes of posterior_rep_kernel.  POST_STATS is 1, so the statistics mode may also be named <TT, true>.
constexpr int POST_TRAJ = 0, POST_STATS = 1, POST_YEARLY = 2, POST_QUANT = 3;

// The quantile mode's selection pass: the value's key into the one bracket of its slot that covers it (brackets of
// a slot are disjoint), as a bin count or a segment entry.  A collected bracket never takes more than its count;
// the cursor still counts, so that the self-check sees any difference between passes.
__device__ __forceinline__ void quant_select(const PostRepParams &P, long long slot, unsigned long long key) {
    const int nb = P.q_slot_nbr[slot];
    for (int m = 0; m < nb; m++) {
        QuantBracket &B = P.q_br[P.q_slot_br[slot * P.n_lev + m]];
        if (key < B.lo || key > B.hi) continue;
        if (B.shift >= 0) {
            atomicAdd(P.q_hist + B.base + (long long)((key - B.lo) >> B.shift), 1u);
        } else {
            const int pos = atomicAdd(&B.cursor, 1);
            if (pos < B.count) P.q_seg[B.base + pos] = key;
        }
        return;
    }
}

// POST_TRAJ: the trajectories (simX, simY, simQ).  POST_STATS: the same draws, reduced in the walk to each
// replicate's drought statistics over its fit's range [lo, hi) (ldsr_posterior_stats_batch).  POST_YEARLY: the
// same draws, reduced across replicates to per-step counts (ldsr_posterior_yearly_batch).  POST_QUANT: the same
// draws, one pass of the quantile selection (ldsr_posterior_quantile_batch; the pass is P.qpass, so that every pass
// runs the same code and computes the same values).  In the reducing modes no trajectory leaves the SM.  All modes
// run the one step body below, so a replicate's Q_t is the same value in each.
// The statistics mode's accumulators take it to 168 registers: three CTAs an SM, stated so that ptxas does not cap
// it at 128 and spill (0 leaves the other modes to ptxas's default: 96 registers for the trajectories).  The
// quantile mode would spill at 128 too and is bounded the same way.
template <int TT, int MODE = POST_TRAJ>
__global__ void __launch_bounds__(REP_WARPS * 32, MODE == POST_STATS || MODE == POST_QUANT ? 3 : 0)
    posterior_rep_kernel(const PostRepParams P) {
    static_assert(32 % TT == 0 && TT <= 16, "a tile's mask bits sit in one word; a half-warp loads a tile row");
    constexpr bool STATS = MODE == POST_STATS, YEARLY = MODE == POST_YEARLY, QUANT = MODE == POST_QUANT,
                   REDUCE = STATS || YEARLY || QUANT;
    LDSR_DYN_SMEM(smem_raw);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const long long blk = (long long)blockIdx.x * REP_WARPS + warp;
    if (blk >= P.n_blk) return;
    const int f = (int)((P.blk0 + blk) / P.wpf);
    const int r0 = (int)((P.blk0 + blk) % P.wpf) * 32; // the warp's first replicate of fit f
    const int n_rows = P.n_reps - r0 < 32 ? P.n_reps - r0 : 32;
    const bool have_z = P.z != nullptr;
    constexpr int TILE = TT * 33;
    constexpr int N_OUT = REDUCE ? 0 : 3; // output tiles
    double *const tiles = reinterpret_cast<double *>(smem_raw) +
                          (size_t)warp * ((N_OUT + (have_z ? 2 : 0)) * TILE + 4 * TT + (REDUCE ? 32 * P.ring : 0));
    double *const tX = tiles, *const tY = tiles + TILE, *const tQ = tiles + 2 * TILE;
    double *const tZq = tiles + N_OUT * TILE, *const tZe = tiles + (N_OUT + 1) * TILE;
    double *const tC = tiles + (N_OUT + (have_z ? 2 : 0)) * TILE; // [m | s | o | J] of the tile's steps
    const long long fp = P.fit_ptr[f];
    const int T = (int)(P.fit_ptr[f + 1] - fp);
    const unsigned *__restrict__ mw = P.masks + P.f_mask_off[f];
    const double C = P.par[4 * f], sR = P.par[4 * f + 1], mu = P.par[4 * f + 2], lam = P.par[4 * f + 3];
    const double il = P.transform == 2 && lam != 0.0 ? 1.0 / lam : 0.0;
    const int tr = P.transform == 2 && lam == 0.0 ? 1 : P.transform;
    const long long base = (long long)P.n_reps * fp + (long long)r0 * T - P.out0; // row rr at base + rr T
    const unsigned long long key = posterior_key(P.seed, f, r0 + lane); // lanes >= n_rows: never stored
    const int half = lane >> 4, hl = lane & 15;
    // statistics state, one replicate per lane.  The walk runs downwards, so at step t the window starting at t is
    // complete: its sum gains Q_t and loses Q_{t+w}, read from the lane's ring (slot (t mod ring) of column `lane`)
    // before Q_t takes that slot.  Updating on <= / >= lets the smaller start, and the earlier run, win ties.
    double *const ring = tC + 4 * TT + lane;
    const int rmask = P.ring - 1;
    const int rlo = REDUCE ? P.range[2 * f] : 0, rhi = REDUCE ? P.range[2 * f + 1] : 0;
    const bool runs = STATS && P.thr != nullptr;
    const double thr = runs || YEARLY ? P.thr[f] : 0.0;
    double wsum[POST_MAX_WIN], wmn[POST_MAX_WIN], wmx[POST_MAX_WIN];
    int wmn_at[POST_MAX_WIN], wmx_at[POST_MAX_WIN];
#pragma unroll
    for (int k = 0; k < POST_MAX_WIN; k++) {
        wsum[k] = 0.0;
        wmn[k] = INFINITY;
        wmx[k] = -INFINITY;
        wmn_at[k] = wmx_at[k] = -1;
    }
    int cur_len = 0, best_len = 0, best_len_at = -1, best_def_at = -1, n_runs = 0;
    double cur_def = 0.0, best_def = 0.0;
    bool finite = true;
    auto close_run = [&](int first) {
        n_runs++;
        if (cur_len >= best_len) best_len = cur_len, best_len_at = first;
        if (cur_def >= best_def) best_def = cur_def, best_def_at = first;
        cur_len = 0;
        cur_def = 0.0;
    };
    // yearly state.  Bit i of `below` / `bad` is whether Q_{t+i} < thr / Q_{t+i} is not finite, for the last 64
    // steps walked (steps at or above hi: neither).  A count of the replicates is kept per step, by lane j for
    // step j of the tile (ballot and popc), and added to the output once a tile by the lanes that hold one.
    // A run's length is known only when it closes, so in_run decides step s with a delay: when the walk reaches
    // t = s - D + 1, down(s) = the consecutive below steps from s downwards, capped at D, is in bits D-1 .. 0 of
    // `below`, and `up` = the consecutive below steps from s upwards.  s lies in a run of length >= L
    // iff below(s) and up + down - 1 >= L; the caps are exact because every L <= D.
    const bool live = lane < n_rows;
    const int D = YEARLY ? P.delay : 1; // (1: the other modes never decide a step)
    unsigned long long below = 0ull, bad = 0ull;
    int up = 0, c_below = 0, c_bad = 0, c_win[POST_MAX_WIN] = {}, c_run[POST_MAX_WIN] = {};
    unsigned long long k_min[POST_MAX_WIN], k_max[POST_MAX_WIN]; // quantile range pass: step j's keys, by lane j
    auto count = [&](int &c, bool pred, int j) { // c of lane j <- the live replicates with pred
        const int n = __popc(__ballot_sync(0xffffffffu, live && pred));
        if (lane == j) c = n;
    };
    auto add = [&](int *out, long long row, int &c) { // the lane's count into out[row]
        if (out && c) atomicAdd(out + row, c);
        c = 0;
    };
    auto decide = [&](int s, int j) { // step s, now that the walk is at s - D + 1 (or below lo)
        const bool b = (below >> (D - 1)) & 1ull;
        up = b ? up + 1 : 0;
        const unsigned long long top = below << (64 - D); // step s in bit 63
        const unsigned nh = ~(unsigned)(top >> 32), nl = ~(unsigned)top;
        const int len = up + (nh ? __clz((int)nh) : 32 + __clz((int)nl)) - 1; // up + down(s) - 1
#pragma unroll
        for (int k = 0; k < POST_MAX_WIN; k++) {
            if (k >= P.n_len) break;
            count(c_run[k], s < rhi && b && len >= P.len[k], j);
        }
    };
    // the coefficients of a tile: half-warp 0 loads m and o, half-warp 1 s and J (128 contiguous bytes each); the
    // next tile's are in flight while this one's chain runs, then read back from shared memory as broadcasts
    const double *__restrict__ ca = (half ? P.s : P.m) + fp, *__restrict__ cb = (half ? P.J : P.o) + fp;
    int lo = ((T - 1) / TT) * TT;
    double na = hl < T - lo ? ca[lo + hl] : 0.0, nb = hl < T - lo ? cb[lo + hl] : 0.0;
    double x1 = 0.0; // x_{t+1}
    for (; lo >= 0 && (!REDUCE || lo + TT > rlo); lo -= TT) { // statistics, yearly: no tile below the range
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
            const double q = tr == 1 ? exp(yq) : (tr == 0 ? yq : pow(fma(yq, lam, 1.0), il));
            if (!REDUCE) {
                tX[j * 33 + lane] = x;
                tY[j * 33 + lane] = y;
                tQ[j * 33 + lane] = q;
            }
            x1 = x;
            if (!REDUCE) continue;
            const int t = lo + j;
            if (t < rlo || t >= rhi) continue;
            finite = finite && fabs(q) < INFINITY; // false for NaN and +-Inf
            const int seen = rhi - t; // steps of the range walked so far, t included
            if constexpr (YEARLY) {
                const bool fin = fabs(q) < INFINITY;
                below = below << 1 | (unsigned long long)(q < thr); // NaN: not below
                bad = bad << 1 | (unsigned long long)!fin;
                count(c_below, q < thr, j);
                count(c_bad, !fin, j);
                // window sums of finite flows only; a window with a non-finite flow (a bit of `bad`) counts nowhere
                const double qf = fin ? q : 0.0;
#pragma unroll
                for (int k = 0; k < POST_MAX_WIN; k++) {
                    if (k >= P.n_win) break;
                    const int w = P.win[k];
                    double sum = wsum[k] + qf;
                    if (seen > w) sum -= ring[((t + w) & rmask) * 32];
                    wsum[k] = sum;
                    count(c_win[k], seen >= w && !(bad & (~0ull >> (64 - w))) && sum < w * thr, j);
                }
                if (P.n_win > 0) ring[(t & rmask) * 32] = qf;
                if (D > 0) decide(t + D - 1, j);
            } else if constexpr (QUANT) {
                // the yearly mode's window sums; the value of a window is its sum over w, as a key
                const bool fin = fabs(q) < INFINITY;
                bad = bad << 1 | (unsigned long long)!fin;
                const double qf = fin ? q : 0.0;
#pragma unroll
                for (int k = 0; k < POST_MAX_WIN; k++) {
                    if (k >= P.n_win) break;
                    const int w = P.win[k];
                    double sum = wsum[k] + qf;
                    if (seen > w) sum -= ring[((t + w) & rmask) * 32];
                    wsum[k] = sum;
                    const bool has = live && seen >= w && !(bad & (~0ull >> (64 - w)));
                    const unsigned long long key = quant_key(sum / (double)w);
                    if (P.qpass == QUANT_RANGE) { // lane j <- step j's count and smallest and largest key
                        count(c_win[k], has, j);
                        unsigned long long mn = has ? key : ~0ull, mx = has ? key : 0ull;
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            const unsigned long long a = __shfl_xor_sync(0xffffffffu, mn, o),
                                                     b = __shfl_xor_sync(0xffffffffu, mx, o);
                            mn = a < mn ? a : mn;
                            mx = b > mx ? b : mx;
                        }
                        if (lane == j) k_min[k] = mn, k_max[k] = mx;
                    } else if (has) {
                        quant_select(P, k * P.n_steps + fp + t, key);
                    }
                }
                ring[(t & rmask) * 32] = qf;
            } else {
#pragma unroll
                for (int k = 0; k < POST_MAX_WIN; k++) {
                    if (k >= P.n_win) break;
                    const int w = P.win[k];
                    double sum = wsum[k] + q;
                    if (seen > w) sum -= ring[((t + w) & rmask) * 32]; // Q_{t+w} leaves the window
                    wsum[k] = sum;
                    if (seen >= w) {
                        if (sum <= wmn[k]) wmn[k] = sum, wmn_at[k] = t;
                        if (sum >= wmx[k]) wmx[k] = sum, wmx_at[k] = t;
                    }
                }
                if (P.n_win > 0) ring[(t & rmask) * 32] = q;
                if (runs) {
                    if (q < thr) {
                        cur_len++;
                        cur_def += thr - q;
                    } else if (cur_len > 0) {
                        close_run(t + 1);
                    }
                }
            }
        }
        if constexpr (YEARLY) { // lane j < TT holds step lo + j's counts, and in_run's of step lo + j + D - 1
            const long long row = fp + lo + lane;
            add(P.y_below, row, c_below);
            add(P.y_nonfinite, row, c_bad);
#pragma unroll
            for (int k = 0; k < POST_MAX_WIN; k++) {
                if (k < P.n_win) add(P.y_wbelow, k * P.n_steps + row, c_win[k]);
                if (k < P.n_len) add(P.y_in_run, k * P.n_steps + row + D - 1, c_run[k]);
            }
        }
        if constexpr (QUANT) { // lane j < TT holds step lo + j's count and keys
            if (P.qpass == QUANT_RANGE) {
#pragma unroll
                for (int k = 0; k < POST_MAX_WIN; k++) {
                    if (k >= P.n_win) break;
                    if (c_win[k]) {
                        const long long i = k * P.n_steps + fp + lo + lane;
                        atomicAdd(P.q_n + i, c_win[k]);
                        atomicMin(P.q_min + i, k_min[k]);
                        atomicMax(P.q_max + i, k_max[k]);
                        c_win[k] = 0;
                    }
                }
            }
        }
        if (!REDUCE) {
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
        }
        __syncwarp();
    }
    if constexpr (YEARLY) {
        // the steps lo - 1 .. lo - D + 1 are not below: this decides lo + D - 2 .. lo, one step at a time (lane 0
        // holds and adds the counts), and clips runs at lo
        for (int s = rlo + D - 2; s >= rlo; s--) {
            below <<= 1;
            decide(s, 0);
#pragma unroll
            for (int k = 0; k < POST_MAX_WIN; k++)
                if (k < P.n_len) add(P.y_in_run, k * P.n_steps + fp + s, c_run[k]);
        }
        return;
    }
    if (!STATS || lane >= n_rows) return;
    if (cur_len > 0) close_run(rlo); // a run reaching the range's lower end
    // one row per lane: consecutive rows across the warp
    const long long row = (long long)P.n_reps * f + r0 + lane;
#pragma unroll
    for (int k = 0; k < POST_MAX_WIN; k++) {
        if (k >= P.n_win) break;
        const double w = P.win[k];
        const bool ok = finite && wmn_at[k] >= 0;
        const long long o = k * P.n_rows + row;
        if (P.wmin) P.wmin[o] = ok ? wmn[k] / w : NAN;
        if (P.wmin_at) P.wmin_at[o] = ok ? wmn_at[k] : -1;
        if (P.wmax) P.wmax[o] = ok ? wmx[k] / w : NAN;
        if (P.wmax_at) P.wmax_at[o] = ok ? wmx_at[k] : -1;
    }
    if (!runs) return;
    if (P.run_len) P.run_len[row] = finite ? best_len : -1;
    if (P.run_at) P.run_at[row] = finite ? best_len_at : -1;
    if (P.deficit) P.deficit[row] = finite ? best_def : NAN;
    if (P.deficit_at) P.deficit_at[row] = finite ? best_def_at : -1;
    if (P.n_runs) P.n_runs[row] = finite ? n_runs : -1;
}

// ---- the quantile selection between the sampler's passes (ldsr_posterior_quantile_batch) ---------------------
// quant_init_kernel (after the range pass) gives every level its rank and first bracket, [min, max] of its slot.
// Then, until no level is active: quant_plan_kernel makes one bracket of each distinct active bracket, the sampler
// runs its selection pass, and quant_bracket_kernel moves each level into the bin that holds its rank (histogram)
// or picks it from the sorted segment (collected).  quant_out_kernel writes the outputs.  Each is a template of no
// parameter, so that it is compiled where it is launched and not in every per-width unit.
struct QuantParams {
    long long n_slots, n_steps; // slots: n_windows n_steps
    int n_lev, nb_log2, cap, n_reps; // levels; log2 of the bins of a histogram; most values of a collected bracket
    double lev[QUANT_MAX_LEV];
    const int *n;               // [n_slots] the values of the slot (-1: a slot without values)
    const unsigned long long *kmin, *kmax;
    QuantLevel *lv;             // [n_slots][n_lev]
    QuantBracket *br;           // up to n_slots n_lev
    int *slot_nbr, *slot_br;    // the slot's brackets (PostRepParams::q_slot_nbr, q_slot_br)
    // [0] brackets, [1] histograms, [2] segment entries of the pass; [3] the lowest slot whose passes disagreed
    // (~0: none)
    unsigned long long *ctr;
    const unsigned *hist;
    const unsigned long long *seg;
    long long n_br;             // brackets of the pass
    double *q;                  // [n_windows][n_lev][n_steps]
    int *nonfinite;             // [n_windows][n_steps]
};

// one thread per slot: rank max(1, ceil(p n)) in IEEE double; the minimum, the maximum and a slot of one key are
// answered at once
template <int = 0> __global__ void quant_init_kernel(const QuantParams Q) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q.n_slots) return;
    const int n = Q.n[i];
    const unsigned long long lo = Q.kmin[i], hi = Q.kmax[i];
    for (int l = 0; l < Q.n_lev; l++) {
        QuantLevel L;
        L.lo = lo;
        L.hi = hi;
        L.key = 0ull;
        L.below = 0;
        L.count = n;
        L.rank = 0;
        L.state = QL_NONE;
        if (n > 0) {
            const long long r = (long long)ceil(Q.lev[l] * (double)n);
            L.rank = r < 1 ? 1 : (int)r;
            L.state = QL_ACTIVE;
            if (lo == hi || L.rank == 1) L.state = QL_DONE, L.key = lo;
            else if (L.rank == n) L.state = QL_DONE, L.key = hi;
        }
        Q.lv[i * Q.n_lev + l] = L;
    }
}

// one thread per slot: a bracket for each distinct bracket of its active levels (the levels of one bracket are
// adjacent, their ranks being ordered); histogram bins of 2^shift keys, the least shift that fits the span
template <int = 0> __global__ void quant_plan_kernel(const QuantParams Q) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q.n_slots) return;
    int nbr = 0;
    unsigned long long plo = 0ull, phi = 0ull;
    for (int l = 0; l < Q.n_lev; l++) {
        const QuantLevel &L = Q.lv[i * Q.n_lev + l];
        if (L.state != QL_ACTIVE || (nbr > 0 && L.lo == plo && L.hi == phi)) continue;
        plo = L.lo;
        phi = L.hi;
        const long long id = (long long)atomicAdd(Q.ctr, 1ull);
        QuantBracket B;
        B.lo = L.lo;
        B.hi = L.hi;
        B.slot = i;
        B.count = L.count;
        B.cursor = 0;
        if (L.count <= Q.cap) {
            B.shift = -1;
            B.base = (long long)atomicAdd(Q.ctr + 2, (unsigned long long)L.count);
        } else {
            int s = 0;
            while (((L.hi - L.lo) >> s) >> Q.nb_log2) s++;
            B.shift = s;
            B.base = (long long)atomicAdd(Q.ctr + 1, 1ull) << Q.nb_log2;
        }
        Q.br[id] = B;
        Q.slot_br[i * Q.n_lev + nbr++] = (int)id;
    }
    Q.slot_nbr[i] = nbr;
}

// Bracket bi of the pass, by a CTA of QUANT_THREADS.  Its levels are the slot's active levels with its bounds.
// Histogram: an exclusive scan of the bins; the thread whose bins hold a level's rank moves the level into that bin
// (a bin of one key answers it).  Collected: the segment, sorted (bitonic, in shared memory), gives each level's
// rank.  Either way the values the pass found must be the bracket's count, else the slot is reported.
__device__ __forceinline__ void quant_bracket(const QuantParams &Q, long long bi) {
    LDSR_STATIC_SMEM(unsigned long long, keys[QUANT_MAX_CAP]);
    LDSR_STATIC_SMEM(int, want[QUANT_MAX_LEV]);
    LDSR_STATIC_SMEM(int, part[QUANT_THREADS / 32]);
    const QuantBracket B = Q.br[bi];
    const int tid = threadIdx.x;
    QuantLevel *const lv = Q.lv + B.slot * Q.n_lev;
    if (tid < QUANT_MAX_LEV) { // the rank inside the bracket of each of its levels, 0 for the others
        want[tid] = 0;
        if (tid < Q.n_lev) {
            const QuantLevel L = lv[tid];
            if (L.state == QL_ACTIVE && L.lo == B.lo && L.hi == B.hi) want[tid] = L.rank - L.below;
        }
    }
    if (B.shift < 0) {
        const int n = B.cursor;
        if (n != B.count) {
            if (tid == 0) atomicMin(Q.ctr + 3, (unsigned long long)B.slot);
            return;
        }
        int m = 1;
        while (m < n) m *= 2;
        for (int j = tid; j < m; j += QUANT_THREADS) keys[j] = j < n ? Q.seg[B.base + j] : ~0ull;
        __syncthreads();
        for (int k = 2; k <= m; k *= 2)
            for (int h = k / 2; h > 0; h /= 2) {
                for (int j = tid; j < m; j += QUANT_THREADS) {
                    const int o = j ^ h;
                    if (o > j) {
                        const unsigned long long a = keys[j], b = keys[o];
                        if ((a > b) == ((j & k) == 0)) keys[j] = b, keys[o] = a;
                    }
                }
                __syncthreads();
            }
        if (tid < Q.n_lev && want[tid] > 0) {
            lv[tid].key = keys[want[tid] - 1];
            lv[tid].state = QL_DONE;
        }
        return;
    }
    // bins [b0, b1) of this thread
    const int nb = 1 << Q.nb_log2, per = (nb + QUANT_THREADS - 1) / QUANT_THREADS;
    const int b0 = min(nb, tid * per), b1 = min(nb, b0 + per);
    const unsigned *const h = Q.hist + B.base;
    int mine = 0;
    for (int b = b0; b < b1; b++) mine += (int)h[b];
    // exclusive scan of `mine` across the CTA
    const int lane = tid & 31, warp = tid >> 5;
    int inc = mine;
    for (int o = 1; o < 32; o *= 2) {
        const int v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) part[warp] = inc;
    __syncthreads();
    int before = inc - mine, total = 0;
    for (int w = 0; w < QUANT_THREADS / 32; w++) {
        if (w < warp) before += part[w];
        total += part[w];
    }
    if (total != B.count) {
        if (tid == 0) atomicMin(Q.ctr + 3, (unsigned long long)B.slot);
        return;
    }
    for (int l = 0; l < Q.n_lev; l++) {
        const int r = want[l];
        if (r <= before || r > before + mine) continue;
        int c = before, b = b0;
        while (c + (int)h[b] < r) c += (int)h[b++];
        QuantLevel &L = lv[l];
        L.below += c;
        L.count = (int)h[b];
        L.lo = B.lo + ((unsigned long long)b << B.shift);
        const unsigned long long width = B.shift == 0 ? 0ull : (~0ull >> (64 - B.shift));
        L.hi = L.lo + (B.hi - L.lo < width ? B.hi - L.lo : width);
        if (L.lo == L.hi) L.state = QL_DONE, L.key = L.lo;
    }
}
// the brackets of the pass, a CTA each (launched with one CTA per bracket; the CPU emulation runs a few CTAs)
template <int = 0> __global__ void __launch_bounds__(QUANT_THREADS) quant_bracket_kernel(const QuantParams Q) {
    for (long long bi = blockIdx.x; bi < Q.n_br; bi += gridDim.x) {
        quant_bracket(Q, bi);
        __syncthreads(); // the shared arrays are free again
    }
}

// one thread per slot: the quantiles (NaN where a level has no value) and the replicates without a value
// (-1 on a slot without values)
template <int = 0> __global__ void quant_out_kernel(const QuantParams Q) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= Q.n_slots) return;
    const int n = Q.n[i];
    const long long k = i / Q.n_steps, row = i % Q.n_steps;
    Q.nonfinite[i] = n < 0 ? -1 : Q.n_reps - n;
    for (int l = 0; l < Q.n_lev; l++) {
        const QuantLevel &L = Q.lv[i * Q.n_lev + l];
        Q.q[(k * Q.n_lev + l) * Q.n_steps + row] = L.state == QL_DONE ? quant_value(L.key) : NAN;
    }
}

} // namespace ldsr
