// ldsr_abi.cu -- host side of the engine: packing, plans, the EM driver loop, multi-GPU sharding,
// and the extern "C" surface declared in include/ldsr_b200.h.
#include "../../include/ldsr_b200.h"
#include "generic_kernels.cuh"
#include "kernel_table.h"
#include "r_rng.cuh"
#include "scan_kernels.cuh"

#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <memory>
#include <mutex>
#include <numeric>
#include <string>
#include <thread>
#include <vector>

namespace ldsr {

// ---- per-PQ kernel tables (kernels_inst.cu, one object per width) --------------------------
// weak: a development build may leave widths out (LDSR_PQ_LIST env of build.py); release has all
#define LDSR_DECL(n) const KernelTable *kernel_table_pq##n() __attribute__((weak));
#define LDSR_PQ_LIST(X) X(1) X(2) X(3) X(4) X(5) X(6) X(7) X(8) X(10) X(12) X(16) X(24) X(32)
LDSR_PQ_LIST(LDSR_DECL)
const KernelTable *kernel_table_for(int need) {
#define LDSR_PICK(n) \
    if (need <= n && kernel_table_pq##n) return kernel_table_pq##n();
    LDSR_PQ_LIST(LDSR_PICK)
    return nullptr;
}

// ---- errors ---------------------------------------------------------------------------------
struct Err {
    int code = LDSR_OK;
    std::string msg;
    bool ok() const { return code == LDSR_OK; }
};
static Err fail(int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    Err e;
    e.code = code;
    e.msg = buf;
    return e;
}
static int report(const Err &e, char *errbuf, int errlen) {
    if (errbuf && errlen > 0) snprintf(errbuf, errlen, "%s", e.msg.c_str());
    return e.code;
}
#define CU(call)                                                                                    \
    do {                                                                                            \
        cudaError_t _e = (call);                                                                    \
        if (_e != cudaSuccess) return fail(LDSR_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(_e)); \
    } while (0)

// ---- device memory pool: grow-only cache of cudaMalloc blocks, one per device ---------------
class DevicePool {
  public:
    explicit DevicePool(int device) : device_(device) {}
    ~DevicePool() {
        cudaSetDevice(device_);
        for (auto &b : blocks_) cudaFree(b.ptr);
        for (auto &b : pinned_) cudaFreeHost(b.ptr);
        for (cudaStream_t s : streams_) cudaStreamDestroy(s);
    }
    // pinned host blocks and streams are cached the same way: a host-buffer call (ldsr_em_batch)
    // creates and destroys a plan every time, and cudaMallocHost / cudaStreamCreate are not cheap
    cudaError_t alloc_pinned(size_t bytes, void **out) {
        bytes = std::max<size_t>((bytes + 255) & ~size_t(255), 256);
        std::lock_guard<std::mutex> lk(mu_);
        for (auto &b : pinned_)
            if (!b.used && b.size >= bytes) {
                b.used = true;
                *out = b.ptr;
                return cudaSuccess;
            }
        void *p = nullptr;
        cudaError_t e = cudaMallocHost(&p, bytes);
        if (e != cudaSuccess) return e;
        pinned_.push_back({p, bytes, true});
        *out = p;
        return cudaSuccess;
    }
    void release_pinned(void *p) {
        std::lock_guard<std::mutex> lk(mu_);
        for (auto &b : pinned_)
            if (b.ptr == p) b.used = false;
    }
    cudaError_t get_stream(cudaStream_t *out) {
        std::lock_guard<std::mutex> lk(mu_);
        if (!streams_.empty()) {
            *out = streams_.back();
            streams_.pop_back();
            return cudaSuccess;
        }
        return cudaStreamCreateWithFlags(out, cudaStreamNonBlocking);
    }
    void put_stream(cudaStream_t s) {
        std::lock_guard<std::mutex> lk(mu_);
        streams_.push_back(s);
    }
    cudaError_t alloc(size_t bytes, void **out) {
        bytes = std::max<size_t>((bytes + 255) & ~size_t(255), 256);
        std::lock_guard<std::mutex> lk(mu_);
        int best = -1;
        for (int i = 0; i < (int)blocks_.size(); i++)
            if (!blocks_[i].used && blocks_[i].size >= bytes && blocks_[i].size <= 2 * bytes + 4096 &&
                (best < 0 || blocks_[i].size < blocks_[best].size))
                best = i;
        if (best >= 0) {
            blocks_[best].used = true;
            *out = blocks_[best].ptr;
            return cudaSuccess;
        }
        void *p = nullptr;
        cudaError_t e = cudaMalloc(&p, bytes);
        if (e == cudaErrorMemoryAllocation) {
            // the cache may be holding blocks of other sizes: give them back and try once more
            cudaGetLastError();
            trim_locked();
            e = cudaMalloc(&p, bytes);
        }
        if (e != cudaSuccess) return e;
        blocks_.push_back({p, bytes, true});
        *out = p;
        return cudaSuccess;
    }
    void release(void *p) {
        std::lock_guard<std::mutex> lk(mu_);
        for (auto &b : blocks_)
            if (b.ptr == p) b.used = false;
    }
    // frees every cached block that is not in use; returns the device bytes given back
    size_t trim() {
        std::lock_guard<std::mutex> lk(mu_);
        return trim_locked();
    }
    size_t cached_bytes() {
        std::lock_guard<std::mutex> lk(mu_);
        size_t n = 0;
        for (auto &b : blocks_) n += b.size;
        return n;
    }
    int device() const { return device_; }

  private:
    struct Block {
        void *ptr;
        size_t size;
        bool used;
    };
    size_t trim_locked() {
        int prev = -1;
        cudaGetDevice(&prev);
        cudaSetDevice(device_);
        size_t freed = 0;
        auto drop = [&](std::vector<Block> &v, bool pinned) {
            size_t keep = 0;
            for (auto &b : v) {
                if (b.used) {
                    v[keep++] = b;
                    continue;
                }
                if (pinned)
                    cudaFreeHost(b.ptr);
                else {
                    cudaFree(b.ptr);
                    freed += b.size;
                }
            }
            v.resize(keep);
        };
        drop(blocks_, false);
        drop(pinned_, true);
        if (prev >= 0) cudaSetDevice(prev);
        return freed;
    }
    int device_;
    std::mutex mu_;
    std::vector<Block> blocks_, pinned_;
    std::vector<cudaStream_t> streams_;
};

// ---- the CUDA resources of one call (or of one plan), given back when it goes out of scope -----
// With a pool, device and pinned blocks (and, after borrow_stream, the stream) come from it, and the owner waits for
// its stream before they go back.  Without one (the entry points that take a device number) device blocks are
// cudaMalloc'd and the work runs on the legacy stream, which cudaFree waits for.  Events die with the owner.
class Resources {
  public:
    explicit Resources(DevicePool *pool = nullptr, cudaStream_t stream = nullptr) : stream(stream), pool_(pool) {}
    Resources(const Resources &) = delete;
    Resources &operator=(const Resources &) = delete;
    ~Resources() {
        if (pool_ && stream) cudaStreamSynchronize(stream);
        for (cudaEvent_t e : events_) cudaEventDestroy(e);
        for (void *p : pinned_) pool_->release_pinned(p);
        for (void *p : blocks_) free_block(p);
        if (own_stream_) pool_->put_stream(stream);
    }
    cudaStream_t stream; // where the work of the call is enqueued
    DevicePool *pool() const { return pool_; }

    cudaError_t borrow_stream() {
        cudaError_t e = pool_->get_stream(&stream);
        own_stream_ = e == cudaSuccess;
        return e;
    }
    template <class T> cudaError_t alloc(T **out, size_t n) {
        const size_t bytes = std::max<size_t>(n, 1) * sizeof(T);
        void *p = nullptr;
        cudaError_t e = pool_ ? pool_->alloc(bytes, &p) : cudaMalloc(&p, bytes);
        if (e != cudaSuccess) return e;
        blocks_.push_back(p);
        *out = static_cast<T *>(p);
        return cudaSuccess;
    }
    // grow a block: the old one goes back at once (a plan re-used with a larger niter or with trace_liks must not
    // accumulate dead blocks until it is destroyed)
    template <class T> cudaError_t realloc(T **ptr, size_t n) {
        if (*ptr) {
            forget(blocks_, *ptr);
            free_block(*ptr);
            *ptr = nullptr;
        }
        return alloc(ptr, n);
    }
    template <class T> cudaError_t upload(T **out, const std::vector<T> &h) {
        cudaError_t e = alloc(out, h.size());
        if (e != cudaSuccess || h.empty()) return e;
        return cudaMemcpyAsync(*out, h.data(), h.size() * sizeof(T), cudaMemcpyHostToDevice, stream);
    }
    template <class T> cudaError_t alloc_pinned(T **out, size_t n) {
        void *p = nullptr;
        cudaError_t e = pool_->alloc_pinned(n * sizeof(T), &p);
        if (e != cudaSuccess) return e;
        pinned_.push_back(p);
        *out = static_cast<T *>(p);
        return cudaSuccess;
    }
    template <class T> cudaError_t realloc_pinned(T **ptr, size_t n) {
        if (*ptr) {
            forget(pinned_, *ptr);
            pool_->release_pinned(*ptr);
            *ptr = nullptr;
        }
        return alloc_pinned(ptr, n);
    }
    cudaError_t event(cudaEvent_t *out, unsigned flags = cudaEventDefault) {
        cudaError_t e = cudaEventCreateWithFlags(out, flags);
        if (e == cudaSuccess) events_.push_back(*out);
        return e;
    }

    // Device time of enqueued work: start() and stop() record a pair of events on the stream around it.
    cudaError_t start() {
        cudaEvent_t a = nullptr, b = nullptr;
        cudaError_t e = event(&a);
        if (e == cudaSuccess) e = event(&b);
        if (e != cudaSuccess) return e;
        laps_.push_back({a, b});
        return cudaEventRecord(a, stream);
    }
    cudaError_t stop() { return cudaEventRecord(laps_.back().second, stream); }
    size_t laps() const { return laps_.size(); }
    // from the start of pair `first` to the stop of pair `last`, once the device has reached that stop
    cudaError_t ms(size_t first, size_t last, float *out) const {
        cudaError_t e = cudaEventSynchronize(laps_[last].second);
        return e != cudaSuccess ? e : cudaEventElapsedTime(out, laps_[first].first, laps_[last].second);
    }
    cudaError_t total_ms(double *out) const {
        *out = 0.0;
        for (size_t i = 0; i < laps_.size(); i++) {
            float m = 0.f;
            cudaError_t e = ms(i, i, &m);
            if (e != cudaSuccess) return e;
            *out += m;
        }
        return cudaSuccess;
    }

  private:
    static void forget(std::vector<void *> &v, void *p) { v.erase(std::remove(v.begin(), v.end(), p), v.end()); }
    void free_block(void *p) {
        if (pool_)
            pool_->release(p);
        else
            cudaFree(p);
    }
    DevicePool *pool_;
    bool own_stream_ = false;
    std::vector<void *> blocks_, pinned_;
    std::vector<cudaEvent_t> events_;
    std::vector<std::pair<cudaEvent_t, cudaEvent_t>> laps_;
};

// Every entry point finds its device here, after validating its arguments: the library has no CPU path.
static Err check_device(int device) {
    const int have = ldsr_device_count();
    if (have < 1) return fail(LDSR_ERR_CUDA, "no CUDA device available (this library has no CPU path)");
    if (device < 0 || device >= have) return fail(LDSR_ERR_ARG, "device %d out of range (have %d)", device, have);
    return Err();
}
static Err use_device(int device) {
    Err e = check_device(device);
    if (!e.ok()) return e;
    CU(cudaSetDevice(device));
    return Err();
}

} // namespace ldsr

using namespace ldsr;

struct ldsr_ctx {
    std::vector<int> devices;
    std::vector<std::unique_ptr<DevicePool>> pools;
};

// ---- plan -----------------------------------------------------------------------------------
// Batches up to this size may run the scan kernel (one CTA per fit), `variant = 5` forces it up to here.  Chosen
// automatically below the measured crossover with the batched kernels (tools/profile_crossover.py, profiles/
// scan_r02_crossover.txt; NP-413, 1000 iterations: scan 3.1 / 3.9 / 5.8 / 7.5 / 9.5 / 10.1 / 10.8 ms for 200 / 400 /
// 600 / 900 / 1200 / 1300 / 1400 fits against 10.3-10.4 ms for the time-split kernel whatever the batch up to
// 4 700 fits): 1200 fits of narrow inputs; 900 of wide ones (p = q = 10, T = 400: 3.8 / 5.9 / 10.8 / 13.3 ms for
// 100 / 300 / 600 / 800 fits against 15.9 ms for the wide-input kernel)
constexpr int SCAN_MAX_FITS = 1500;
inline int scan_auto_fits(int pq) { return pq <= 4 ? 1200 : 900; }
constexpr size_t COUNTS_CAP = 256; // (tasks, live fits) per chunk: room for 128 chunks without regrowing
struct ldsr_plan {
    ldsr_plan(int device, DevicePool *pool)
        : device(device), own_pool(pool ? nullptr : new DevicePool(device)), cuda(pool ? pool : own_pool.get()) {}
    ~ldsr_plan() { cudaSetDevice(device); } // then `cuda` waits for the plan's stream and gives everything back
    int device = 0;
    int n_sm = 148;
    std::unique_ptr<DevicePool> own_pool;
    Resources cuda; // the plan's stream, its device blocks and pinned blocks
    const KernelTable *kt = nullptr;
    int PQ = 0, TL = 0;
    int n_series = 0, n_groups = 0, n_fits = 0, theta_stride = 0;
    int max_T = 0, max_seg = 0;
    int max_units = 0; // time-split kernel: upper bound on units per series (em_split_kernel.cuh)
    int wide_units = 0, wide_msteps = 0; // wide-input kernel: units / steps of observed units (em_wide_kernel.cuh)
    size_t max_blob_bytes = 0;
    bool blob_in_smem = true;
    int last_niter = 0;
    // host metadata (internal order)
    std::vector<SeriesDev> h_series;
    std::vector<int> g_user, f_user, h_g_series, h_g_fit_ptr, h_f_group;
    std::vector<int> s_p, s_q, s_T;
    std::vector<int> user_fit_series; // per USER fit: its series (filled only when the rows differ in width)
    std::vector<long long> h_traj_ptr_user; // per USER group: offset of its trajectory row
    long long traj_total = 0;
    std::vector<long long> h_g_mask_off; // per group: its first mask word
    // one job per fit with its rows in the caller's fit order (ldsr_smoother_batch's layout): per USER fit the
    // offset of its rows, and per fit the job's row offset and theta row
    std::vector<long long> fit_row_user, fit_job_row;
    std::vector<int> fit_job_theta;
    // device
    SeriesDev *d_series = nullptr;
    double *d_blobs = nullptr, *d_sconst = nullptr, *d_gconst = nullptr, *d_uwin = nullptr;
    int *d_g_series = nullptr, *d_g_status = nullptr, *d_g_nobs = nullptr, *d_g_fit_ptr = nullptr;
    int *d_held_ptr = nullptr, *d_held_idx = nullptr;
    unsigned *d_masks = nullptr;
    long long *d_g_mask_off = nullptr;
    int *d_f_group = nullptr, *d_f_user = nullptr;
    double *d_theta0 = nullptr, *d_theta = nullptr, *d_l1 = nullptr, *d_l2 = nullptr, *d_lik = nullptr;
    int *d_ne = nullptr, *d_done = nullptr, *d_status = nullptr;
    double *d_liks = nullptr;
    size_t liks_cap = 0;
    int *d_active = nullptr, *d_task_off = nullptr, *d_n_live = nullptr, *d_counts = nullptr;
    size_t counts_cap = COUNTS_CAP;
    int4 *d_tasks = nullptr;
    int max_tasks = 0;
    unsigned long long *d_sum = nullptr;
    unsigned *d_ticket = nullptr; // compact_kernel's last-block counter (0 between launches)
    int *d_share_flags = nullptr; // [max_tasks] hand-over flags of em_split_kernel's iteration-level task sharing
    int *d_share_ctl = nullptr, *d_share_order = nullptr, *d_share_key = nullptr; // its ranked task assignment
                                                                                  // (SHARE_CTL_LEN, max_tasks, max_tasks)
    int share_epoch = 0;          // one value per launch: the flags need no reset
    double *d_ckpt = nullptr;
    size_t ckpt_cap = 0;
    int *d_best = nullptr;
    // winners' trajectories (internal group order rows)
    double *d_X = nullptr, *d_Y = nullptr, *d_V = nullptr, *d_J = nullptr;
    // results block in the caller's order (pack_results_kernel), fetched with one copy:
    // [theta nf x stride | lik nf | iters nf, status nf, best ng (int) | X | Y | V | J]
    double *d_res = nullptr, *h_res = nullptr; // h_res pinned
    size_t res_head = 0, res_total = 0;        // doubles: everything before X, everything
    int *d_g_user = nullptr;
    bool same_width = true; // every series has p + q + 6 == theta_stride
    int *d_job_group = nullptr, *d_job_theta = nullptr;
    long long *d_job_row = nullptr;
    int *h_counts = nullptr; // pinned
    bool em_done = false;
};

namespace ldsr {

// pad a caller theta (p,q) into the device layout (PQ,PQ).  Without u (v) the caller's B (D)
// entries are not used by any kernel and come back as zeros (EM.cpp:186,154).
static void pad_theta(const double *src, int p, int q, bool has_u, bool has_v, int PQ, double *dst) {
    std::fill(dst, dst + 2 * PQ + 6, 0.0);
    dst[0] = src[0];
    if (has_u)
        for (int j = 0; j < p; j++) dst[1 + j] = src[1 + j];
    dst[1 + PQ] = src[1 + p];
    if (has_v)
        for (int j = 0; j < q; j++) dst[2 + PQ + j] = src[2 + p + j];
    for (int k = 0; k < 4; k++) dst[2 + 2 * PQ + k] = src[2 + p + q + k];
}
static void unpad_theta(const double *src, int p, int q, bool has_u, bool has_v, int PQ, double *dst) {
    dst[0] = src[0];
    for (int j = 0; j < p; j++) dst[1 + j] = has_u ? src[1 + j] : 0.0;
    dst[1 + p] = src[1 + PQ];
    for (int j = 0; j < q; j++) dst[2 + p + j] = has_v ? src[2 + PQ + j] : 0.0;
    for (int k = 0; k < 4; k++) dst[2 + p + q + k] = src[2 + 2 * PQ + k];
}
// a caller's theta table (user fit order, theta_stride apart) in the plan's fit order and padded layout
static std::vector<double> padded_thetas(const ldsr_plan *P, const double *theta) {
    std::vector<double> th((size_t)P->n_fits * P->TL);
    for (int fi = 0; fi < P->n_fits; fi++) {
        const int s = P->h_g_series[P->h_f_group[fi]];
        pad_theta(theta + (size_t)P->f_user[fi] * P->theta_stride, P->s_p[s], P->s_q[s], P->h_series[s].has_u != 0,
                  P->h_series[s].has_v != 0, P->PQ, &th[(size_t)fi * P->TL]);
    }
    return th;
}

// the smoother / propagate / coefficient kernels over n_jobs jobs of a plan's series and masks
static SmootherParams smoother_params(const ldsr_plan *P, int n_jobs, const int *job_group, const int *job_theta,
                                      const long long *job_row, const double *theta, double *X, double *Y, double *V,
                                      double *J, double *lik, int stdlik, double *aux) {
    SmootherParams sp;
    sp.series = P->d_series;
    sp.blobs = P->d_blobs;
    sp.g_series = P->d_g_series;
    sp.masks = P->d_masks;
    sp.g_mask_off = P->d_g_mask_off;
    sp.g_nobs = P->d_g_nobs;
    sp.n_jobs = n_jobs;
    sp.job_group = job_group;
    sp.job_theta = job_theta;
    sp.job_row = job_row;
    sp.theta = theta;
    sp.X = X;
    sp.Y = Y;
    sp.V = V;
    sp.J = J;
    sp.lik = lik;
    sp.stdlik = stdlik;
    sp.aux = aux;
    return sp;
}

static Err validate(const ldsr_batch *b) {
    if (!b) return fail(LDSR_ERR_ARG, "batch is NULL");
    if (b->n_series < 1 || b->n_groups < 1 || b->n_fits < 1)
        return fail(LDSR_ERR_ARG, "n_series, n_groups and n_fits must all be >= 1");
    if (!b->T || !b->p || !b->q || !b->y || !b->group_series || !b->fit_group || !b->theta0)
        return fail(LDSR_ERR_ARG, "a required table pointer is NULL");
    for (int s = 0; s < b->n_series; s++) {
        if (b->T[s] < 2) return fail(LDSR_ERR_ARG, "series %d: T=%d, need T >= 2", s, b->T[s]);
        if (b->p[s] < 0 || b->q[s] < 0) return fail(LDSR_ERR_ARG, "series %d: negative p or q", s);
        if (b->p[s] > LDSR_MAX_PQ || b->q[s] > LDSR_MAX_PQ)
            return fail(LDSR_ERR_UNSUPPORTED, "series %d: p=%d q=%d exceeds LDSR_MAX_PQ=%d", s, b->p[s], b->q[s],
                        LDSR_MAX_PQ);
        if (!b->y[s]) return fail(LDSR_ERR_ARG, "series %d: y is NULL", s);
        if (b->u && b->u[s] && b->p[s] < 1) return fail(LDSR_ERR_ARG, "series %d: u given but p=0", s);
        if (b->v && b->v[s] && b->q[s] < 1) return fail(LDSR_ERR_ARG, "series %d: v given but q=0", s);
        if (b->theta_stride < b->p[s] + b->q[s] + 6)
            return fail(LDSR_ERR_ARG, "theta_stride=%d < p+q+6=%d (series %d)", b->theta_stride,
                        b->p[s] + b->q[s] + 6, s);
        for (int t = 0; t < b->T[s]; t++)
            if (std::isinf(b->y[s][t])) return fail(LDSR_ERR_ARG, "series %d: y[%d] is +-Inf", s, t);
    }
    for (int g = 0; g < b->n_groups; g++) {
        const int s = b->group_series[g];
        if (s < 0 || s >= b->n_series) return fail(LDSR_ERR_ARG, "group %d: series id %d out of range", g, s);
        if (b->held_ptr) {
            if (b->held_ptr[g + 1] < b->held_ptr[g]) return fail(LDSR_ERR_ARG, "held_ptr not monotone at group %d", g);
            for (int k = b->held_ptr[g]; k < b->held_ptr[g + 1]; k++)
                if (b->held_idx[k] < 0 || b->held_idx[k] >= b->T[s])
                    return fail(LDSR_ERR_ARG, "group %d: held-out step %d outside 0..%d", g, b->held_idx[k],
                                b->T[s] - 1);
        }
    }
    for (int f = 0; f < b->n_fits; f++) {
        const int g = b->fit_group[f];
        if (g < 0 || g >= b->n_groups) return fail(LDSR_ERR_ARG, "fit %d: group id %d out of range", f, g);
        if (f > 0 && g < b->fit_group[f - 1])
            return fail(LDSR_ERR_ARG, "fit_group must be non-decreasing (fit %d)", f);
    }
    return Err();
}

// The widest input row of a batch (series s has input rows u[s] of width p[s], v[s] of width q[s], either may be
// absent): the kernels are compiled per padded width.
static int input_width(int n_series, const double *const *u, const double *const *v, const int *p, const int *q) {
    int need = 1;
    for (int s = 0; s < n_series; s++) {
        if (u && u[s]) need = std::max(need, p[s]);
        if (v && v[s]) need = std::max(need, q[s]);
    }
    return need;
}

// per group: its fits are lo[g] .. hi[g] - 1 (fit_group is non-decreasing), or lo[g] = hi[g] = -1 without fits
static void fit_ranges(const ldsr_batch *b, std::vector<int> &lo, std::vector<int> &hi) {
    lo.assign(b->n_groups, -1);
    hi.assign(b->n_groups, -1);
    for (int f = 0; f < b->n_fits; f++) {
        const int g = b->fit_group[f];
        if (lo[g] < 0) lo[g] = f;
        hi[g] = f + 1;
    }
}

// A call given no context runs on a temporary one, which `tmp` owns: device 0, or the devices of ldsr_options.
static Err default_ctx(ldsr_ctx *&ctx, std::unique_ptr<ldsr_ctx> &tmp, int n_devices = 1, const int *devices = nullptr) {
    if (ctx) return Err();
    char buf[256];
    const int rc = ldsr_ctx_create(n_devices, devices, &ctx, buf, sizeof buf);
    if (rc != LDSR_OK) return fail(rc, "%s", buf);
    tmp.reset(ctx);
    return Err();
}

// b has passed validate()
static Err plan_build(const ldsr_batch *b, int device, DevicePool *pool, ldsr_plan **out) {
    Err e = use_device(device);
    if (!e.ok()) return e;

    std::unique_ptr<ldsr_plan> P(new ldsr_plan(device, pool));
    CU(P->cuda.borrow_stream());
    CU(P->cuda.alloc_pinned(&P->h_counts, COUNTS_CAP));
    CU(cudaDeviceGetAttribute(&P->n_sm, cudaDevAttrMultiProcessorCount, device));

    const int ns = b->n_series, ng = b->n_groups, nf = b->n_fits;
    P->n_series = ns;
    P->n_groups = ng;
    P->n_fits = nf;
    P->theta_stride = b->theta_stride;
    const int need = input_width(ns, b->u, b->v, b->p, b->q);
    P->kt = kernel_table_for(need);
    if (!P->kt) return fail(LDSR_ERR_UNSUPPORTED, "input width %d has no kernel instantiation", need);
    const int PQ = P->PQ = P->kt->pq;
    P->TL = 2 * PQ + 6;
    P->s_p.assign(b->p, b->p + ns);
    P->s_q.assign(b->q, b->q + ns);
    P->s_T.assign(b->T, b->T + ns);

    // ---- internal order: groups sorted by series (stable), fits follow their groups
    std::vector<int> fit_lo, fit_hi;
    fit_ranges(b, fit_lo, fit_hi);
    P->g_user.resize(ng);
    std::iota(P->g_user.begin(), P->g_user.end(), 0);
    std::stable_sort(P->g_user.begin(), P->g_user.end(),
                     [&](int a, int c) { return b->group_series[a] < b->group_series[c]; });
    P->h_g_series.resize(ng);
    P->h_g_fit_ptr.assign(ng + 1, 0);
    P->f_user.clear();
    P->h_f_group.clear();
    for (int gi = 0; gi < ng; gi++) {
        const int gu = P->g_user[gi];
        P->h_g_series[gi] = b->group_series[gu];
        P->h_g_fit_ptr[gi] = (int)P->f_user.size();
        if (fit_lo[gu] >= 0)
            for (int f = fit_lo[gu]; f < fit_hi[gu]; f++) {
                P->f_user.push_back(f);
                P->h_f_group.push_back(gi);
            }
    }
    P->h_g_fit_ptr[ng] = (int)P->f_user.size();
    P->fit_row_user.assign(nf + 1, 0);
    for (int f = 0; f < nf; f++) P->fit_row_user[f + 1] = P->fit_row_user[f] + b->T[b->group_series[b->fit_group[f]]];
    P->fit_job_row.resize(nf);
    for (int fi = 0; fi < nf; fi++) P->fit_job_row[fi] = P->fit_row_user[P->f_user[fi]];
    P->fit_job_theta.resize(nf);
    std::iota(P->fit_job_theta.begin(), P->fit_job_theta.end(), 0);

    // ---- series blobs
    P->h_series.resize(ns);
    std::vector<double> blobs, uwin;
    long long sconst_off = 0;
    for (int s = 0; s < ns; s++) {
        SeriesDev &S = P->h_series[s];
        std::memset(&S, 0, sizeof S);
        const int T = b->T[s], p = b->p[s], q = b->q[s];
        const double *u = b->u ? b->u[s] : nullptr, *v = b->v ? b->v[s] : nullptr;
        S.T = T;
        S.p = p;
        S.q = q;
        S.has_u = u != nullptr;
        S.has_v = v != nullptr;
        S.same_uv = (u && v && p == q && (u == v || std::memcmp(u, v, sizeof(double) * (size_t)p * T) == 0)) ||
                    (!u && !v);
        const int Ty = (T + 1) & ~1;
        const int nuv = T * PQ;
        S.y_off = 0;
        S.u_off = Ty;
        S.v_off = S.same_uv ? S.u_off : ((S.u_off + nuv + 1) & ~1);
        S.blob_doubles = ((S.v_off + nuv) + 1) & ~1;
        S.blob_off = (long long)blobs.size();
        S.sconst_off = sconst_off;
        sconst_off += PQ * PQ + 1;
        blobs.resize(blobs.size() + S.blob_doubles, 0.0);
        double *B = blobs.data() + S.blob_off;
        for (int t = 0; t < T; t++) {
            B[t] = b->y[s][t];
            if (u)
                for (int j = 0; j < p; j++) B[S.u_off + (size_t)t * PQ + j] = u[(size_t)t * p + j];
            if (v && !S.same_uv)
                for (int j = 0; j < q; j++) B[S.v_off + (size_t)t * PQ + j] = v[(size_t)t * q + j];
        }
        P->max_T = std::max(P->max_T, T);
        P->max_units = std::max(P->max_units, split_units_upper_bound(b->y[s], T, P->kt->split_mseg, P->kt->split_uw));
        if (P->kt->wide_nw > 0) {
            int nu = 0, nm = 0;
            wide_count_units(b->y[s], T, P->kt->wide_mseg, P->kt->split_uw, &nu, &nm);
            P->wide_units = std::max(P->wide_units, nu);
            P->wide_msteps = std::max(P->wide_msteps, nm);
        }
        { // window Gram blocks of u for the time-split kernel's unobserved units (theta-independent)
            const int UWn = P->kt->split_uw, nwin = (T + UWn - 1) / UWn;
            S.uwin_off = (int)uwin.size();
            uwin.resize(uwin.size() + (size_t)nwin * PQ * PQ, 0.0);
            if (u)
                for (int t = 0; t < T; t++) {
                    double *G = uwin.data() + S.uwin_off + (size_t)(t / UWn) * PQ * PQ;
                    for (int a = 0; a < p; a++)
                        for (int c = 0; c < p; c++) G[a * PQ + c] += u[(size_t)t * p + a] * u[(size_t)t * p + c];
                }
        }
        P->max_blob_bytes = std::max(P->max_blob_bytes, (size_t)S.blob_doubles * 8);
    }
    // fit ranges per series (internal order is series-major)
    {
        int f = 0;
        for (int s = 0; s < ns; s++) {
            P->h_series[s].fit_begin = f;
            while (f < (int)P->h_f_group.size() && P->h_g_series[P->h_f_group[f]] == s) f++;
            P->h_series[s].fit_end = f;
        }
    }
    P->max_seg = (P->max_T + EM_SEG - 1) / EM_SEG;
    P->blob_in_smem = P->max_blob_bytes <= 200 * 1024;

    // ---- masks, hold-outs (internal group order)
    P->h_g_mask_off.resize(ng);
    long long nwords = 0;
    std::vector<int> held_ptr(ng + 1, 0), held_idx;
    for (int gi = 0; gi < ng; gi++) {
        const int gu = P->g_user[gi];
        P->h_g_mask_off[gi] = nwords;
        nwords += (b->T[P->h_g_series[gi]] + 31) / 32;
        if (b->held_ptr)
            for (int k = b->held_ptr[gu]; k < b->held_ptr[gu + 1]; k++) held_idx.push_back(b->held_idx[k]);
        held_ptr[gi + 1] = (int)held_idx.size();
    }
    // ---- trajectory rows: user-order prefix sum of T
    P->h_traj_ptr_user.resize(ng + 1);
    P->h_traj_ptr_user[0] = 0;
    for (int g = 0; g < ng; g++) P->h_traj_ptr_user[g + 1] = P->h_traj_ptr_user[g] + b->T[b->group_series[g]];
    P->traj_total = P->h_traj_ptr_user[ng];

    // ---- upload
    Resources &cuda = P->cuda;
    CU(cuda.upload(&P->d_series, P->h_series));
    CU(cuda.upload(&P->d_blobs, blobs));
    if (uwin.empty()) uwin.push_back(0.0);
    CU(cuda.upload(&P->d_uwin, uwin));
    CU(cuda.upload(&P->d_g_series, P->h_g_series));
    CU(cuda.upload(&P->d_g_fit_ptr, P->h_g_fit_ptr));
    CU(cuda.upload(&P->d_g_mask_off, P->h_g_mask_off));
    CU(cuda.upload(&P->d_held_ptr, held_ptr));
    if (held_idx.empty()) held_idx.push_back(0);
    CU(cuda.upload(&P->d_held_idx, held_idx));
    CU(cuda.upload(&P->d_f_group, P->h_f_group));
    CU(cuda.upload(&P->d_f_user, P->f_user));
    CU(cuda.upload(&P->d_g_user, P->g_user));
    for (int s = 0; s < ns; s++) P->same_width = P->same_width && b->p[s] + b->q[s] + 6 == b->theta_stride;
    if (!P->same_width) {
        P->user_fit_series.resize(nf);
        for (int f = 0; f < nf; f++) P->user_fit_series[f] = b->group_series[b->fit_group[f]];
    }
    P->res_head = (size_t)nf * b->theta_stride + nf + ((size_t)2 * nf + ng + 1) / 2;
    P->res_total = P->res_head + 4 * (size_t)P->traj_total; // allocated by the first ldsr_plan_em
    CU(cuda.upload(&P->d_theta0, padded_thetas(P.get(), b->theta0)));
    CU(cuda.alloc(&P->d_masks, (size_t)nwords));
    CU(cuda.alloc(&P->d_sconst, (size_t)sconst_off));
    CU(cuda.alloc(&P->d_gconst, (size_t)ng * gconst_stride(PQ)));
    CU(cuda.alloc(&P->d_g_status, ng));
    CU(cuda.alloc(&P->d_g_nobs, ng));
    CU(cuda.alloc(&P->d_theta, (size_t)nf * P->TL));
    CU(cuda.alloc(&P->d_l1, nf));
    CU(cuda.alloc(&P->d_l2, nf));
    CU(cuda.alloc(&P->d_lik, nf));
    CU(cuda.alloc(&P->d_ne, nf));
    CU(cuda.alloc(&P->d_done, nf));
    CU(cuda.alloc(&P->d_status, nf));
    CU(cuda.alloc(&P->d_active, nf));
    CU(cuda.alloc(&P->d_n_live, ns));
    CU(cuda.alloc(&P->d_task_off, ns + 1));
    CU(cuda.alloc(&P->d_counts, COUNTS_CAP));
    CU(cuda.alloc(&P->d_sum, 1));
    CU(cuda.alloc(&P->d_ticket, 1));
    CU(cudaMemsetAsync(P->d_ticket, 0, sizeof(unsigned), cuda.stream));
    // the time-split kernels take 32 fits per CTA; the small-batch scan kernel one fit per CTA
    P->max_tasks = std::max(nf / 32, std::min(nf, SCAN_MAX_FITS)) + ns + 1;
    CU(cuda.alloc(&P->d_tasks, P->max_tasks));
    CU(cuda.alloc(&P->d_share_flags, P->max_tasks));
    CU(cudaMemsetAsync(P->d_share_flags, 0, (size_t)P->max_tasks * sizeof(int), cuda.stream));
    CU(cuda.alloc(&P->d_share_ctl, SHARE_CTL_LEN));
    CU(cuda.alloc(&P->d_share_order, P->max_tasks));
    CU(cuda.alloc(&P->d_share_key, P->max_tasks));
    CU(cuda.alloc(&P->d_best, ng));

    // ---- set-up kernel: masks + Gram constants
    SetupParams sp;
    sp.series = P->d_series;
    sp.blobs = P->d_blobs;
    sp.n_series = ns;
    sp.n_groups = ng;
    sp.g_series = P->d_g_series;
    sp.held_ptr = P->d_held_ptr;
    sp.held_idx = P->d_held_idx;
    sp.masks = P->d_masks;
    sp.g_mask_off = P->d_g_mask_off;
    sp.gconst = P->d_gconst;
    sp.sconst = P->d_sconst;
    sp.g_status = P->d_g_status;
    sp.g_nobs = P->d_g_nobs;
    sp.pq = PQ;
    const size_t sh = (size_t)(2 * PQ * PQ + 2 * PQ + 4) * sizeof(double);
    setup_kernel<<<ng + ns, 128, sh, cuda.stream>>>(sp);
    CU(cudaGetLastError());
    merge_status_kernel<<<(ng + 127) / 128, 128, 0, cuda.stream>>>(P->d_series, P->d_sconst, P->d_g_series, ng, PQ,
                                                                P->d_g_status);
    CU(cudaGetLastError());
    // No synchronisation here: cudaMemcpyAsync from pageable memory returns once the source has
    // been staged, so the host vectors above may go out of scope; errors surface at the first sync.
    *out = P.release();
    return Err();
}

// ---- the EM driver ---------------------------------------------------------------------------
#ifdef LDSR_PHASE_CLOCKS
static long long *sp_clk_last = nullptr; // development build only (DESIGN.md 4.5)
// per-warp phase clocks of one launch of `grid` CTAs of nw warps: 21 counters per warp, the first `rows` printed
static void dump_phase_clocks(const char *kernel, const char *const *names, int rows, int width, int grid, int nw,
                              int chunk, cudaStream_t st) {
    std::vector<long long> h((size_t)grid * nw * 21);
    cudaStreamSynchronize(st);
    cudaMemcpy(h.data(), sp_clk_last, h.size() * sizeof(long long), cudaMemcpyDeviceToHost);
    std::fprintf(stderr, "[ldsr] %sphase clocks of launch 1 (cycles per iteration, mean over %d CTAs), per warp:\n",
                 kernel, grid);
    for (int i = 0; i < rows; i++) {
        std::fprintf(stderr, "[ldsr]   %-14s", names[i]);
        for (int w = 0; w < nw; w++) {
            double sum = 0;
            for (int b = 0; b < grid; b++) sum += (double)h[((size_t)b * nw + w) * 21 + i];
            std::fprintf(stderr, " %*.0f", width, sum / grid / chunk);
        }
        std::fprintf(stderr, "\n");
    }
}
#endif
static Err plan_em(ldsr_plan *P, int niter, double tol, const ldsr_options *opt, cudaStream_t st, bool want_liks,
                   std::atomic<int> *abort_flag, long long *stats) {
    if (niter < 2) return fail(LDSR_ERR_ARG, "niter=%d: the reference requires niter >= 2 (EM.cpp:247,256)", niter);
    if (!(tol == tol)) return fail(LDSR_ERR_ARG, "tol is NaN");
    CU(cudaSetDevice(P->device));
    if (!st) st = P->cuda.stream;
    Resources clk(nullptr, st); // events on the stream the EM runs on
    if (st != P->cuda.stream) {
        // the plan's uploads and set-up kernels were enqueued on its own stream: order the caller's after them
        cudaEvent_t ready = nullptr;
        CU(clk.event(&ready, cudaEventDisableTiming));
        CU(cudaEventRecord(ready, P->cuda.stream));
        CU(cudaStreamWaitEvent(st, ready, 0));
    }
    const int nf = P->n_fits, ns = P->n_series, ng = P->n_groups;
    int chunk = (opt && opt->chunk_iters > 0) ? opt->chunk_iters : 100;
    long long launches = 0, chunks = 0;
    double em_ms = 0.0;
    P->last_niter = niter;
    P->em_done = false;

    if (want_liks) {
        const size_t need = (size_t)nf * niter;
        if (P->liks_cap < need) {
            P->liks_cap = 0;
            CU(P->cuda.realloc(&P->d_liks, need));
            P->liks_cap = need;
        }
        fill_nan_kernel<<<(unsigned)((need + 255) / 256), 256, 0, st>>>(P->d_liks, need);
        launches++;
    }
    {
        const int n = nf * P->TL;
        init_state_kernel<<<(n + 255) / 256, 256, 0, st>>>(nf, P->TL, P->d_theta0, P->d_theta, P->d_l1, P->d_l2,
                                                           P->d_lik, P->d_ne, P->d_done);
        CU(cudaGetLastError());
        launches++;
    }
    // shared-memory plan: series blob (TMA-staged) [+ checkpoints of the CTA's warps]
    const size_t blob_sm = (P->max_blob_bytes + 127) & ~size_t(127);
    const size_t ck_sm = (size_t)EM_WARPS * P->max_seg * 64 * sizeof(double);
    int mode = 0;
    size_t smem = 0;
    if (P->blob_in_smem) {
        mode = 1;
        smem = blob_sm;
        if (blob_sm + ck_sm <= 220 * 1024 && !(opt && opt->variant == 1)) {
            mode = 2;
            smem = blob_sm + ck_sm;
        }
    }
    // time-split kernels: 32 fits per CTA, the warps of the CTA share the time axis.
    //   em_split_kernel (em_split_kernel.cuh): everything in registers -- the kernel of narrow inputs;
    //   em_wide_kernel  (em_wide_kernel.cuh): the input-row work in separate phases through shared memory --
    //   the kernel of wide inputs (PQ >= 5) whenever its shared-memory plan fits.
    // variant: 0 auto, 1 lane kernel with global checkpoints, 2 lane kernel, 3 time-split kernel,
    //          4 wide-input time-split kernel
    // 6 = automatic, but never the small-batch scan kernel: what the workers of a sharded call get when the WHOLE
    // batch is above the scan kernel's range, so that the kernel family -- and with it the last bits of the
    // results -- does not depend on the number of devices the batch is shared by
    const bool no_scan = opt && opt->variant == 6;
    const int variant = (opt && !no_scan) ? opt->variant : 0;
    const int max_uunits = (P->max_T + P->kt->split_uw - 1) / P->kt->split_uw;
    const size_t split_sm = blob_sm + split_smem_bytes(P->PQ, P->kt->split_nw, P->max_units, max_uunits);
    const size_t wide_blob_sm = wide_blob_smem(P->max_blob_bytes, P->max_T);
    const size_t wide_sm = P->kt->wide_nw > 0
                               ? wide_blob_sm + wide_smem_bytes(P->PQ, P->kt->wide_nw, P->max_T, P->wide_units, P->wide_msteps)
                               : ~size_t(0);
    const bool use_wide = P->kt->wide_nw > 0 && P->blob_in_smem && wide_sm <= 227 * 1024 && (variant == 0 || variant == 4);
    if (variant == 4 && !use_wide)
        return fail(LDSR_ERR_UNSUPPORTED, "variant 4 (wide-input kernel) needs width >= 5 and %zu bytes of shared memory",
                    wide_sm);
    // small batches of narrow inputs: one CTA per fit, the time axis spread over its threads (em_scan_kernel.cuh).
    // A batched kernel needs 10 us per iteration however few fits it holds; the scan kernel 2-3 us for up
    // to one fit per SM and about n/148 times that beyond, so it wins below a few hundred fits.
    // steps per thread: 4 (series up to 1024 steps).  Measured on NP-413, 100 fits x 1000 iterations: 2.91 ms with
    // 4 steps per thread (4 warps), 3.36 ms with 2 (7 warps: the cross-warp chains and barriers outweigh the
    // shorter per-thread recursions).  LDSR_SCAN_L=2 (development) selects the latter where it fits.
    // Wider inputs (5 .. SCAN_MAX_PQ) keep one set of rows in registers: 2 steps per thread (T <= 512), v == u.
    int scan_steps = P->PQ <= 4 ? 4 : 2;
    if (const char *ev = std::getenv("LDSR_SCAN_L"))
        if (std::atoi(ev) == 2 && P->max_T <= 2 * 32 * SCAN_MAX_WARPS) scan_steps = 2;
    bool scan_uv_ok = true;
    if (P->PQ >= SCAN_SHARE_UV_FROM)
        for (const SeriesDev &S : P->h_series) scan_uv_ok = scan_uv_ok && S.same_uv != 0 && S.has_u != 0;
    const bool scan_ok = P->kt->scan_l > 0 && scan_uv_ok && P->max_T <= scan_steps * 32 * SCAN_MAX_WARPS;
    const bool use_scan = scan_ok && !no_scan &&
                          ((variant == 0 && nf <= scan_auto_fits(P->PQ)) || (variant == 5 && nf <= SCAN_MAX_FITS));
    if (variant == 5 && !use_scan)
        return fail(LDSR_ERR_UNSUPPORTED,
                    "variant 5 (scan kernel) needs input width <= %d, T <= %d (%d and v == u for width > 4) and at most %d fits",
                    SCAN_MAX_PQ, 32 * SCAN_L * SCAN_MAX_WARPS, 32 * 2 * SCAN_MAX_WARPS, SCAN_MAX_FITS);
    bool use_split = !use_scan && !use_wide && P->blob_in_smem && split_sm <= 227 * 1024 && (variant == 0 || variant == 3);
    if (variant == 3 && !use_split)
        return fail(LDSR_ERR_UNSUPPORTED, "variant 3 (time-split kernel) needs %zu bytes of shared memory", split_sm);
    if (use_scan) {
        smem = 0;
    } else if (use_wide) {
        smem = wide_sm;
        CU(P->kt->em_wide_prepare(smem));
    } else if (use_split) {
        smem = split_sm;
        CU(P->kt->em_split_prepare(smem));
    } else {
        CU(P->kt->em_prepare(std::max<size_t>(smem, 1024)));
    }
    const int fits_per_cta = use_scan ? 1 : ((use_split || use_wide) ? 32 : 32 * EM_WARPS);

    EmParams ep;
    ep.series = P->d_series;
    ep.blobs = P->d_blobs;
    ep.sconst = P->d_sconst;
    ep.uwin = P->d_uwin;
    ep.g_series = P->d_g_series;
    ep.masks = P->d_masks;
    ep.g_mask_off = P->d_g_mask_off;
    ep.gconst = P->d_gconst;
    ep.g_status = P->d_g_status;
    ep.f_group = P->d_f_group;
    ep.theta = P->d_theta;
    ep.l1 = P->d_l1;
    ep.l2 = P->d_l2;
    ep.lik = P->d_lik;
    ep.ne = P->d_ne;
    ep.done = P->d_done;
    ep.liks = want_liks ? P->d_liks : nullptr;
    ep.f_user = P->d_f_user;
    ep.active = P->d_active;
    ep.tasks = P->d_tasks;
    ep.max_seg = P->max_seg;
    ep.niter = niter;
    // One CTA per fit needs no compaction between launches (a finished fit's CTA simply leaves its loop): without a
    // poll callback, and unless the caller fixed the chunk length, the scan kernel runs all iterations in ONE launch
    // (config 1: 24 launches -> 6, 0.2 ms of a 3.2 ms call).
    if (use_scan && !(opt && opt->chunk_iters > 0) && !(opt && opt->poll) && abort_flag == nullptr) chunk = niter;
    ep.chunk = chunk;
    ep.tol = tol;
    ep.mode = mode;
    ep.ckpt_smem_off = (int)blob_sm;
    ep.ckpt = nullptr;

    // Chunk loop.  Every chunk is compact -> build task list -> EM kernel.  The number of chunks is
    // bounded by ceil(niter/chunk), and the task count can only shrink, so without a poll callback
    // the whole sequence is enqueued at once: each EM launch uses the first chunk's grid and reads
    // its actual task count from device memory (CTAs beyond it exit immediately).  With a poll
    // callback the host synchronises after every chunk, as the reference polls for interrupts
    // every 100 iterations (EM.cpp:261).
    const int max_chunks = (niter + chunk - 1) / chunk;
    // abort_flag != NULL: this is a per-device worker of a sharded call whose CALLER polls.  The worker
    // never runs the callback itself (it belongs to the calling thread: an R shim runs
    // R_CheckUserInterrupt there); it only looks at the flag the calling thread raises.
    const bool sync_each = (opt && opt->poll) || abort_flag != nullptr;
    int grid0 = 0; // task count of the first chunk: every fit is live
    for (int s = 0; s < ns; s++)
        grid0 += (P->h_series[s].fit_end - P->h_series[s].fit_begin + fits_per_cta - 1) / fits_per_cta;
    // Batches of one to four waves of the time-split kernel (10 000 fits: 313 tasks for 2 x 148 CTAs): a co-resident
    // grid shares the tasks by ITERATIONS (em_split_kernel.cuh, task loop), so the chunk costs its share of a
    // wave (313/296) instead of a second wave or a third CTA per SM with 168 registers.  Beyond four waves the
    // hardware's dealing of whole tasks balances better: tasks end early as their fits converge.
    int share_slots = 0;
    bool share_ranked = false;
    if (use_split && P->kt->em_split_resident) {
        static const bool no_share = std::getenv("LDSR_NO_SHARE") != nullptr; // development: A/B measurement
        int coop = 0, dev = 0;
        CU(cudaGetDevice(&dev));
        CU(cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, dev));
        const int slots = P->kt->em_split_resident(smem) * P->n_sm;
        if (!no_share && !std::getenv("LDSR_MAX_GRID") && coop && slots > 0 && grid0 > P->n_sm && grid0 <= 4 * slots &&
            (long long)(grid0 + 1) * chunk < (1ll << 31)) // the kernel's line of task-iterations is an int
            share_slots = slots;
        // later launches (at most one task per CTA): ranked assignment + extra iterations, see the kernel.  Needs
        // exactly two CTAs on every SM.
        static const bool no_rank = std::getenv("LDSR_NO_RANK") != nullptr; // development: A/B measurement
        share_ranked = share_slots == 2 * P->n_sm && share_slots <= 1024 && !no_rank;
    }
    if ((int)P->counts_cap < 2 * max_chunks) {
        CU(P->cuda.realloc(&P->d_counts, (size_t)2 * max_chunks));
        P->counts_cap = 2 * max_chunks;
        CU(P->cuda.realloc_pinned(&P->h_counts, (size_t)2 * max_chunks));
    }
    const size_t ck_need = (mode == 2 || use_split || use_wide || use_scan) ? 0 : (size_t)grid0 * EM_WARPS * P->max_seg * 64;
    if (P->ckpt_cap < ck_need) {
        P->ckpt_cap = 0;
        CU(P->cuda.realloc(&P->d_ckpt, ck_need));
        P->ckpt_cap = ck_need;
    }
    ep.ckpt = P->d_ckpt;
    int enq = 0;
    for (int c = 0; c < max_chunks; ++c) {
        int *cnt = P->d_counts + 2 * c;
        compact_kernel<<<ns, 1024, 0, st>>>(P->d_series, ns, P->d_done, P->d_active, P->d_n_live, fits_per_cta,
                                            P->d_tasks, P->d_task_off, cnt, P->d_ticket, P->d_ne,
                                            share_ranked ? P->d_share_ctl : nullptr, P->d_share_order, P->d_share_key);
        launches++;
        // Later chunks have at most grid0 tasks.  For a batch that fits the machine in one wave the
        // grid is capped at two CTAs per SM: CTAs are dealt to SMs in launch order, so idle CTAs
        // ahead of live ones would push three live CTAs onto some SMs while others hold one
        // (measured: 2.48 ms instead of 1.83 ms per chunk on the 10 000-fit job).
        int grid = (c == 0 || grid0 > 3 * P->n_sm) ? grid0 : std::min(grid0, 2 * P->n_sm);
        // the wide-input kernel holds one CTA per SM: one CTA per task, dealt to the SMs by the hardware as
        // they finish (tasks differ in length: fits stop at different iterations)
        if (use_wide || use_scan) grid = grid0;
        int plain_grid = grid; // one CTA per task (first launch) / the task loop of a capped grid
        if (share_slots > 0) grid = share_slots;
        // development: LDSR_MAX_GRID caps the grid so that a small batch exercises the task loop of the
        // kernels (tools/sanitize.py runs it under compute-sanitizer)
        static const int grid_cap = std::getenv("LDSR_MAX_GRID") ? std::atoi(std::getenv("LDSR_MAX_GRID")) : 0;
        if (grid_cap > 0) grid = std::min(grid, grid_cap);
        if (sync_each) {
            CU(cudaMemcpyAsync(P->h_counts + 2 * c, cnt, 2 * sizeof(int), cudaMemcpyDeviceToHost, st));
            CU(cudaStreamSynchronize(st));
            grid = plain_grid = std::max(1, P->h_counts[2 * c]);
            if (share_slots > 0) grid = share_ranked ? share_slots : std::min(grid, share_slots);
            if (P->h_counts[2 * c + 1] == 0) break;
            if (abort_flag) {
                if (abort_flag->load()) return fail(LDSR_ERR_INTERRUPTED, "interrupted");
            } else if (opt->poll(opt->poll_arg)) {
                return fail(LDSR_ERR_INTERRUPTED, "interrupted by the poll callback");
            }
        }
        ep.n_tasks = cnt;
        if (stats) CU(clk.start());
        if (use_scan) {
            ep.max_seg = P->max_T; // the scan kernel sizes its block from the longest series
            ep.mode = nf > 2 * P->n_sm ? 1 : 0; // more than two fits per SM: the three-CTAs-per-SM build (em_scan_kernel.cuh)
            CU(P->kt->em_scan(ep, grid, scan_steps, st));
        } else if (use_wide) {
            WideParams wp;
            wp.em = ep;
            wp.max_units = P->wide_units;
            wp.max_msteps = P->wide_msteps;
            wp.max_T = P->max_T;
            wp.blob_smem = (int)wide_blob_sm;
            // relative cost of an unobserved word and of an observed unit in P2 + P4 (scalar work only:
            // about 8.5 instructions per unobserved step, 90 per step of an observed unit)
            wp.cost_u = P->kt->split_uw * 17 / 2;
            wp.cost_m = P->kt->wide_mseg * 90;
            if (const char *ev = std::getenv("LDSR_WIDE_COST_M")) wp.cost_m = std::atoi(ev); // development: piece balancing
#ifdef LDSR_PHASE_CLOCKS
            if (!sp_clk_last) cudaMalloc(&sp_clk_last, sizeof(long long) * 4096 * 21 * 8);
            wp.clk = (c == 1 && grid <= 2048) ? sp_clk_last : nullptr;
#endif
            CU(P->kt->em_wide(wp, grid, smem, st));
#ifdef LDSR_PHASE_CLOCKS
            if (c == 1 && grid <= 2048) {
                static const char *names[21] = {"P1", "B1 wait", "prefix+P2", "B2 wait", "P4", "B3 wait", "-",
                                                "B4 wait", "store sums", "B5 wait", "totals", "B5b wait", "matvec rows",
                                                "B5c wait", "M-step scalars", "B6 wait", "phase A", "chain+stop", "phase C", "-", "-"};
                dump_phase_clocks("wide kernel, ", names, 19, 8, grid, P->kt->wide_nw, chunk, st);
            }
#endif
        } else if (use_split) {
            SplitParams sp;
            sp.em = ep;
            sp.max_units = P->max_units;
            sp.max_uunits = max_uunits;
            sp.blob_smem = (int)blob_sm;
            // instructions per step of a U / M unit, measured at PQ = 3 (profiles/em_r01_split3_lines.txt);
            // scaling them with the input width was tried and balanced the PQ = 10 job worse (46.2 vs 45.0 ms)
            sp.cost_u = P->kt->split_uw * 22;
            sp.cost_m = P->kt->split_mseg * 168;
#ifdef LDSR_PHASE_CLOCKS
            if (!sp_clk_last) cudaMalloc(&sp_clk_last, sizeof(long long) * 4096 * 21 * 8);
            sp.clk = (c == 1 && grid <= 4096) ? sp_clk_last : nullptr; // the second launch: a two-per-SM wave
#endif
            sp.flags = share_slots > 0 ? P->d_share_flags : nullptr;
            sp.epoch = ++P->share_epoch;
            sp.ctl = share_ranked ? P->d_share_ctl : nullptr;
            sp.order = P->d_share_order;
            sp.n_sm = P->n_sm;
            // one wave of at most two CTAs per SM: the 255-register build of the kernel
            cudaError_t le = (grid <= 2 * P->n_sm || sp.flags) ? P->kt->em_split_wide(sp, grid, smem, st)
                                                               : P->kt->em_split(sp, grid, smem, st);
            if (le == cudaErrorCooperativeLaunchTooLarge && sp.flags) {
                // fewer SMs than the device reports are ours (a partitioned GPU): one CTA per task from here on.
                // Nothing of this launch ran; the control block compact_kernel prepared is simply not used.
                cudaGetLastError();
                share_slots = 0;
                share_ranked = false;
                sp.flags = nullptr;
                sp.ctl = nullptr;
                grid = plain_grid;
                le = grid <= 2 * P->n_sm ? P->kt->em_split_wide(sp, grid, smem, st) : P->kt->em_split(sp, grid, smem, st);
            }
            CU(le);
        } else {
            CU(P->kt->em_chunk(ep, grid, smem, st));
        }
        if (stats) CU(clk.stop());
#ifdef LDSR_PHASE_CLOCKS
        if (use_split && c == 1 && grid <= 4096) {
            static const char *names[21] = {"P1 loops", "B1 wait", "P2", "B2 wait", "chain+stop", "B2' wait",
                                            "P4", "B3 wait", "M-step", "constants", "prefix", "reduce",
                                            "-", "P2 U words", "P2 M units", "P2 M1 units",
                                            "P2 US units", "P4 U words", "P4 M units", "P4 M1 units", "P4 US units"};
            dump_phase_clocks("", names, 21, 9, grid, P->kt->split_nw, chunk, st);
        }
#endif
        launches++;
        enq++;
    }
    if (!sync_each) {
        CU(cudaMemcpyAsync(P->h_counts, P->d_counts, (size_t)2 * max_chunks * sizeof(int), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        if (abort_flag && abort_flag->load()) return fail(LDSR_ERR_INTERRUPTED, "interrupted");
    } else {
        CU(cudaStreamSynchronize(st));
    }
    static const bool trace_chunks = std::getenv("LDSR_TIMING") != nullptr;
    for (int c = 0; c < enq; ++c) {
        if (P->h_counts[2 * c + 1] > 0) chunks++; // launches that had live fits
        if (stats) {
            float ms = 0.f;
            CU(clk.ms(c, c, &ms));
            if (P->h_counts[2 * c + 1] > 0) em_ms += ms;
            if (trace_chunks)
                std::fprintf(stderr, "[ldsr] chunk %d: %d tasks, %d live fits, %.3f ms\n", c, P->h_counts[2 * c],
                             P->h_counts[2 * c + 1], ms);
        }
    }
    // ---- selection + the winners' smoothed trajectories
    const bool trace_tail = trace_chunks && stats;
    if (trace_tail) CU(clk.start());
    select_kernel<<<(ng + 3) / 4, 128, 0, st>>>(ng, P->d_g_fit_ptr, P->d_theta, P->TL, 1 + P->PQ, P->d_lik,
                                                    P->d_g_status, P->d_best, P->d_status);
    CU(cudaGetLastError());
    launches++;
    if (!P->d_X) {
        CU(P->cuda.alloc(&P->d_res, P->res_total));
        P->d_X = P->d_res + P->res_head;
        P->d_Y = P->d_X + P->traj_total;
        P->d_V = P->d_Y + P->traj_total;
        P->d_J = P->d_V + P->traj_total;
        std::vector<int> jg(ng);
        std::vector<long long> jr(ng);
        for (int gi = 0; gi < ng; gi++) {
            jg[gi] = gi;
            jr[gi] = P->h_traj_ptr_user[P->g_user[gi]];
        }
        CU(P->cuda.alloc(&P->d_job_group, ng));
        CU(cudaMemcpyAsync(P->d_job_group, jg.data(), ng * sizeof(int), cudaMemcpyHostToDevice, st));
        CU(P->cuda.alloc(&P->d_job_row, ng));
        CU(cudaMemcpyAsync(P->d_job_row, jr.data(), ng * sizeof(long long), cudaMemcpyHostToDevice, st));
    }
    // job_theta: the best fit (internal index) or -1
    const SmootherParams sp = smoother_params(P, ng, P->d_job_group, P->d_best, P->d_job_row, P->d_theta, P->d_X,
                                              P->d_Y, P->d_V, P->d_J, nullptr, 1, nullptr);
    // One thread per winner walks 2 T dependent steps (0.12 ms at T = 413, however few the groups); where the scan
    // kernel applies (its width / length / v == u conditions, whatever the batch size) its E-step does it in a few us
    static const bool seq_traj = std::getenv("LDSR_SEQ_TRAJ") != nullptr; // development: A/B measurement
    if (scan_ok && !seq_traj) {
        EmParams tp = ep;
        tp.max_seg = P->max_T;
        tp.n_jobs = ng;
        tp.job_group = sp.job_group;
        tp.job_theta = sp.job_theta;
        tp.job_row = sp.job_row;
        tp.tX = sp.X;
        tp.tY = sp.Y;
        tp.tV = sp.V;
        tp.tJ = sp.J;
        CU(P->kt->em_scan_traj(tp, scan_steps, st));
    } else {
        CU(P->kt->smoother(sp, st));
    }
    launches++;
    if (trace_tail) CU(clk.stop());
    CU(cudaMemsetAsync(P->d_sum, 0, sizeof(unsigned long long), st));
    sum_int_kernel<<<64, 256, 0, st>>>(P->d_ne, nf, P->d_sum);
    launches++;
    unsigned long long total = 0;
    CU(cudaMemcpyAsync(&total, P->d_sum, sizeof total, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    CU(cudaGetLastError());
    P->em_done = true;
    if (trace_tail) { // the last pair; pairs 0 .. enq - 1 are the chunks
        float ms = 0.f, all = 0.f;
        clk.ms(enq, enq, &ms);
        if (enq > 0) clk.ms(0, enq, &all);
        std::fprintf(stderr, "[ldsr] selection + winners' smoother %.3f ms; first chunk start -> end %.3f ms\n", ms, all);
    }
    if (stats) {
        stats[0] = launches;
        stats[1] = chunks;
        stats[2] = (long long)total;
        stats[3] = (long long)(em_ms * 1e6);
        stats[4] = use_scan ? 3 : (use_wide ? 2 : (use_split ? 1 : 0)); // which EM kernel ran
        stats[5] = share_slots; // > 0: the CTAs of a co-resident grid shared the tasks by iterations
        stats[6] = stats[7] = 0;
    }
    return Err();
}

// Where the rows of a sub-batch (one device's share of a sharded call) go in the caller's arrays: local
// fit i is the caller's fit fits[i], local group gl the caller's group groups[gl], whose trajectory
// row starts at traj_ptr[groups[gl]].  Workers of different devices write disjoint rows.
struct FetchMap {
    const int *fits, *groups;
    const long long *traj_ptr; // caller-wide, [n_groups + 1]
    int niter;
};

static Err plan_fetch(ldsr_plan *P, ldsr_em_result *out, const FetchMap *map = nullptr) {
    if (!P->em_done) return fail(LDSR_ERR_ARG, "ldsr_plan_fetch before a successful ldsr_plan_em");
    if (!out) return fail(LDSR_ERR_ARG, "result struct is NULL");
    CU(cudaSetDevice(P->device));
    const int nf = P->n_fits, ng = P->n_groups, stride = P->theta_stride;
    cudaStream_t st = P->cuda.stream;
    // pack on the device (caller's order and layout), one copy into pinned memory, then plain memcpys
    double *d_theta_u = P->d_res, *d_lik_u = d_theta_u + (size_t)nf * stride;
    int *d_int = reinterpret_cast<int *>(d_lik_u + nf);
    PackParams pk;
    pk.n_fits = nf;
    pk.n_groups = ng;
    pk.theta_len = P->TL;
    pk.pq = P->PQ;
    pk.stride = stride;
    pk.series = P->d_series;
    pk.g_series = P->d_g_series;
    pk.f_group = P->d_f_group;
    pk.f_user = P->d_f_user;
    pk.g_user = P->d_g_user;
    pk.theta = P->d_theta;
    pk.lik = P->d_lik;
    pk.iters = P->d_ne;
    pk.status = P->d_status;
    pk.best = P->d_best;
    pk.theta_u = d_theta_u;
    pk.lik_u = d_lik_u;
    pk.iters_u = d_int;
    pk.status_u = d_int + nf;
    pk.best_u = d_int + 2 * (size_t)nf;
    pack_results_kernel<<<(std::max(nf, ng) + 255) / 256, 256, 0, st>>>(pk);
    CU(cudaGetLastError());
    if (!P->h_res) CU(P->cuda.alloc_pinned(&P->h_res, P->res_total));
    const bool traj = out->X || out->Y || out->V || out->J;
    CU(cudaMemcpyAsync(P->h_res, P->d_res, (traj ? P->res_total : P->res_head) * sizeof(double),
                       cudaMemcpyDeviceToHost, st));
    std::vector<double> liks_tmp; // sharded call: the trace rows are scattered on the host
    if (out->liks) {
        if (!P->d_liks) return fail(LDSR_ERR_ARG, "liks requested at fetch but not at ldsr_plan_em time");
        double *dst = out->liks;
        if (map) {
            liks_tmp.resize((size_t)nf * P->last_niter);
            dst = liks_tmp.data();
        }
        CU(cudaMemcpyAsync(dst, P->d_liks, (size_t)nf * P->last_niter * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    CU(cudaStreamSynchronize(st));
    const double *h_theta = P->h_res, *h_lik = h_theta + (size_t)nf * stride;
    const int *h_int = reinterpret_cast<const int *>(h_lik + nf);
    if (map) {
        // straight from the pinned block into the caller's rows (no per-shard staging vectors)
        const int *h_it = h_int, *h_st = h_int + nf, *h_best = h_int + 2 * (size_t)nf;
        for (int i = 0; i < nf; i++) {
            const int f = map->fits[i];
            if (out->theta) { // the tail of a caller row beyond its series' p + q + 6 is left as the caller set it
                int w = stride;
                if (!P->same_width) {
                    const int s = P->user_fit_series[i];
                    w = P->s_p[s] + P->s_q[s] + 6;
                }
                std::memcpy(out->theta + (size_t)f * stride, h_theta + (size_t)i * stride, sizeof(double) * w);
            }
            if (out->lik) out->lik[f] = h_lik[i];
            if (out->iters) out->iters[f] = h_it[i];
            if (out->status) out->status[f] = h_st[i];
            if (out->liks)
                std::memcpy(out->liks + (size_t)f * map->niter, &liks_tmp[(size_t)i * P->last_niter],
                            sizeof(double) * P->last_niter);
        }
        const size_t tt = (size_t)P->traj_total;
        const double *h_traj = P->h_res + P->res_head;
        for (int gl = 0; gl < ng; gl++) {
            const int g = map->groups[gl];
            if (out->best) out->best[g] = h_best[gl] < 0 ? -1 : map->fits[h_best[gl]];
            const size_t n = (size_t)(P->h_traj_ptr_user[gl + 1] - P->h_traj_ptr_user[gl]) * sizeof(double);
            const size_t src = (size_t)P->h_traj_ptr_user[gl], dst = (size_t)map->traj_ptr[g];
            if (out->X) std::memcpy(out->X + dst, h_traj + src, n);
            if (out->Y) std::memcpy(out->Y + dst, h_traj + tt + src, n);
            if (out->V) std::memcpy(out->V + dst, h_traj + 2 * tt + src, n);
            if (out->J) std::memcpy(out->J + dst, h_traj + 3 * tt + src, n);
        }
        return Err();
    }
    if (out->theta) {
        if (P->same_width)
            std::memcpy(out->theta, h_theta, sizeof(double) * (size_t)nf * stride);
        else // the tail of a caller row beyond its series' p + q + 6 is left as the caller set it
            for (int fi = 0; fi < nf; fi++) {
                const int s = P->h_g_series[P->h_f_group[fi]];
                const size_t row = (size_t)P->f_user[fi] * stride;
                std::memcpy(out->theta + row, h_theta + row, sizeof(double) * (P->s_p[s] + P->s_q[s] + 6));
            }
    }
    if (out->lik) std::memcpy(out->lik, h_lik, sizeof(double) * nf);
    if (out->iters) std::memcpy(out->iters, h_int, sizeof(int) * nf);
    if (out->status) std::memcpy(out->status, h_int + nf, sizeof(int) * nf);
    if (out->best) std::memcpy(out->best, h_int + 2 * (size_t)nf, sizeof(int) * ng);
    const size_t tt = (size_t)P->traj_total, tb = tt * sizeof(double);
    const double *h_traj = P->h_res + P->res_head;
    if (out->X) std::memcpy(out->X, h_traj, tb);
    if (out->Y) std::memcpy(out->Y, h_traj + tt, tb);
    if (out->V) std::memcpy(out->V, h_traj + 2 * tt, tb);
    if (out->J) std::memcpy(out->J, h_traj + 3 * tt, tb);
    return Err();
}

// ---- sub-batch for one device: a subset of groups with their fits ---------------------------
struct SubBatch {
    ldsr_batch b;
    std::vector<int> groups; // user group ids
    std::vector<int> group_series, held_ptr, held_idx, fit_group, fits; // fits = user fit ids
    std::vector<double> theta0;
    std::vector<long long> traj_ptr; // local prefix sums of T
};

static void make_sub(const ldsr_batch *b, const std::vector<int> &groups, const std::vector<int> &fit_lo,
                     const std::vector<int> &fit_hi, SubBatch &sb) {
    sb.groups = groups;
    sb.b = *b;
    sb.held_ptr.assign(1, 0);
    sb.traj_ptr.assign(1, 0);
    for (int gl = 0; gl < (int)groups.size(); gl++) {
        const int g = groups[gl];
        sb.group_series.push_back(b->group_series[g]);
        if (b->held_ptr)
            for (int k = b->held_ptr[g]; k < b->held_ptr[g + 1]; k++) sb.held_idx.push_back(b->held_idx[k]);
        sb.held_ptr.push_back((int)sb.held_idx.size());
        sb.traj_ptr.push_back(sb.traj_ptr.back() + b->T[b->group_series[g]]);
        for (int f = fit_lo[g]; f >= 0 && f < fit_hi[g]; f++) {
            sb.fits.push_back(f);
            sb.fit_group.push_back(gl);
        }
    }
    sb.theta0.resize(sb.fits.size() * (size_t)b->theta_stride);
    for (size_t i = 0; i < sb.fits.size(); i++)
        std::memcpy(&sb.theta0[i * b->theta_stride], b->theta0 + (size_t)sb.fits[i] * b->theta_stride,
                    sizeof(double) * b->theta_stride);
    if (sb.held_idx.empty()) sb.held_idx.push_back(0);
    sb.b.n_groups = (int)groups.size();
    sb.b.group_series = sb.group_series.data();
    sb.b.held_ptr = sb.held_ptr.data();
    sb.b.held_idx = sb.held_idx.data();
    sb.b.n_fits = (int)sb.fits.size();
    sb.b.fit_group = sb.fit_group.data();
    sb.b.theta0 = sb.theta0.data();
}

// Greedy longest-processing-time partition of the groups over n_shards devices; the cost of a
// group is restarts * T * (p+q+8) (iteration counts are not known in advance).  Deterministic.
static void shard_groups(const ldsr_batch *b, int n_shards, int *group_shard) {
    const int ng = b->n_groups;
    std::vector<double> cost(ng, 0.0);
    for (int f = 0; f < b->n_fits; f++) {
        const int g = b->fit_group[f], s = b->group_series[g];
        cost[g] += (double)b->T[s] * (b->p[s] + b->q[s] + 8);
    }
    std::vector<int> order(ng);
    std::iota(order.begin(), order.end(), 0);
    std::stable_sort(order.begin(), order.end(), [&](int a, int c) { return cost[a] > cost[c]; });
    std::vector<double> load(n_shards, 0.0);
    for (int g : order) {
        const int d = (int)(std::min_element(load.begin(), load.end()) - load.begin());
        group_shard[g] = d;
        load[d] += cost[g];
    }
}

static Err em_batch(ldsr_ctx *ctx, const ldsr_batch *b, int niter, double tol, const ldsr_options *opt,
                    ldsr_em_result *out) {
    Err e = validate(b);
    if (!e.ok()) return e;
    if (!out) return fail(LDSR_ERR_ARG, "result struct is NULL");
    std::unique_ptr<ldsr_ctx> tmp_ctx;
    if (!(e = default_ctx(ctx, tmp_ctx, opt ? opt->n_devices : 0, opt ? opt->devices : nullptr)).ok()) return e;
    int nd = (int)ctx->devices.size();
    if (opt && opt->n_devices > 0) nd = std::min(nd, opt->n_devices);
    nd = std::max(1, std::min(nd, b->n_groups));
    const bool want_liks = out->liks != nullptr;

    // single device, whole batch: no sub-batch copies
    if (nd == 1) {
        // LDSR_TIMING=1 (development): wall-clock split of the host-buffer call on stderr
        static const bool timing = std::getenv("LDSR_TIMING") != nullptr;
        auto now = [] { return std::chrono::steady_clock::now(); };
        auto ms = [](std::chrono::steady_clock::time_point a, std::chrono::steady_clock::time_point c) {
            return std::chrono::duration<double, std::milli>(c - a).count();
        };
        const auto t0 = now();
        ldsr_plan *P = nullptr;
        e = plan_build(b, ctx->devices[0], ctx->pools[0].get(), &P);
        if (!e.ok()) return e;
        const auto t1 = now();
        {
            std::unique_ptr<ldsr_plan> guard(P);
            e = plan_em(P, niter, tol, opt, nullptr, want_liks, nullptr, nullptr);
            if (!e.ok()) return e;
            const auto t2 = now();
            e = plan_fetch(P, out);
            const auto t3 = now();
            guard.reset();
            if (timing)
                std::fprintf(stderr, "ldsr_em_batch: build %.3f ms, em %.3f ms, fetch %.3f ms, destroy %.3f ms\n",
                             ms(t0, t1), ms(t1, t2), ms(t2, t3), ms(t3, now()));
        }
        return e;
    }

    // ---- shard groups over devices (no data-path collective: a group's restarts stay together)
    const int ng = b->n_groups;
    std::vector<int> fit_lo, fit_hi;
    fit_ranges(b, fit_lo, fit_hi);
    {   // a group without fits costs nothing: never more shards than groups that have work, so that no
        // device is handed an empty sub-batch
        int nonempty = 0;
        for (int g = 0; g < ng; g++) nonempty += fit_lo[g] >= 0 ? 1 : 0;
        nd = std::max(1, std::min(nd, nonempty));
    }
    std::vector<int> shard(ng);
    shard_groups(b, nd, shard.data());
    std::vector<std::vector<int>> dev_groups(nd);
    for (int g = 0; g < ng; g++) dev_groups[shard[g]].push_back(g);
    std::vector<long long> traj_ptr(ng + 1, 0);
    for (int g = 0; g < ng; g++) traj_ptr[g + 1] = traj_ptr[g] + b->T[b->group_series[g]];

    // Workers never run the caller's poll callback (it belongs to the calling thread: the R shim's
    // callback enters the R API).  When the caller polls, the workers synchronise after every chunk
    // and look at abort_flag, which the calling thread raises; otherwise they enqueue the whole run.
    ldsr_options wopt;
    std::memset(&wopt, 0, sizeof wopt);
    if (opt) wopt = *opt;
    wopt.poll = nullptr;
    wopt.poll_arg = nullptr;
    if (wopt.variant == 0) { // the kernel follows the whole batch, not the shard (see plan_em, variant 6)
        const KernelTable *kt_all = kernel_table_for(input_width(b->n_series, b->u, b->v, b->p, b->q));
        if (kt_all && b->n_fits > scan_auto_fits(kt_all->pq)) wopt.variant = 6;
    }
    const bool caller_polls = opt && opt->poll;
    std::vector<SubBatch> subs(nd);
    std::vector<Err> errs(nd);
    std::atomic<int> abort_flag(0);
    std::mutex mu;
    std::condition_variable cv;
    int running = nd;
    static const bool timing = std::getenv("LDSR_TIMING") != nullptr;
    std::vector<double> dev_ms(nd, 0.0);
    std::vector<std::thread> workers;
    for (int d = 0; d < nd; d++) {
        workers.emplace_back([&, d]() {
            const auto t0 = std::chrono::steady_clock::now();
            SubBatch &sb = subs[d];
            make_sub(b, dev_groups[d], fit_lo, fit_hi, sb); // each worker packs its own share
            Err er;
            if (sb.fits.empty()) { // only groups without fits: nothing to run
                const double nan = std::nan("");
                for (int g : sb.groups) {
                    if (out->best) out->best[g] = -1;
                    for (double *rowp : {out->X, out->Y, out->V, out->J})
                        if (rowp) std::fill(rowp + traj_ptr[g], rowp + traj_ptr[g + 1], nan);
                }
            } else {
                ldsr_plan *P = nullptr;
                er = plan_build(&sb.b, ctx->devices[d], ctx->pools[d].get(), &P);
                if (er.ok()) {
                    std::unique_ptr<ldsr_plan> guard(P);
                    er = plan_em(P, niter, tol, &wopt, nullptr, want_liks, caller_polls ? &abort_flag : nullptr, nullptr);
                    if (er.ok()) {
                        FetchMap map{sb.fits.data(), sb.groups.data(), traj_ptr.data(), niter};
                        er = plan_fetch(P, out, &map);
                    }
                }
            }
            if (!er.ok()) abort_flag.store(1);
            errs[d] = er;
            dev_ms[d] = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
            {
                std::lock_guard<std::mutex> lk(mu);
                running--;
            }
            cv.notify_all();
        });
    }
    // the poll callback runs HERE, on the calling thread; completion is signalled, not polled for
    bool interrupted = false;
    {
        std::unique_lock<std::mutex> lk(mu);
        while (running > 0) {
            if (!caller_polls) {
                cv.wait(lk);
                continue;
            }
            cv.wait_for(lk, std::chrono::milliseconds(20));
            if (running > 0 && !interrupted) {
                lk.unlock();
                const bool stop = opt->poll(opt->poll_arg) != 0;
                lk.lock();
                if (stop) {
                    interrupted = true;
                    abort_flag.store(1);
                }
            }
        }
    }
    for (auto &w : workers) w.join();
    if (timing)
        for (int d = 0; d < nd; d++)
            std::fprintf(stderr, "ldsr_em_batch: device %d: %zu groups, %zu fits, %.3f ms\n", ctx->devices[d],
                         subs[d].groups.size(), subs[d].fits.size(), dev_ms[d]);
    if (interrupted) return fail(LDSR_ERR_INTERRUPTED, "interrupted by the poll callback");
    for (int d = 0; d < nd; d++)
        if (!errs[d].ok() && errs[d].code != LDSR_ERR_INTERRUPTED) return errs[d];
    for (int d = 0; d < nd; d++)
        if (!errs[d].ok()) return errs[d];
    return Err();
}

// device time (CUDA events) of the replicate kernels of the last ldsr_rep_batch* / ldsr_posterior_rep_batch /
// ldsr_posterior_stats_batch / ldsr_posterior_yearly_batch call of this thread (ldsr_last_device_ms)
static thread_local double g_last_device_ms = 0.0;

// ---- single-step batched entry points (one device: ctx device 0) ----------------------------
enum class StepKind { Smoother, Propagate };

static Err step_batch(ldsr_ctx *ctx, const ldsr_batch *b, StepKind kind, int stdlik, double *X, double *Y, double *V,
                      double *J, double *lik, double *aux = nullptr, bool rows_to_host = true) {
    if (rows_to_host && (!X || !Y || !V)) return fail(LDSR_ERR_ARG, "X, Y and V outputs are required");
    Err e = validate(b);
    if (!e.ok()) return e;
    std::unique_ptr<ldsr_ctx> tmp_ctx;
    if (!(e = default_ctx(ctx, tmp_ctx)).ok()) return e;
    ldsr_plan *P = nullptr;
    if (!(e = plan_build(b, ctx->devices[0], ctx->pools[0].get(), &P)).ok()) return e;
    std::unique_ptr<ldsr_plan> guard(P);
    Resources &cuda = P->cuda;
    const int nf = P->n_fits;
    const size_t tot = (size_t)P->fit_row_user[nf];
    double *dX, *dY, *dV, *dJ = nullptr, *dlik, *daux = nullptr;
    int *d_jt;
    long long *d_jr;
    CU(cuda.alloc(&dX, tot));
    CU(cuda.alloc(&dY, tot));
    CU(cuda.alloc(&dV, tot));
    if (J) CU(cuda.alloc(&dJ, tot));
    CU(cuda.alloc(&dlik, nf));
    if (aux) CU(cuda.alloc(&daux, nf));
    CU(cuda.upload(&d_jt, P->fit_job_theta));
    CU(cuda.upload(&d_jr, P->fit_job_row));
    const SmootherParams sp =
        smoother_params(P, nf, P->d_f_group, d_jt, d_jr, P->d_theta0, dX, dY, dV, dJ, dlik, stdlik, daux);
    CU(kind == StepKind::Smoother ? P->kt->smoother(sp, cuda.stream) : P->kt->propagate(sp, cuda.stream));
    CU(cudaStreamSynchronize(cuda.stream));
    if (rows_to_host) {
        CU(cudaMemcpy(X, dX, tot * sizeof(double), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(Y, dY, tot * sizeof(double), cudaMemcpyDeviceToHost));
        CU(cudaMemcpy(V, dV, tot * sizeof(double), cudaMemcpyDeviceToHost));
        if (J) CU(cudaMemcpy(J, dJ, tot * sizeof(double), cudaMemcpyDeviceToHost));
    }
    if (aux) {
        std::vector<double> a(nf);
        CU(cudaMemcpy(a.data(), daux, nf * sizeof(double), cudaMemcpyDeviceToHost));
        for (int fi = 0; fi < nf; fi++) aux[P->f_user[fi]] = a[fi];
    }
    if (lik) {
        std::vector<double> l(nf);
        CU(cudaMemcpy(l.data(), dlik, nf * sizeof(double), cudaMemcpyDeviceToHost));
        for (int fi = 0; fi < nf; fi++) lik[P->f_user[fi]] = l[fi];
    }
    return Err();
}

static Err mstep_batch(ldsr_ctx *ctx, const ldsr_batch *b, const double *X, const double *V, const double *J,
                       double *theta_out, int *status) {
    if (!X || !V || !J || !theta_out) return fail(LDSR_ERR_ARG, "X, V, J and theta_out are required");
    Err e = validate(b);
    if (!e.ok()) return e;
    std::unique_ptr<ldsr_ctx> tmp_ctx;
    if (!(e = default_ctx(ctx, tmp_ctx)).ok()) return e;
    ldsr_plan *P = nullptr;
    if (!(e = plan_build(b, ctx->devices[0], ctx->pools[0].get(), &P)).ok()) return e;
    std::unique_ptr<ldsr_plan> guard(P);
    Resources &cuda = P->cuda;
    const int nf = P->n_fits;
    const size_t tot = (size_t)P->fit_row_user[nf];
    double *dX, *dV, *dJ, *dth;
    int *dst;
    long long *d_fr;
    CU(cuda.alloc(&dX, tot));
    CU(cuda.alloc(&dV, tot));
    CU(cuda.alloc(&dJ, tot));
    CU(cuda.alloc(&dth, (size_t)nf * P->TL));
    CU(cuda.alloc(&dst, nf));
    CU(cuda.upload(&d_fr, P->fit_job_row));
    CU(cudaMemcpyAsync(dX, X, tot * sizeof(double), cudaMemcpyHostToDevice, cuda.stream));
    CU(cudaMemcpyAsync(dV, V, tot * sizeof(double), cudaMemcpyHostToDevice, cuda.stream));
    CU(cudaMemcpyAsync(dJ, J, tot * sizeof(double), cudaMemcpyHostToDevice, cuda.stream));
    MstepParams mp;
    mp.series = P->d_series;
    mp.blobs = P->d_blobs;
    mp.sconst = P->d_sconst;
    mp.g_series = P->d_g_series;
    mp.masks = P->d_masks;
    mp.g_mask_off = P->d_g_mask_off;
    mp.gconst = P->d_gconst;
    mp.g_status = P->d_g_status;
    mp.n_fits = nf;
    mp.f_group = P->d_f_group;
    mp.f_row = d_fr;
    mp.X = dX;
    mp.V = dV;
    mp.J = dJ;
    mp.theta_out = dth;
    mp.status = dst;
    CU(P->kt->mstep(mp, cuda.stream));
    CU(cudaStreamSynchronize(cuda.stream));
    std::vector<double> th((size_t)nf * P->TL);
    std::vector<int> stt(nf);
    CU(cudaMemcpy(th.data(), dth, th.size() * sizeof(double), cudaMemcpyDeviceToHost));
    CU(cudaMemcpy(stt.data(), dst, nf * sizeof(int), cudaMemcpyDeviceToHost));
    for (int fi = 0; fi < nf; fi++) {
        const int s = P->h_g_series[P->h_f_group[fi]];
        unpad_theta(&th[(size_t)fi * P->TL], P->s_p[s], P->s_q[s], P->h_series[s].has_u != 0,
                    P->h_series[s].has_v != 0, P->PQ, theta_out + (size_t)P->f_user[fi] * P->theta_stride);
        if (status) status[P->f_user[fi]] = stt[fi];
    }
    return Err();
}

// The output pipeline of the replicate entry points.  Up to three outputs (simX, simY, simQ; null ones are
// skipped) of lo.back() doubles each live in the caller's (pageable) memory.  Chunk c covers elements
// lo[c] .. lo[c+1]-1 of every output and elements zlo[c] .. zlo[c+1]-1 of the noise (caller noise z on the host,
// or z_dev already on the device).  One pass: the kernel of chunk c+1 runs while chunk c crosses PCIe into a
// pinned slot and chunk c-1 is copied from its slot into the caller's arrays by host threads.
// `launch(c, z, out)` enqueues chunk c's kernel on run.stream (c = -1: one launch for every chunk), reading noise
// from z (the chunk's first element on the device, or null) and writing output k from out[k] (the chunk's first
// element).  Every producer the kernels depend on is on run.stream too, and the device blocks come from `run`.
// g_last_device_ms is the time of every piece of work timed on `run`: the caller's and the kernels.
struct RepOutputs {
    double *outs[3];
    std::vector<size_t> lo, zlo;
    const double *z = nullptr, *z_dev = nullptr;
};
using RepLaunch = std::function<Err(int c, const double *zdev, double *const *out)>;

static Err rep_pipeline(Resources &run, const RepOutputs &R, const RepLaunch &launch) {
    double *const *outs = R.outs;
    const cudaStream_t sk = run.stream;
    int n_out = 0;
    for (int o = 0; o < 3; o++) n_out += outs[o] ? 1 : 0;
    g_last_device_ms = 0.0;
    if (n_out == 0) {
        CU(run.total_ms(&g_last_device_ms));
        return Err();
    }
    const int n_chunks = (int)R.lo.size() - 1;
    size_t chunk = 0, zchunk = 0;
    for (int c = 0; c < n_chunks; c++) {
        chunk = std::max(chunk, R.lo[c + 1] - R.lo[c]);
        if (R.z) zchunk = std::max(zchunk, R.zlo[c + 1] - R.zlo[c]);
    }
    const size_t tot = R.lo[n_chunks], ztot = R.z ? R.zlo[n_chunks] : 0;
    // When the whole output fits comfortably in HBM (up to 8 GB here) ONE kernel simulates every replicate --
    // 782 CTAs for 100 000 replicates instead of 58 per chunk, each warp's 813-step chain hidden behind the
    // others -- and only the copies are chunked.  Otherwise kernel and copies are chunked alike.
    // (LDSR_REP_CHUNKED=1, development / tests: take the chunked path whatever the size)
    static const bool force_chunked = std::getenv("LDSR_REP_CHUNKED") != nullptr;
    const bool whole = !force_chunked && ((size_t)n_out * tot + ztot) * 8 <= ((size_t)8 << 30);
    const size_t slot_doubles = (size_t)n_out * chunk;
    double *d_whole = nullptr;
    constexpr int SLOTS = 2;
    double *d_out[SLOTS] = {nullptr, nullptr}, *h_out[SLOTS] = {nullptr, nullptr}, *d_z[SLOTS] = {nullptr, nullptr};
    cudaEvent_t ev_k[SLOTS] = {nullptr, nullptr}, ev_c[SLOTS] = {nullptr, nullptr};
    // the copy stream with its pinned slots and events (given back once the copy stream is idle; the device
    // blocks stay with `run` until run.stream is)
    Resources copy(run.pool());
    CU(copy.borrow_stream());
    const cudaStream_t sc = copy.stream;
    for (int i = 0; i < SLOTS && i < n_chunks; i++) {
        if (!whole) CU(run.alloc(&d_out[i], slot_doubles));
        CU(copy.alloc_pinned(&h_out[i], slot_doubles));
        if (R.z && !whole) CU(run.alloc(&d_z[i], zchunk));
        CU(copy.event(&ev_k[i], cudaEventDisableTiming));
        CU(copy.event(&ev_c[i], cudaEventDisableTiming));
    }
    auto copy_out = [&](int c) { // pinned slot -> the caller's arrays, a few host threads
        const int slot = c % SLOTS;
        const size_t bytes = (R.lo[c + 1] - R.lo[c]) * 8;
        std::vector<std::thread> th;
        int k = 0;
        for (int o = 0; o < 3; o++) {
            if (!outs[o]) continue;
            const char *src = reinterpret_cast<const char *>(h_out[slot] + (size_t)k * chunk);
            char *dst = reinterpret_cast<char *>(outs[o] + R.lo[c]);
            const int parts = bytes > ((size_t)4 << 20) ? 2 : 1;
            for (int pi = 0; pi < parts; pi++) {
                const size_t lo = bytes * pi / parts, hi = bytes * (pi + 1) / parts;
                th.emplace_back([=] { std::memcpy(dst + lo, src + lo, hi - lo); });
            }
            k++;
        }
        for (auto &t : th) t.join();
    };
    auto timed_launch = [&](int c, const double *zdev, double *base, size_t out_stride) -> Err {
        double *o3[3] = {nullptr, nullptr, nullptr};
        int k = 0;
        for (int o = 0; o < 3; o++)
            if (outs[o]) o3[o] = base + (size_t)(k++) * out_stride;
        CU(run.start());
        Err e = launch(c, zdev, o3);
        if (!e.ok()) return e;
        CU(run.stop());
        return Err();
    };
    if (whole) {
        CU(run.alloc(&d_whole, (size_t)n_out * tot));
        const double *zdev = R.z_dev;
        if (R.z) {
            double *dzw = nullptr;
            CU(run.alloc(&dzw, ztot));
            CU(cudaMemcpyAsync(dzw, R.z, ztot * 8, cudaMemcpyHostToDevice, sk));
            zdev = dzw;
        }
        Err e = timed_launch(-1, zdev, d_whole, tot);
        if (!e.ok()) return e;
        CU(cudaEventRecord(ev_k[0], sk));
        CU(cudaStreamWaitEvent(sc, ev_k[0], 0));
    }
    for (int c = 0; c < n_chunks; c++) {
        const int slot = c % SLOTS;
        if (c >= SLOTS) { // the slot's previous chunk must have left the device, then leave the pinned block
            CU(cudaEventSynchronize(ev_c[slot]));
            copy_out(c - SLOTS);
        }
        if (whole) { // the kernel is done (or running ahead of the copy stream's wait): only the copies are chunked
            for (int k = 0; k < n_out; k++)
                CU(cudaMemcpyAsync(h_out[slot] + (size_t)k * chunk, d_whole + (size_t)k * tot + R.lo[c],
                                   (R.lo[c + 1] - R.lo[c]) * 8, cudaMemcpyDeviceToHost, sc));
            CU(cudaEventRecord(ev_c[slot], sc));
            continue;
        }
        const double *zdev = nullptr;
        if (R.z) {
            CU(cudaMemcpyAsync(d_z[slot], R.z + R.zlo[c], (R.zlo[c + 1] - R.zlo[c]) * 8, cudaMemcpyHostToDevice, sk));
            zdev = d_z[slot];
        } else if (R.z_dev) {
            zdev = R.z_dev + R.zlo[c];
        }
        Err e = timed_launch(c, zdev, d_out[slot], chunk);
        if (!e.ok()) return e;
        CU(cudaEventRecord(ev_k[slot], sk));
        CU(cudaStreamWaitEvent(sc, ev_k[slot], 0));
        CU(cudaMemcpyAsync(h_out[slot], d_out[slot], slot_doubles * 8, cudaMemcpyDeviceToHost, sc));
        CU(cudaEventRecord(ev_c[slot], sc));
        // (the next kernel into this slot is enqueued only after the host has seen ev_c[slot], above)
    }
    for (int c = std::max(0, n_chunks - SLOTS); c < n_chunks; c++) {
        CU(cudaEventSynchronize(ev_c[c % SLOTS]));
        copy_out(c);
    }
    CU(cudaStreamSynchronize(sk));
    CU(run.total_ms(&g_last_device_ms));
    return Err();
}

static Err rep_batch(ldsr_ctx *ctx, const double *theta, const double *u, const double *v, int n, int p, int q,
                     int n_reps, const double *z, unsigned long long seed, double mu, int exp_trans, double *simX,
                     double *simY, double *simQ, const unsigned *r_seed = nullptr) {
    if (!theta || n < 1 || n_reps < 1 || p < 0 || q < 0) return fail(LDSR_ERR_ARG, "bad theta/n/n_reps/p/q");
    if (p > LDSR_MAX_PQ || q > LDSR_MAX_PQ) return fail(LDSR_ERR_UNSUPPORTED, "p or q exceeds LDSR_MAX_PQ");
    std::unique_ptr<ldsr_ctx> tmp_ctx;
    Err e = default_ctx(ctx, tmp_ctx);
    if (!e.ok()) return e;
    CU(cudaSetDevice(ctx->devices[0]));
    const int need = input_width(1, &u, &v, &p, &q);
    const KernelTable *kt = kernel_table_for(need);
    if (!kt) return fail(LDSR_ERR_UNSUPPORTED, "input width %d has no kernel instantiation", need);
    const int PQ = kt->pq;
    std::vector<double> th(2 * PQ + 6), up((size_t)n * PQ, 0.0), vp((size_t)n * PQ, 0.0);
    pad_theta(theta, p, q, u != nullptr, v != nullptr, PQ, th.data());
    for (int t = 0; t < n; t++) {
        if (u)
            for (int j = 0; j < p; j++) up[(size_t)t * PQ + j] = u[(size_t)t * p + j];
        if (v)
            for (int j = 0; j < q; j++) vp[(size_t)t * PQ + j] = v[(size_t)t * q + j];
    }
    Resources run(ctx->pools[0].get());
    CU(run.borrow_stream());
    double *dth, *du, *dv, *dz_all = nullptr;
    CU(run.upload(&dth, th));
    CU(run.upload(&du, up));
    CU(run.upload(&dv, vp));
    const size_t zrow = 1 + 2 * (size_t)n;
    if (r_seed) { // the reference's own stream: set.seed(*r_seed); rnorm(...) in replicate order, made on the device
        const long long nz = (long long)n_reps * (long long)zrow;
        CU(run.alloc(&dz_all, (size_t)nz));
        CU(r_rnorm_device(*r_seed, nz, dz_all, run.stream));
    }
    // ~48 MB per output and chunk, a multiple of a CTA's 128 replicates (at T = 813: 58 CTAs per launch)
    int chunk = (int)std::max<size_t>(128, ((size_t)48 << 20) / ((size_t)n * 8));
    chunk = std::min(n_reps, (chunk + 127) / 128 * 128);
    RepOutputs R{{simX, simY, simQ}, {}, {}, z, dz_all};
    for (int r0 = 0;; r0 = std::min(n_reps, r0 + chunk)) {
        R.lo.push_back((size_t)r0 * n);
        R.zlo.push_back((size_t)r0 * zrow);
        if (r0 == n_reps) break;
    }
    return rep_pipeline(run, R, [&](int c, const double *zdev, double *const *o3) -> Err {
        const int r0 = c < 0 ? 0 : c * chunk;
        RepParams rp;
        rp.theta = dth;
        rp.u = du;
        rp.v = dv;
        rp.z = zdev;
        rp.seed = seed;
        rp.n = n;
        rp.n_reps = c < 0 ? n_reps : std::min(chunk, n_reps - r0);
        rp.rep0 = r0;
        rp.mu = mu;
        rp.exp_trans = exp_trans;
        rp.simX = o3[0];
        rp.simY = o3[1];
        rp.simQ = o3[2];
        CU(kt->rep(rp, run.stream));
        return Err();
    });
}

// ---- replicates conditioned on the observed record (forward filtering, backward sampling) -----
// The argument checks of the conditioned replicates (no device touched) and the per-fit table C, sqrt(R), mu, lambda.
static Err posterior_args(const ldsr_batch *b, int n_reps, const double *mu, int transform, const double *lambda,
                          std::vector<double> &par) {
    Err e = validate(b);
    if (!e.ok()) return e;
    if (n_reps < 1) return fail(LDSR_ERR_ARG, "n_reps=%d, need n_reps >= 1", n_reps);
    if (transform < 0 || transform > 2) return fail(LDSR_ERR_ARG, "transform=%d, need 0 (none), 1 (log) or 2 (Box-Cox)", transform);
    if (transform == 2 && !lambda) return fail(LDSR_ERR_ARG, "transform 2 (Box-Cox) needs lambda");
    const int nf = b->n_fits;
    par.assign((size_t)4 * nf, 0.0);
    for (int f = 0; f < nf; f++) {
        const int s = b->group_series[b->fit_group[f]];
        const double *th = b->theta0 + (size_t)f * b->theta_stride;
        const double R = th[3 + b->p[s] + b->q[s]];
        if (!(R >= 0.0)) return fail(LDSR_ERR_ARG, "fit %d: R=%g, need R >= 0", f, R);
        par[4 * f] = th[1 + b->p[s]];
        par[4 * f + 1] = std::sqrt(R);
        par[4 * f + 2] = mu ? mu[f] : 0.0;
        par[4 * f + 3] = transform == 2 ? lambda[f] : 0.0;
    }
    return Err();
}

// The device half of the set-up both conditioned-replicate entry points share: the plan, the backward-sampling
// coefficient rows (smoother_kernel's coefficient mode, timed on the plan's Resources), and every PostRepParams
// field but the launch range, the noise and the outputs.
struct PosteriorSetup {
    std::unique_ptr<ldsr_ctx> tmp_ctx;
    std::unique_ptr<ldsr_plan> plan;
    PostRepParams pp{};
    std::vector<long long> fit_ptr; // user order, as ldsr_smoother_batch's rows
};

static Err posterior_setup(ldsr_ctx *ctx, const ldsr_batch *b, int n_reps, unsigned long long seed, int transform,
                           const std::vector<double> &par, PosteriorSetup &S) {
    Err e = default_ctx(ctx, S.tmp_ctx);
    if (!e.ok()) return e;
    ldsr_plan *P = nullptr;
    if (!(e = plan_build(b, ctx->devices[0], ctx->pools[0].get(), &P)).ok()) return e;
    S.plan.reset(P);
    Resources &cuda = P->cuda;
    const int nf = b->n_fits;
    // per USER fit: its group's first mask word
    std::vector<long long> f_mask_off(nf);
    for (int fi = 0; fi < nf; fi++) f_mask_off[P->f_user[fi]] = P->h_g_mask_off[P->h_f_group[fi]];
    S.fit_ptr = P->fit_row_user;
    const size_t tot = (size_t)S.fit_ptr[nf];
    double *dm, *dO, *ds, *dJ, *d_par;
    int *d_jt;
    long long *d_jr, *d_fit_ptr, *d_fmo;
    CU(cuda.alloc(&dm, tot));
    CU(cuda.alloc(&dO, tot));
    CU(cuda.alloc(&ds, tot));
    CU(cuda.alloc(&dJ, tot));
    CU(cuda.upload(&d_jt, P->fit_job_theta));
    CU(cuda.upload(&d_jr, P->fit_job_row));
    CU(cuda.upload(&d_fit_ptr, S.fit_ptr));
    CU(cuda.upload(&d_fmo, f_mask_off));
    CU(cuda.upload(&d_par, par));
    // the coefficient rows (user order, as ldsr_smoother_batch): m, o, s, J
    const SmootherParams sp =
        smoother_params(P, nf, P->d_f_group, d_jt, d_jr, P->d_theta0, dm, dO, ds, dJ, nullptr, 0, nullptr);
    CU(cuda.start()); // the coefficient pass counts as device time too
    CU(P->kt->smoother_coef(sp, cuda.stream));
    CU(cuda.stop());
    PostRepParams &pp = S.pp;
    pp.m = dm;
    pp.o = dO;
    pp.s = ds;
    pp.J = dJ;
    pp.fit_ptr = d_fit_ptr;
    pp.par = d_par;
    pp.masks = P->d_masks;
    pp.f_mask_off = d_fmo;
    pp.seed = seed;
    pp.n_reps = n_reps;
    pp.wpf = (n_reps + 31) / 32; // warps: (fit, 32 replicates) blocks in output order
    pp.transform = transform;
    return Err();
}

static Err posterior_rep_batch(ldsr_ctx *ctx, const ldsr_batch *b, int n_reps, const double *z,
                               unsigned long long seed, const double *mu, int transform, const double *lambda,
                               double *simX, double *simY, double *simQ) {
    std::vector<double> par;
    Err e = posterior_args(b, n_reps, mu, transform, lambda, par);
    if (!e.ok()) return e;
    PosteriorSetup S;
    if (!(e = posterior_setup(ctx, b, n_reps, seed, transform, par, S)).ok()) return e;
    const int nf = b->n_fits;
    const std::vector<long long> &fit_ptr = S.fit_ptr;
    // a chunk is a range of whole (fit, 32 replicates) blocks (~48 MB per output)
    const int wpf = S.pp.wpf;
    const long long n_blk = (long long)nf * wpf;
    auto blk_end = [&](long long k) { // output offset just past block k
        const int f = (int)(k / wpf), r1 = std::min(n_reps, (int)(k % wpf) * 32 + 32);
        return (size_t)n_reps * fit_ptr[f] + (size_t)r1 * (fit_ptr[f + 1] - fit_ptr[f]);
    };
    const size_t chunk_target = ((size_t)48 << 20) / 8;
    std::vector<long long> cb{0};
    RepOutputs R{{simX, simY, simQ}, {0}, {0}, z, nullptr};
    for (long long k = 0; k < n_blk; k++)
        if (k == n_blk - 1 || blk_end(k) - R.lo.back() >= chunk_target) {
            cb.push_back(k + 1);
            R.lo.push_back(blk_end(k));
            R.zlo.push_back(2 * blk_end(k));
        }
    Resources &cuda = S.plan->cuda;
    return rep_pipeline(cuda, R, [&](int c, const double *zdev, double *const *o3) -> Err {
        PostRepParams pp = S.pp;
        pp.z = zdev;
        pp.blk0 = c < 0 ? 0 : cb[c];
        pp.n_blk = c < 0 ? n_blk : cb[c + 1] - cb[c];
        pp.out0 = c < 0 ? 0 : (long long)R.lo[c];
        pp.simX = o3[0];
        pp.simY = o3[1];
        pp.simQ = o3[2];
        const size_t smem = posterior_smem_bytes<REP_TT>(zdev != nullptr);
        CU(cudaFuncSetAttribute(posterior_rep_kernel<REP_TT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)posterior_smem_bytes<REP_TT>(true)));
        const int per_cta = REP_WARPS;
        posterior_rep_kernel<REP_TT><<<(unsigned)((pp.n_blk + per_cta - 1) / per_cta), REP_WARPS * 32, smem, cuda.stream>>>(pp);
        CU(cudaGetLastError());
        return Err();
    });
}

// ---- drought statistics of the conditioned replicates, reduced in the sampler's walk -------------------------
// The checks and device set-up that the statistics and the yearly calls share.
// A list of n window or run lengths: at most LDSR_STATS_MAX_WINDOWS, each 1 .. LDSR_STATS_MAX_WINDOW.
static Err posterior_lengths(const char *name, int n, const int *v) {
    if (n < 0 || n > LDSR_STATS_MAX_WINDOWS)
        return fail(LDSR_ERR_ARG, "n_%s=%d, need 0 .. %d", name, n, LDSR_STATS_MAX_WINDOWS);
    if (n > 0 && !v) return fail(LDSR_ERR_ARG, "%s is NULL", name);
    for (int k = 0; k < n; k++)
        if (v[k] < 1 || v[k] > LDSR_STATS_MAX_WINDOW)
            return fail(LDSR_ERR_ARG, "%s[%d]=%d, need 1 .. %d", name, k, v[k], LDSR_STATS_MAX_WINDOW);
    return Err();
}

// Per fit, the step range [lo, hi) (spec_range NULL: the whole series) and, when there is one, a finite threshold.
static Err posterior_ranges(const ldsr_batch *b, const int *spec_range, const double *threshold,
                            std::vector<int> &range) {
    const int nf = b->n_fits;
    range.assign((size_t)2 * nf, 0);
    for (int f = 0; f < nf; f++) {
        const int T = b->T[b->group_series[b->fit_group[f]]];
        const int lo = spec_range ? spec_range[2 * f] : 0, hi = spec_range ? spec_range[2 * f + 1] : T;
        if (!(0 <= lo && lo < hi && hi <= T))
            return fail(LDSR_ERR_ARG, "fit %d: range [%d, %d), need 0 <= lo < hi <= T = %d", f, lo, hi, T);
        if (threshold && !std::isfinite(threshold[f]))
            return fail(LDSR_ERR_ARG, "fit %d: threshold %g is not finite", f, threshold[f]);
        range[2 * f] = lo;
        range[2 * f + 1] = hi;
    }
    return Err();
}

// One launch over every (fit, 32 replicates) block: caller noise uploaded whole (the test and parity path), the
// ranges, thresholds and windows, and a Q ring of the smallest power of two >= the longest window.
static cudaError_t posterior_reduce_params(Resources &cuda, const double *z, long long n_steps,
                                           const std::vector<int> &range, const double *threshold, int nw,
                                           const int *windows, PostRepParams &pp) {
    const int nf = (int)(range.size() / 2);
    pp.blk0 = 0;
    pp.n_blk = (long long)nf * pp.wpf;
    pp.out0 = 0;
    cudaError_t ce = cudaSuccess;
    if (z) {
        double *dz;
        const size_t nz = 2 * (size_t)pp.n_reps * (size_t)n_steps;
        if ((ce = cuda.alloc(&dz, nz)) != cudaSuccess) return ce;
        if ((ce = cudaMemcpyAsync(dz, z, nz * sizeof(double), cudaMemcpyHostToDevice, cuda.stream)) != cudaSuccess)
            return ce;
        pp.z = dz;
    }
    pp.n_win = nw;
    int wmax = 0;
    for (int k = 0; k < nw; k++) wmax = std::max(wmax, pp.win[k] = windows[k]);
    pp.ring = 1;
    while (pp.ring < wmax) pp.ring *= 2;
    if (nw == 0) pp.ring = 0;
    int *d_range;
    if ((ce = cuda.upload(&d_range, range)) != cudaSuccess) return ce;
    pp.range = d_range;
    if (threshold) {
        double *d_thr;
        if ((ce = cuda.upload(&d_thr, std::vector<double>(threshold, threshold + nf))) != cudaSuccess) return ce;
        pp.thr = d_thr;
    }
    return cudaSuccess;
}

// One timed launch of a reducing mode over every (fit, 32 replicates) block.
template <int MODE> static Err posterior_reduce_launch(Resources &cuda, const PostRepParams &pp) {
    const size_t smem = posterior_stats_smem_bytes<REP_TT>(pp.z != nullptr, pp.ring);
    CU(cudaFuncSetAttribute(posterior_rep_kernel<REP_TT, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)posterior_stats_smem_bytes<REP_TT>(true, POST_MAX_RING)));
    CU(cuda.start());
    posterior_rep_kernel<REP_TT, MODE>
        <<<(unsigned)((pp.n_blk + REP_WARPS - 1) / REP_WARPS), REP_WARPS * 32, smem, cuda.stream>>>(pp);
    CU(cudaGetLastError());
    CU(cuda.stop());
    return Err();
}

// The one launch of a reducing mode, the copies of its outputs into the caller's arrays, and the device time.
template <int MODE>
static Err posterior_reduce_run(Resources &cuda, const PostRepParams &pp,
                                const std::vector<std::function<cudaError_t()>> &copies) {
    Err e = posterior_reduce_launch<MODE>(cuda, pp);
    if (!e.ok()) return e;
    for (auto &c : copies) CU(c());
    CU(cudaStreamSynchronize(cuda.stream));
    g_last_device_ms = 0.0;
    CU(cuda.total_ms(&g_last_device_ms));
    return Err();
}

static Err posterior_stats_batch(ldsr_ctx *ctx, const ldsr_batch *b, int n_reps, const double *z,
                                 unsigned long long seed, const double *mu, int transform, const double *lambda,
                                 const ldsr_stats_spec *spec, const ldsr_stats_out *out) {
    std::vector<double> par;
    Err e = posterior_args(b, n_reps, mu, transform, lambda, par);
    if (!e.ok()) return e;
    if (!spec || !out) return fail(LDSR_ERR_ARG, "spec and out are required");
    const int nw = spec->n_windows, nf = b->n_fits;
    if (!(e = posterior_lengths("windows", nw, spec->windows)).ok()) return e;
    if (nw == 0 && !spec->threshold) return fail(LDSR_ERR_ARG, "no statistics asked for: no window and no threshold");
    if (!spec->threshold && (out->run_len || out->run_at || out->deficit || out->deficit_at || out->n_runs))
        return fail(LDSR_ERR_ARG, "run outputs need a threshold");
    std::vector<int> range;
    if (!(e = posterior_ranges(b, spec->range, spec->threshold, range)).ok()) return e;
    PosteriorSetup S;
    if (!(e = posterior_setup(ctx, b, n_reps, seed, transform, par, S)).ok()) return e;
    Resources &cuda = S.plan->cuda;
    const long long rows = (long long)nf * n_reps, wrows = rows * nw;
    PostRepParams pp = S.pp;
    CU(posterior_reduce_params(cuda, z, S.fit_ptr[nf], range, spec->threshold, nw, spec->windows, pp));
    pp.n_rows = rows;
    // device outputs of the requested statistics, copied into the caller's arrays once the kernel is done
    std::vector<std::function<cudaError_t()>> copies;
    auto out_block = [&](auto **dev, auto *host, long long n) -> cudaError_t {
        *dev = nullptr;
        if (!host) return cudaSuccess;
        cudaError_t ce = cuda.alloc(dev, (size_t)n);
        if (ce == cudaSuccess) {
            auto *d = *dev;
            copies.push_back([=, &cuda] {
                return cudaMemcpyAsync(host, d, (size_t)n * sizeof(*host), cudaMemcpyDeviceToHost, cuda.stream);
            });
        }
        return ce;
    };
    CU(out_block(&pp.wmin, out->wmin, wrows));
    CU(out_block(&pp.wmin_at, out->wmin_at, wrows));
    CU(out_block(&pp.wmax, out->wmax, wrows));
    CU(out_block(&pp.wmax_at, out->wmax_at, wrows));
    CU(out_block(&pp.run_len, out->run_len, rows));
    CU(out_block(&pp.run_at, out->run_at, rows));
    CU(out_block(&pp.deficit, out->deficit, rows));
    CU(out_block(&pp.deficit_at, out->deficit_at, rows));
    CU(out_block(&pp.n_runs, out->n_runs, rows));
    return posterior_reduce_run<POST_STATS>(cuda, pp, copies);
}

// ---- year-by-year drought counts of the conditioned replicates, reduced across replicates --------------------
static Err posterior_yearly_batch(ldsr_ctx *ctx, const ldsr_batch *b, int n_reps, const double *z,
                                  unsigned long long seed, const double *mu, int transform, const double *lambda,
                                  const ldsr_yearly_spec *spec, const ldsr_yearly_out *out) {
    std::vector<double> par;
    Err e = posterior_args(b, n_reps, mu, transform, lambda, par);
    if (!e.ok()) return e;
    if (!spec || !out) return fail(LDSR_ERR_ARG, "spec and out are required");
    const int nw = spec->n_windows, nl = spec->n_lengths, nf = b->n_fits;
    if (!(e = posterior_lengths("windows", nw, spec->windows)).ok()) return e;
    if (!(e = posterior_lengths("lengths", nl, spec->lengths)).ok()) return e;
    if (!spec->threshold) return fail(LDSR_ERR_ARG, "threshold is required");
    std::vector<int> range;
    if (!(e = posterior_ranges(b, spec->range, spec->threshold, range)).ok()) return e;
    PosteriorSetup S;
    if (!(e = posterior_setup(ctx, b, n_reps, seed, transform, par, S)).ok()) return e;
    Resources &cuda = S.plan->cuda;
    const long long ns = S.fit_ptr[nf];
    PostRepParams pp = S.pp;
    CU(posterior_reduce_params(cuda, z, ns, range, spec->threshold, nw, spec->windows, pp));
    pp.n_len = nl;
    for (int k = 0; k < nl; k++) pp.delay = std::max(pp.delay, pp.len[k] = spec->lengths[k]);
    pp.n_steps = ns;
    // the counts start at 0 on the steps that have them (window k: starts lo .. hi - w) and -1 elsewhere; the
    // kernel adds to them, and they are copied into the caller's arrays once it is done
    std::vector<std::function<cudaError_t()>> copies;
    auto out_block = [&](int **dev, int *host, int n, const int *w) -> cudaError_t {
        *dev = nullptr;
        if (!host) return cudaSuccess;
        std::vector<int> init((size_t)n * ns, -1);
        for (int k = 0; k < n; k++)
            for (int f = 0; f < nf; f++) {
                const long long hi = range[2 * f + 1] - (w ? w[k] - 1 : 0);
                for (long long t = range[2 * f]; t < hi; t++) init[(size_t)(k * ns + S.fit_ptr[f] + t)] = 0;
            }
        cudaError_t ce = cuda.upload(dev, init);
        if (ce == cudaSuccess) {
            int *d = *dev;
            const size_t bytes = init.size() * sizeof(int);
            copies.push_back([=, &cuda] { return cudaMemcpyAsync(host, d, bytes, cudaMemcpyDeviceToHost, cuda.stream); });
        }
        return ce;
    };
    CU(out_block(&pp.y_below, out->below, 1, nullptr));
    CU(out_block(&pp.y_in_run, out->in_run, nl, nullptr));
    CU(out_block(&pp.y_wbelow, out->wbelow, nw, spec->windows));
    CU(out_block(&pp.y_nonfinite, out->nonfinite, 1, nullptr));
    return posterior_reduce_run<POST_YEARLY>(cuda, pp, copies);
}

// ---- per-step quantiles of w-step means over the conditioned replicates, selected exactly -----------------------
// The sampler draws the same values on every run, so the selection takes passes instead of storing the values: a
// range pass (count, smallest and largest key per slot), then selection passes until no level is active, each
// followed by quant_bracket_kernel<>.  Each histogram pass removes log2(bins) bits of a bracket's span, so a level is
// settled after at most ceil(64 / log2(bins)) of them and one collecting pass.
static Err posterior_quantile_batch(ldsr_ctx *ctx, const ldsr_batch *b, int n_reps, const double *z,
                                    unsigned long long seed, const double *mu, int transform, const double *lambda,
                                    const ldsr_quant_spec *spec, const ldsr_quant_out *out) {
    std::vector<double> par;
    Err e = posterior_args(b, n_reps, mu, transform, lambda, par);
    if (!e.ok()) return e;
    if (!spec || !out) return fail(LDSR_ERR_ARG, "spec and out are required");
    const int nw = spec->n_windows, nl = spec->n_levels, nf = b->n_fits;
    if (!(e = posterior_lengths("windows", nw, spec->windows)).ok()) return e;
    if (nw == 0) return fail(LDSR_ERR_ARG, "n_windows=0, need at least one window");
    if (nl < 1 || nl > LDSR_QUANT_MAX_LEVELS)
        return fail(LDSR_ERR_ARG, "n_levels=%d, need 1 .. %d", nl, LDSR_QUANT_MAX_LEVELS);
    if (!spec->levels) return fail(LDSR_ERR_ARG, "levels is NULL");
    for (int l = 0; l < nl; l++) {
        const double p = spec->levels[l];
        if (!(p >= 0.0 && p <= 1.0)) return fail(LDSR_ERR_ARG, "levels[%d]=%g, need 0 <= p <= 1", l, p);
        if (l > 0 && !(p > spec->levels[l - 1]))
            return fail(LDSR_ERR_ARG, "levels[%d]=%g, need strictly increasing levels", l, p);
    }
    if (!out->q && !out->nonfinite && !out->passes) return fail(LDSR_ERR_ARG, "no output asked for");
    std::vector<int> range;
    if (!(e = posterior_ranges(b, spec->range, nullptr, range)).ok()) return e;
    PosteriorSetup S;
    if (!(e = posterior_setup(ctx, b, n_reps, seed, transform, par, S)).ok()) return e;
    Resources &cuda = S.plan->cuda;
    const long long ns = S.fit_ptr[nf], n_slots = nw * ns;
    PostRepParams pp = S.pp;
    CU(posterior_reduce_params(cuda, z, ns, range, nullptr, nw, spec->windows, pp));
    pp.n_steps = ns;
    pp.n_lev = nl;
    // bins of a histogram and most values of a collected bracket (LDSR_QUANT_TINY=1, tests: 4 and 3, which takes
    // every path of the selection at a few replicates)
    static const bool tiny = std::getenv("LDSR_QUANT_TINY") != nullptr;
    QuantParams Q{};
    Q.n_slots = n_slots;
    Q.n_steps = ns;
    Q.n_lev = nl;
    Q.nb_log2 = tiny ? 2 : 11;
    Q.cap = tiny ? 3 : QUANT_MAX_CAP;
    Q.n_reps = n_reps;
    for (int l = 0; l < nl; l++) Q.lev[l] = spec->levels[l];
    // values per slot: 0 where the slot has values (starts lo .. hi - w), -1 elsewhere
    std::vector<int> n0((size_t)n_slots, -1);
    for (int k = 0; k < nw; k++)
        for (int f = 0; f < nf; f++)
            for (long long t = range[2 * f]; t <= range[2 * f + 1] - spec->windows[k]; t++)
                n0[(size_t)(k * ns + S.fit_ptr[f] + t)] = 0;
    unsigned long long *d_min, *d_max, *d_ctr;
    double *d_q;
    int *d_nonfinite;
    CU(cuda.upload(&pp.q_n, n0));
    CU(cuda.alloc(&d_min, n_slots));
    CU(cuda.alloc(&d_max, n_slots));
    CU(cuda.alloc(&Q.lv, (size_t)n_slots * nl));
    CU(cuda.alloc(&Q.br, (size_t)n_slots * nl));
    CU(cuda.alloc(&Q.slot_nbr, n_slots));
    CU(cuda.alloc(&Q.slot_br, (size_t)n_slots * nl));
    CU(cuda.alloc(&d_ctr, 4));
    CU(cuda.alloc(&d_q, (size_t)n_slots * nl));
    CU(cuda.alloc(&d_nonfinite, n_slots));
    CU(cudaMemsetAsync(d_min, 0xFF, n_slots * sizeof(unsigned long long), cuda.stream));
    CU(cudaMemsetAsync(d_max, 0, n_slots * sizeof(unsigned long long), cuda.stream));
    CU(cudaMemsetAsync(d_ctr, 0xFF, 4 * sizeof(unsigned long long), cuda.stream));
    pp.q_min = d_min;
    pp.q_max = d_max;
    pp.q_slot_nbr = Q.slot_nbr;
    pp.q_slot_br = Q.slot_br;
    pp.q_br = Q.br;
    Q.n = pp.q_n;
    Q.kmin = d_min;
    Q.kmax = d_max;
    Q.ctr = d_ctr;
    Q.q = d_q;
    Q.nonfinite = d_nonfinite;
    const unsigned slot_grid = (unsigned)((n_slots + 255) / 256);
    auto small = [&](void (*kernel)(QuantParams), unsigned grid, unsigned block) -> Err {
        CU(cuda.start());
        kernel<<<grid, block, 0, cuda.stream>>>(Q);
        CU(cudaGetLastError());
        CU(cuda.stop());
        return Err();
    };
    pp.qpass = QUANT_RANGE;
    if (!(e = posterior_reduce_launch<POST_QUANT>(cuda, pp)).ok()) return e;
    int passes = 1;
    if (!(e = small(quant_init_kernel<>, slot_grid, 256)).ok()) return e;
    // the histograms and the segments, grown when a pass needs more
    unsigned *d_hist = nullptr;
    unsigned long long *d_seg = nullptr;
    size_t hist_cap = 0, seg_cap = 0;
    const int max_passes = 2 + (64 + Q.nb_log2 - 1) / Q.nb_log2;
    for (;;) {
        CU(cudaMemsetAsync(d_ctr, 0, 3 * sizeof(unsigned long long), cuda.stream));
        if (!(e = small(quant_plan_kernel<>, slot_grid, 256)).ok()) return e;
        unsigned long long h[4];
        CU(cudaMemcpyAsync(h, d_ctr, sizeof h, cudaMemcpyDeviceToHost, cuda.stream));
        CU(cudaStreamSynchronize(cuda.stream));
        if (h[3] != ~0ull) { // a bracket's values in the last pass were not those the pass before had counted
            const long long k = (long long)(h[3] / ns), row = (long long)(h[3] % ns);
            const int f = (int)(std::upper_bound(S.fit_ptr.begin(), S.fit_ptr.end(), row) - S.fit_ptr.begin()) - 1;
            return fail(LDSR_ERR_CUDA, "fit %d, window %d, step %lld: two sampler passes disagreed", f,
                        spec->windows[k], row - S.fit_ptr[f]);
        }
        if (h[0] == 0) break;
        if (passes >= max_passes) return fail(LDSR_ERR_CUDA, "quantile selection did not settle in %d passes", passes);
        const size_t bins = (size_t)h[1] << Q.nb_log2;
        if (bins > hist_cap) CU(cuda.realloc(&d_hist, hist_cap = bins));
        if (h[2] > seg_cap) CU(cuda.realloc(&d_seg, seg_cap = h[2]));
        if (bins) CU(cudaMemsetAsync(d_hist, 0, bins * sizeof(unsigned), cuda.stream));
        pp.qpass = QUANT_SELECT;
        pp.q_hist = d_hist;
        pp.q_seg = d_seg;
        Q.hist = d_hist;
        Q.seg = d_seg;
        if (!(e = posterior_reduce_launch<POST_QUANT>(cuda, pp)).ok()) return e;
        passes++;
        Q.n_br = (long long)h[0];
        if (!(e = small(quant_bracket_kernel<>, (unsigned)h[0], QUANT_THREADS)).ok()) return e;
    }
    if (!(e = small(quant_out_kernel<>, slot_grid, 256)).ok()) return e;
    if (out->q) CU(cudaMemcpyAsync(out->q, d_q, (size_t)n_slots * nl * sizeof(double), cudaMemcpyDeviceToHost, cuda.stream));
    if (out->nonfinite)
        CU(cudaMemcpyAsync(out->nonfinite, d_nonfinite, (size_t)n_slots * sizeof(int), cudaMemcpyDeviceToHost, cuda.stream));
    CU(cudaStreamSynchronize(cuda.stream));
    if (out->passes) *out->passes = passes;
    g_last_device_ms = 0.0;
    CU(cuda.total_ms(&g_last_device_ms));
    return Err();
}

} // namespace ldsr

// =============================================================================================
// extern "C"
// =============================================================================================
extern "C" {

int ldsr_abi_version(void) { return LDSR_ABI_VERSION; }

int ldsr_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

int ldsr_ctx_create(int n_devices, const int *devices, ldsr_ctx **out, char *errbuf, int errlen) {
    if (!out) return report(fail(LDSR_ERR_ARG, "out is NULL"), errbuf, errlen);
    if (n_devices <= 0) n_devices = std::max(1, ldsr_device_count());
    std::unique_ptr<ldsr_ctx> c(new ldsr_ctx());
    for (int i = 0; i < n_devices; i++) {
        const int d = devices ? devices[i] : i;
        Err e = check_device(d);
        if (!e.ok()) return report(e, errbuf, errlen);
        c->devices.push_back(d);
        c->pools.emplace_back(new DevicePool(d));
    }
    *out = c.release();
    return LDSR_OK;
}

void ldsr_ctx_destroy(ldsr_ctx *ctx) { delete ctx; }

long long ldsr_ctx_trim(ldsr_ctx *ctx, long long *cached_bytes) {
    long long freed = 0, kept = 0;
    if (ctx)
        for (auto &p : ctx->pools) {
            freed += (long long)p->trim();
            kept += (long long)p->cached_bytes();
        }
    if (cached_bytes) *cached_bytes = kept;
    return freed;
}

int ldsr_em_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int niter, double tol, const ldsr_options *opt,
                  ldsr_em_result *out, char *errbuf, int errlen) {
    return report(em_batch(ctx, batch, niter, tol, opt, out), errbuf, errlen);
}

int ldsr_plan_create(const ldsr_batch *batch, int device, ldsr_plan **out, char *errbuf, int errlen) {
    if (!out) return report(fail(LDSR_ERR_ARG, "out is NULL"), errbuf, errlen);
    Err e = validate(batch);
    if (e.ok()) e = plan_build(batch, device, nullptr, out);
    return report(e, errbuf, errlen);
}

int ldsr_plan_em(ldsr_plan *plan, int niter, double tol, const ldsr_options *opt, void *stream, long long *stats,
                 char *errbuf, int errlen) {
    if (!plan) return report(fail(LDSR_ERR_ARG, "plan is NULL"), errbuf, errlen);
    return report(plan_em(plan, niter, tol, opt, (cudaStream_t)stream, opt && opt->trace_liks != 0, nullptr, stats),
                  errbuf, errlen);
}

int ldsr_plan_set_theta0(ldsr_plan *plan, const double *theta0_host, char *errbuf, int errlen) {
    auto run = [&]() -> Err {
        if (!plan || !theta0_host) return fail(LDSR_ERR_ARG, "plan or theta0 is NULL");
        CU(cudaSetDevice(plan->device));
        // on the plan's stream: after the plan's own upload of theta0, and before its next ldsr_plan_em
        const std::vector<double> th0 = padded_thetas(plan, theta0_host);
        const cudaStream_t st = plan->cuda.stream;
        CU(cudaMemcpyAsync(plan->d_theta0, th0.data(), th0.size() * sizeof(double), cudaMemcpyHostToDevice, st));
        CU(cudaStreamSynchronize(st));
        return Err();
    };
    return report(run(), errbuf, errlen);
}

int ldsr_plan_fetch(ldsr_plan *plan, ldsr_em_result *out, char *errbuf, int errlen) {
    if (!plan) return report(fail(LDSR_ERR_ARG, "plan is NULL"), errbuf, errlen);
    return report(plan_fetch(plan, out), errbuf, errlen);
}

void ldsr_plan_destroy(ldsr_plan *plan) { delete plan; }

int ldsr_smoother_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int stdlik, double *X, double *Y, double *V, double *J,
                        double *lik, char *errbuf, int errlen) {
    return report(step_batch(ctx, batch, StepKind::Smoother, stdlik, X, Y, V, J, lik), errbuf, errlen);
}

int ldsr_mstep_batch(ldsr_ctx *ctx, const ldsr_batch *batch, const double *X, const double *V, const double *J,
                     double *theta_out, int *status, char *errbuf, int errlen) {
    return report(mstep_batch(ctx, batch, X, V, J, theta_out, status), errbuf, errlen);
}

int ldsr_propagate_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int stdlik, double *X, double *Y, double *V,
                         double *lik, char *errbuf, int errlen) {
    return report(step_batch(ctx, batch, StepKind::Propagate, stdlik, X, Y, V, nullptr, lik), errbuf, errlen);
}

int ldsr_rep_batch(ldsr_ctx *ctx, const double *theta, const double *u, const double *v, int n, int p, int q,
                   int n_reps, const double *z, unsigned long long seed, double mu, int exp_trans, double *simX,
                   double *simY, double *simQ, char *errbuf, int errlen) {
    return report(rep_batch(ctx, theta, u, v, n, p, q, n_reps, z, seed, mu, exp_trans, simX, simY, simQ), errbuf,
                  errlen);
}

int ldsr_rep_batch_r(ldsr_ctx *ctx, const double *theta, const double *u, const double *v, int n, int p, int q,
                     int n_reps, unsigned int r_seed, double mu, int exp_trans, double *simX, double *simY,
                     double *simQ, char *errbuf, int errlen) {
    return report(rep_batch(ctx, theta, u, v, n, p, q, n_reps, nullptr, 0ull, mu, exp_trans, simX, simY, simQ, &r_seed),
                  errbuf, errlen);
}

int ldsr_posterior_rep_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int n_reps, const double *z,
                             unsigned long long seed, const double *mu, int transform, const double *lambda,
                             double *simX, double *simY, double *simQ, char *errbuf, int errlen) {
    return report(posterior_rep_batch(ctx, batch, n_reps, z, seed, mu, transform, lambda, simX, simY, simQ), errbuf,
                  errlen);
}

int ldsr_posterior_stats_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int n_reps, const double *z,
                               unsigned long long seed, const double *mu, int transform, const double *lambda,
                               const ldsr_stats_spec *spec, const ldsr_stats_out *out, char *errbuf, int errlen) {
    return report(posterior_stats_batch(ctx, batch, n_reps, z, seed, mu, transform, lambda, spec, out), errbuf,
                  errlen);
}

int ldsr_posterior_yearly_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int n_reps, const double *z,
                                unsigned long long seed, const double *mu, int transform, const double *lambda,
                                const ldsr_yearly_spec *spec, const ldsr_yearly_out *out, char *errbuf, int errlen) {
    return report(posterior_yearly_batch(ctx, batch, n_reps, z, seed, mu, transform, lambda, spec, out), errbuf,
                  errlen);
}

int ldsr_posterior_quantile_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int n_reps, const double *z,
                                  unsigned long long seed, const double *mu, int transform, const double *lambda,
                                  const ldsr_quant_spec *spec, const ldsr_quant_out *out, char *errbuf, int errlen) {
    return report(posterior_quantile_batch(ctx, batch, n_reps, z, seed, mu, transform, lambda, spec, out), errbuf,
                  errlen);
}

struct ldsr_r_rng {
    ldsr::RMersenne g;
    explicit ldsr_r_rng(unsigned seed) : g(seed) {}
};

double ldsr_last_device_ms(void) { return g_last_device_ms; }

int ldsr_r_rng_create(unsigned int seed, ldsr_r_rng **out, char *errbuf, int errlen) {
    if (!out) return report(fail(LDSR_ERR_ARG, "out is NULL"), errbuf, errlen);
    *out = new (std::nothrow) ldsr_r_rng(seed);
    if (!*out) return report(fail(LDSR_ERR_ARG, "out of memory"), errbuf, errlen);
    return LDSR_OK;
}
int ldsr_r_rng_unif(ldsr_r_rng *rng, int n, double a, double b, double *out, char *errbuf, int errlen) {
    if (!rng || n < 0 || (n > 0 && !out)) return report(fail(LDSR_ERR_ARG, "rng / out is NULL or n < 0"), errbuf, errlen);
    for (int i = 0; i < n; i++) out[i] = a + (b - a) * rng->g.unif(); // runif.c
    return LDSR_OK;
}
int ldsr_r_rng_norm(ldsr_r_rng *rng, int n, double *out, char *errbuf, int errlen) {
    if (!rng || n < 0 || (n > 0 && !out)) return report(fail(LDSR_ERR_ARG, "rng / out is NULL or n < 0"), errbuf, errlen);
    for (int i = 0; i < n; i++) out[i] = rng->g.norm();
    return LDSR_OK;
}
int ldsr_r_rng_sample(ldsr_r_rng *rng, int n, int k, int *out, char *errbuf, int errlen) {
    if (!rng || n < 1 || k < 0 || k > n || (k > 0 && !out))
        return report(fail(LDSR_ERR_ARG, "need rng, 0 <= k <= n, n >= 1 and out"), errbuf, errlen);
    rng->g.sample_int(n, k, out);
    return LDSR_OK;
}
void ldsr_r_rng_destroy(ldsr_r_rng *rng) { delete rng; }

int ldsr_r_rnorm_device(int device, unsigned int seed, long long n, double *out, char *errbuf, int errlen) {
    auto run = [&]() -> Err {
        if (n < 1 || !out) return fail(LDSR_ERR_ARG, "need n >= 1 and out");
        Err e = use_device(device);
        if (!e.ok()) return e;
        Resources cuda;
        double *d = nullptr;
        CU(cuda.alloc(&d, (size_t)n));
        CU(r_rnorm_device(seed, n, d, 0));
        CU(cudaMemcpy(out, d, sizeof(double) * (size_t)n, cudaMemcpyDeviceToHost));
        return Err();
    };
    return report(run(), errbuf, errlen);
}

int ldsr_shard_groups(const ldsr_batch *batch, int n_shards, int *group_shard, char *errbuf, int errlen) {
    Err e = validate(batch);
    if (e.ok() && (n_shards < 1 || !group_shard)) e = fail(LDSR_ERR_ARG, "n_shards < 1 or group_shard is NULL");
    if (e.ok()) shard_groups(batch, n_shards, group_shard);
    return report(e, errbuf, errlen);
}

int ldsr_objective_batch(ldsr_ctx *ctx, const ldsr_batch *batch, int kind, double lambda, double *values, char *errbuf,
                         int errlen) {
    auto run = [&]() -> Err {
        if (!values) return fail(LDSR_ERR_ARG, "values is NULL");
        if (kind < 0 || kind > 2) return fail(LDSR_ERR_ARG, "kind must be 0 (penalized_likelihood), 1 (negLogLik) or 2 (ssqTrain)");
        if (!batch) return fail(LDSR_ERR_ARG, "batch is NULL");
        const int nf = batch->n_fits;
        std::vector<double> lik(std::max(nf, 1)), aux(std::max(nf, 1));
        Err e = step_batch(ctx, batch, kind == 0 ? StepKind::Smoother : StepKind::Propagate, kind == 0 ? 0 : 1, nullptr,
                           nullptr, nullptr, nullptr, lik.data(), aux.data(), false);
        if (!e.ok()) return e;
        for (int f = 0; f < nf; f++)
            values[f] = kind == 0 ? lik[f] - lambda * aux[f] : (kind == 1 ? -lik[f] : aux[f]);
        return Err();
    };
    return report(run(), errbuf, errlen);
}

// construct_rec over stations of different lengths (one launch); ldsr_construct_rec_batch is its one-station case.
static Err construct_rec_stations(int device, int n_stations, const int *T, const int *member_ptr, const double *X,
                                  const double *V, const double *Y, const double *C, const double *R, const double *mu,
                                  const double *lambda, int transform, double *out, double *mean) {
    if (n_stations < 1) return fail(LDSR_ERR_ARG, "need n_stations >= 1");
    if (!T || !member_ptr || !X || !V || !Y || !C || !R || !mu || !out) return fail(LDSR_ERR_ARG, "a required pointer is NULL");
    if (transform < 0 || transform > 2) return fail(LDSR_ERR_ARG, "transform must be 0 (none), 1 (log) or 2 (boxcox)");
    if (transform == 2 && !lambda) return fail(LDSR_ERR_ARG, "lambda is required with transform 2 (boxcox)");
    if (member_ptr[0] != 0) return fail(LDSR_ERR_ARG, "member_ptr[0] must be 0");
    std::vector<long long> row_off(n_stations), t_off(n_stations);
    std::vector<double> lam(n_stations, 0.0);
    long long rows = 0, years = 0;
    int max_T = 0;
    for (int s = 0; s < n_stations; s++) {
        if (T[s] < 1) return fail(LDSR_ERR_ARG, "station %d: need T >= 1", s);
        if (member_ptr[s + 1] <= member_ptr[s]) return fail(LDSR_ERR_ARG, "station %d: member_ptr not increasing (every station needs a member)", s);
        row_off[s] = rows;
        t_off[s] = years;
        rows += (long long)(member_ptr[s + 1] - member_ptr[s]) * T[s];
        years += T[s];
        max_T = std::max(max_T, T[s]);
        if (lambda) lam[s] = lambda[s];
    }
    const int n = member_ptr[n_stations];
    Err e = use_device(device);
    if (!e.ok()) return e;
    const size_t nT = (size_t)rows, S = (size_t)n_stations;
    // one arena: X V Y | C R | mu lambda | out | mean | row_off t_off (8-byte integers) | T member_ptr (ints)
    const size_t n_dbl = 3 * nT + 2 * (size_t)n + 2 * S + 6 * nT + 2 * (size_t)years + 2 * S;
    Resources cuda;
    char *arena = nullptr;
    CU(cuda.alloc(&arena, sizeof(double) * n_dbl + sizeof(int) * (2 * S + 1)));
    double *d = reinterpret_cast<double *>(arena);
    double *dX = d, *dV = dX + nT, *dY = dV + nT, *dC = dY + nT, *dR = dC + n, *dmu = dR + n, *dlam = dmu + S;
    double *dO = dlam + S, *dM = dO + 6 * nT;
    long long *d_roff = reinterpret_cast<long long *>(dM + 2 * years), *d_toff = d_roff + S;
    int *d_T = reinterpret_cast<int *>(d_toff + S), *d_mp = d_T + S;
    CU(cudaMemcpy(dX, X, sizeof(double) * nT, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dV, V, sizeof(double) * nT, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dY, Y, sizeof(double) * nT, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dC, C, sizeof(double) * n, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dR, R, sizeof(double) * n, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dmu, mu, sizeof(double) * S, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(dlam, lam.data(), sizeof(double) * S, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_roff, row_off.data(), sizeof(long long) * S, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_toff, t_off.data(), sizeof(long long) * S, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_T, T, sizeof(int) * S, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_mp, member_ptr, sizeof(int) * (S + 1), cudaMemcpyHostToDevice));
    const dim3 grid((max_T + 127) / 128, std::min(n_stations, 65535));
    construct_rec_kernel<<<grid, 128>>>(n_stations, d_T, d_mp, d_roff, d_toff, dX, dV, dY, dC, dR, dmu, dlam, transform,
                                        dO, mean ? dM : nullptr);
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, dO, sizeof(double) * 6 * nT, cudaMemcpyDeviceToHost));
    if (mean) CU(cudaMemcpy(mean, dM, sizeof(double) * 2 * (size_t)years, cudaMemcpyDeviceToHost));
    return Err();
}

int ldsr_construct_rec_stations(int device, int n_stations, const int *T, const int *member_ptr, const double *X,
                                const double *V, const double *Y, const double *C, const double *R, const double *mu,
                                const double *lambda, int transform, double *out, double *mean, char *errbuf,
                                int errlen) {
    return report(construct_rec_stations(device, n_stations, T, member_ptr, X, V, Y, C, R, mu, lambda, transform, out,
                                         mean),
                  errbuf, errlen);
}

int ldsr_construct_rec_batch(int device, int n, int T, const double *X, const double *V, const double *Y,
                             const double *C, const double *R, double mu, int transform, double lambda, double *out,
                             double *mean, char *errbuf, int errlen) {
    const int member_ptr[2] = {0, n};
    return report(construct_rec_stations(device, 1, &T, member_ptr, X, V, Y, C, R, &mu, &lambda, transform, out, mean),
                  errbuf, errlen);
}

// cv metrics over stations of different lengths (one launch); ldsr_cv_metrics_batch is its one-station case.
static Err cv_metrics_stations(int device, int n_stations, const int *n, const int *fold_ptr, const double *sim,
                               const double *obs, const int *z_ptr, const int *z_idx, int exp_trans, double *out) {
    if (n_stations < 1) return fail(LDSR_ERR_ARG, "need n_stations >= 1");
    if (!n || !fold_ptr || !sim || !obs || !z_ptr || !z_idx || !out) return fail(LDSR_ERR_ARG, "a required pointer is NULL");
    if (fold_ptr[0] != 0) return fail(LDSR_ERR_ARG, "fold_ptr[0] must be 0");
    for (int s = 0; s < n_stations; s++) {
        if (n[s] < 2) return fail(LDSR_ERR_ARG, "station %d: need a target of length n >= 2", s);
        if (fold_ptr[s + 1] < fold_ptr[s]) return fail(LDSR_ERR_ARG, "fold_ptr not monotone at station %d", s);
    }
    const int n_folds = fold_ptr[n_stations];
    if (n_folds < 1) return fail(LDSR_ERR_ARG, "need n_folds >= 1");
    if (z_ptr[0] < 0) return fail(LDSR_ERR_ARG, "z_ptr[0] < 0");
    // per fold: length, offset of its station's target, offset of its sim row (= of its hold-out marks)
    std::vector<int> f_n(n_folds);
    std::vector<long long> f_obs(n_folds), f_row(n_folds);
    long long n_obs = 0, n_sim = 0;
    for (int s = 0; s < n_stations; s++) {
        for (int f = fold_ptr[s]; f < fold_ptr[s + 1]; f++) {
            f_n[f] = n[s];
            f_obs[f] = n_obs;
            f_row[f] = n_sim;
            n_sim += n[s];
        }
        n_obs += n[s];
    }
    std::vector<unsigned char> held((size_t)n_sim, 0);
    for (int f = 0; f < n_folds; f++) {
        if (z_ptr[f + 1] < z_ptr[f]) return fail(LDSR_ERR_ARG, "z_ptr not monotone at fold %d", f);
        for (int k = z_ptr[f]; k < z_ptr[f + 1]; k++) {
            const int i = z_idx[k] - 1; // R indices are 1-based
            if (i < 0 || i >= f_n[f]) return fail(LDSR_ERR_ARG, "fold %d: hold-out index %d outside 1..%d", f, z_idx[k], f_n[f]);
            held[(size_t)f_row[f] + i] = 1;
        }
    }
    Err e = use_device(device);
    if (!e.ok()) return e;
    Resources cuda;
    double *d_sim = nullptr, *d_obs = nullptr, *d_out = nullptr;
    unsigned char *d_held = nullptr;
    long long *d_off = nullptr;
    int *d_n = nullptr;
    CU(cuda.alloc(&d_sim, (size_t)n_sim));
    CU(cuda.alloc(&d_obs, (size_t)n_obs));
    CU(cuda.alloc(&d_out, (size_t)n_folds * 5));
    CU(cuda.alloc(&d_held, held.size()));
    CU(cuda.alloc(&d_off, 2 * (size_t)n_folds));
    CU(cuda.alloc(&d_n, (size_t)n_folds));
    CU(cudaMemcpy(d_sim, sim, sizeof(double) * (size_t)n_sim, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_obs, obs, sizeof(double) * (size_t)n_obs, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_held, held.data(), held.size(), cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_off, f_obs.data(), sizeof(long long) * n_folds, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_off + n_folds, f_row.data(), sizeof(long long) * n_folds, cudaMemcpyHostToDevice));
    CU(cudaMemcpy(d_n, f_n.data(), sizeof(int) * n_folds, cudaMemcpyHostToDevice));
    cv_metrics_kernel<<<(n_folds + 3) / 4, 128>>>(n_folds, d_n, d_off, d_off + n_folds, d_sim, d_obs, d_held, exp_trans,
                                                  d_out);
    CU(cudaGetLastError());
    CU(cudaMemcpy(out, d_out, sizeof(double) * (size_t)n_folds * 5, cudaMemcpyDeviceToHost));
    return Err();
}

int ldsr_cv_metrics_stations(int device, int n_stations, const int *n, const int *fold_ptr, const double *sim,
                             const double *obs, const int *z_ptr, const int *z_idx, int exp_trans, double *out,
                             char *errbuf, int errlen) {
    return report(cv_metrics_stations(device, n_stations, n, fold_ptr, sim, obs, z_ptr, z_idx, exp_trans, out), errbuf,
                  errlen);
}

int ldsr_cv_metrics_batch(int device, int n, int n_folds, const double *sim, const double *obs, const int *z_ptr,
                          const int *z_idx, int exp_trans, double *out, char *errbuf, int errlen) {
    const int fold_ptr[2] = {0, n_folds};
    return report(cv_metrics_stations(device, 1, &n, fold_ptr, sim, obs, z_ptr, z_idx, exp_trans, out), errbuf, errlen);
}

int ldsr_smoother_d_batch(int device, int d, int T, int p, int q, const double *y, const double *u, const double *v,
                          int n_fits, const double *theta, int theta_stride, int stdlik, int method, int chunk,
                          double *X, double *V, double *Y, double *lik, double *kernel_ms, char *errbuf,
                          int errlen) {
    auto run = [&]() -> Err {
        if (d < 1 || d > LDSR_MAX_STATE_DIM)
            return fail(LDSR_ERR_UNSUPPORTED, "state dimension %d outside 1..%d", d, LDSR_MAX_STATE_DIM);
        if (T < 2 || p < 0 || q < 0 || n_fits < 1) return fail(LDSR_ERR_ARG, "need T >= 2, p,q >= 0, n_fits >= 1");
        if (!y || !theta || !lik) return fail(LDSR_ERR_ARG, "y, theta and lik are required");
        if ((u && p < 1) || (v && q < 1)) return fail(LDSR_ERR_ARG, "u/v given with p/q = 0");
        const int tl = 2 * d * d + d * p + d + q + 1 + d + d * d;
        if (theta_stride < tl) return fail(LDSR_ERR_ARG, "theta_stride=%d < %d", theta_stride, tl);
        if (method != 0 && method != 1) return fail(LDSR_ERR_ARG, "method must be 0 (sequential) or 1 (scan)");
        for (int t = 0; t < T; t++)
            if (std::isinf(y[t])) return fail(LDSR_ERR_ARG, "y[%d] is +-Inf", t);
        Err e = use_device(device);
        if (!e.ok()) return e;
        ScanParams P;
        std::memset(&P, 0, sizeof P);
        P.n_fits = n_fits;
        P.T = T;
        P.p = p;
        P.q = q;
        P.stdlik = stdlik;
        P.theta_len = tl;
        if (method == 0) {
            P.L = T; // one chunk: the "down" kernels are the sequential recursion
        } else if (chunk > 0) {
            P.L = std::min(chunk, T);
        } else {
            // One CTA per fit in the scan stages (short series): chunk phases ~2 L combines deep, scan phase
            // ~2 T/(256 L) + 14: balance, power of two in 8..64.
            int L = 8;
            while (L < 64 && (long long)L * L * 256 < T) L *= 2;
            // Long series (SCAN_GROUPS CTAs per fit): the scan stages cost a few combines per chunk ELEMENT, spread
            // over the machine, the chunk phases 2 L steps of latency: L ~ 0.05 sqrt(n_fits T), the power of two
            // nearest in ratio, 4..64 (measured optima, d = 4: T = 20 000 / 100 000 / 1 000 000 with one
            // parameter set: 4-8 / 16 / 64; T = 100 000 with 8 / 32 sets: 32 / 32-64 -- profiles/scan_smoother_r02.txt)
            const double want = 0.05 * std::sqrt((double)n_fits * (double)T);
            int Lg = 4;
            while (Lg < 64 && (double)Lg * 1.41421356 < want) Lg *= 2;
            if (scan_groups_for((T + Lg - 1) / Lg) > 1) L = Lg;
            P.L = L;
        }
        P.n_chunks = (T + P.L - 1) / P.L;
        Resources cuda;
        const size_t nT = (size_t)n_fits * T, D = d, nC = (size_t)n_fits * P.n_chunks;
        double *dy = nullptr, *du = nullptr, *dv_in = nullptr, *dth = nullptr;
        CU(cuda.alloc(&dy, T));
        CU(cudaMemcpy(dy, y, sizeof(double) * T, cudaMemcpyHostToDevice));
        if (u) {
            CU(cuda.alloc(&du, (size_t)T * p));
            CU(cudaMemcpy(du, u, sizeof(double) * (size_t)T * p, cudaMemcpyHostToDevice));
        }
        if (v) {
            CU(cuda.alloc(&dv_in, (size_t)T * q));
            CU(cudaMemcpy(dv_in, v, sizeof(double) * (size_t)T * q, cudaMemcpyHostToDevice));
        }
        std::vector<double> th((size_t)n_fits * tl);
        for (int f = 0; f < n_fits; f++) std::memcpy(&th[(size_t)f * tl], theta + (size_t)f * theta_stride, sizeof(double) * tl);
        CU(cuda.alloc(&dth, th.size()));
        CU(cudaMemcpy(dth, th.data(), sizeof(double) * th.size(), cudaMemcpyHostToDevice));
        P.y = dy;
        P.u = du;
        P.v = dv_in;
        P.theta = dth;
        CU(cuda.alloc(&P.c, nT * D));
        CU(cuda.alloc(&P.dv, nT));
        CU(cuda.alloc(&P.Xu, nT * D));
        CU(cuda.alloc(&P.Vu, nT * D * D));
        CU(cuda.alloc(&P.fagg, nC * (3 * D * D + 2 * D)));
        CU(cuda.alloc(&P.sagg, nC * (2 * D * D + D)));
        CU(cuda.alloc(&P.pre, nC * (D + D * D)));
        CU(cuda.alloc(&P.suf, nC * (D + D * D)));
        CU(cuda.alloc(&P.likp, nC * 2));
        P.n_groups = scan_groups_for(P.n_chunks);
        if (const char *ev = std::getenv("LDSR_SCAN_GROUPS")) // development: 1 = one CTA per fit scans all chunks
            if (std::atoi(ev) == 1) P.n_groups = 1;
        if (P.n_groups > 1) {
            const size_t nG = (size_t)n_fits * P.n_groups;
            CU(cuda.alloc(&P.fgagg, nG * (3 * D * D + 2 * D)));
            CU(cuda.alloc(&P.fgpre, nG * (3 * D * D + 2 * D)));
            CU(cuda.alloc(&P.sgagg, nG * (2 * D * D + D)));
            CU(cuda.alloc(&P.sgsuf, nG * (2 * D * D + D)));
        }
        CU(cuda.alloc(&P.X, nT * D));
        CU(cuda.alloc(&P.V, nT * D * D));
        CU(cuda.alloc(&P.Y, nT));
        CU(cuda.alloc(&P.lik, n_fits));
        CU(cuda.start());
        CU(scan_smoother_launch(d, P, nullptr));
        CU(cuda.stop());
        float ms = 0.f;
        CU(cuda.ms(0, 0, &ms));
        CU(cudaGetLastError());
        if (kernel_ms) *kernel_ms = ms;
        CU(cudaMemcpy(lik, P.lik, sizeof(double) * n_fits, cudaMemcpyDeviceToHost));
        if (X) CU(cudaMemcpy(X, P.X, sizeof(double) * nT * D, cudaMemcpyDeviceToHost));
        if (V) CU(cudaMemcpy(V, P.V, sizeof(double) * nT * D * D, cudaMemcpyDeviceToHost));
        if (Y) CU(cudaMemcpy(Y, P.Y, sizeof(double) * nT, cudaMemcpyDeviceToHost));
        return Err();
    };
    return report(run(), errbuf, errlen);
}

int ldsr_measure_fp64_peak(int device, double *tflops, char *errbuf, int errlen) {
    auto run = [&]() -> Err {
        if (!tflops) return fail(LDSR_ERR_ARG, "tflops is NULL");
        Err e = use_device(device);
        if (!e.ok()) return e;
        cudaDeviceProp prop;
        CU(cudaGetDeviceProperties(&prop, device));
        Resources cuda;
        double *d = nullptr;
        CU(cuda.alloc(&d, 8));
        const int blocks = prop.multiProcessorCount * 2, threads = 1024, iters = 4096;
        double best = 0.0;
        for (int rep = 0; rep < 6; rep++) {
            CU(cuda.start());
            dfma_peak_kernel<<<blocks, threads>>>(d, iters, 1.0000001, 1e-9);
            CU(cuda.stop());
            float ms = 0.f;
            CU(cuda.ms(rep, rep, &ms));
            const double fl = 2.0 * 64.0 * iters * (double)blocks * threads;
            if (rep > 0) best = std::max(best, fl / (ms * 1e-3) / 1e12);
        }
        *tflops = best;
        return Err();
    };
    return report(run(), errbuf, errlen);
}

} // extern "C"
