// host_simt.h -- TEST INFRASTRUCTURE: runs the SOURCE of a CUDA kernel on the CPU, one cooperative
// coroutine (ucontext) per CUDA thread, so that the kernels' control flow, shared-memory carve-up,
// barrier placement and cross-warp exchanges can be checked here (no GPU in the build container, and
// compute-sanitizer is closed on the GPU pool).
//
//  * a CTA is run to completion before the next one starts; its threads are resumed round-robin and
//    run until their next synchronisation point (__syncthreads, a warp collective, an mbarrier wait);
//  * the ORDER in which the threads of a CTA are resumed is a parameter (forward, reverse or a seeded
//    shuffle re-drawn at every scheduling round).  A kernel whose results depend on that order has a
//    shared-memory race: two accesses to the same word that no barrier orders.  tests/test_host_simt.py
//    runs every kernel under several orders and demands bit-identical results (the racecheck stand-in);
//  * dynamic shared memory ends at an inaccessible page and starts filled with 0xFF (NaN doubles):
//    reading past the end traps, reading a word that was never written poisons the result
//    (the memcheck / initcheck stand-in).
//
// Include this header BEFORE the kernel headers, with -DLDSR_HOST_SIM.
#pragma once
#ifndef LDSR_HOST_SIM
#error "compile with -DLDSR_HOST_SIM"
#endif
#include <sys/mman.h>
#include <ucontext.h>
#include <unistd.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <random>
#include <vector>

#define __device__
#define __host__
#define __global__
#define __forceinline__ inline __attribute__((always_inline))
#define __launch_bounds__(...)
#define __align__(n) __attribute__((aligned(n)))

struct double2 {
    double x, y;
};
struct int4 {
    int x, y, z, w;
};
static inline int4 make_int4(int x, int y, int z, int w) { return int4{x, y, z, w}; }
struct hostsim_uint3 {
    unsigned x, y, z;
};

namespace hostsim {

struct Thread {
    ucontext_t ctx;
    std::vector<char> stack;
    bool done = false;
};
struct Group { // a barrier among `n` threads
    int count = 0;
    unsigned gen = 0;
};

struct State {
    ucontext_t sched;
    std::vector<Thread> threads;
    int cur = -1;
    unsigned char *dyn = nullptr;
    Group block;
    std::vector<Group> warps;
    std::vector<std::vector<unsigned long long>> xchg; // per warp, 32 slots of 8 bytes
    std::function<void()> body;
    long long yields = 0;
};
inline State &st() {
    static State s;
    return s;
}

inline void yield() {
    State &s = st();
    s.yields++;
    swapcontext(&s.threads[s.cur].ctx, &s.sched);
}
inline void sync_group(Group &g, int n) {
    const unsigned gen = g.gen;
    if (++g.count == n) {
        g.count = 0;
        g.gen++;
    } else {
        while (g.gen == gen) yield();
    }
}
inline unsigned char *dyn_smem() { return st().dyn; }

} // namespace hostsim

// the built-in variables: one CTA runs at a time on one OS thread, the scheduler sets them on resume
static hostsim_uint3 threadIdx, blockIdx, blockDim, gridDim;

namespace hostsim {

inline void trampoline() {
    State &s = st();
    s.body();
    s.threads[s.cur].done = true;
    swapcontext(&s.threads[s.cur].ctx, &s.sched);
}

// order: 0 forward, 1 reverse, >= 2 seed of a shuffle re-drawn every round
// highest_cta_first: for kernels whose CTAs wait for flags raised by higher-numbered CTAs (one CTA runs at a time)
template <class F>
void launch(unsigned grid, unsigned block, size_t smem_bytes, int order, F kernel_call, bool highest_cta_first = false) {
    State &s = st();
    const size_t page = (size_t)sysconf(_SC_PAGESIZE);
    const size_t need = (smem_bytes + 127) & ~size_t(127);
    const size_t map_len = ((need + page - 1) / page + 1) * page;
    unsigned char *base = static_cast<unsigned char *>(
        mmap(nullptr, map_len, PROT_READ | PROT_WRITE, MAP_PRIVATE | MAP_ANONYMOUS, -1, 0));
    if (base == MAP_FAILED) {
        perror("mmap");
        abort();
    }
    mprotect(base + map_len - page, page, PROT_NONE); // reading or writing past the end traps
    unsigned char *dyn = base + map_len - page - need;
    std::mt19937 rng((unsigned)order * 2654435761u + 12345u);
    gridDim = {grid, 1, 1};
    blockDim = {block, 1, 1};
    for (unsigned bi = 0; bi < grid; bi++) {
        const unsigned b = highest_cta_first ? grid - 1 - bi : bi;
        std::memset(dyn, 0xFF, need);
        s.dyn = dyn;
        s.block = Group();
        s.warps.assign((block + 31) / 32, Group());
        s.xchg.assign((block + 31) / 32, std::vector<unsigned long long>(32, 0ull));
        s.body = kernel_call;
        s.threads.clear();
        s.threads.resize(block);
        blockIdx = {b, 0, 0};
        for (unsigned t = 0; t < block; t++) {
            Thread &th = s.threads[t];
            th.stack.resize(256 * 1024);
            getcontext(&th.ctx);
            th.ctx.uc_stack.ss_sp = th.stack.data();
            th.ctx.uc_stack.ss_size = th.stack.size();
            th.ctx.uc_link = nullptr;
            makecontext(&th.ctx, (void (*)())trampoline, 0);
        }
        std::vector<int> ord(block);
        for (unsigned t = 0; t < block; t++) ord[t] = order == 1 ? (int)(block - 1 - t) : (int)t;
        for (;;) {
            if (order >= 2) std::shuffle(ord.begin(), ord.end(), rng);
            bool any = false;
            for (int t : ord) {
                if (s.threads[t].done) continue;
                any = true;
                s.cur = t;
                threadIdx = {(unsigned)t, 0, 0};
                swapcontext(&s.sched, &s.threads[t].ctx);
            }
            if (!any) break;
        }
    }
    munmap(base, map_len);
}

inline int lane_id() { return (int)(threadIdx.x & 31u); }
inline int warp_id() { return (int)(threadIdx.x >> 5); }
inline int warp_width() { // threads of this warp that exist
    const int w = warp_id(), n = (int)blockDim.x - w * 32;
    return n < 32 ? n : 32;
}
template <class T> inline T warp_exchange(T v, int src_lane) {
    static_assert(sizeof(T) <= 8, "8-byte exchange slots");
    State &s = st();
    const int w = warp_id();
    unsigned long long raw = 0;
    std::memcpy(&raw, &v, sizeof(T));
    // the built-ins must be re-read after every yield: another thread ran in between
    s.xchg[w][lane_id()] = raw;
    sync_group(s.warps[w], warp_width());
    const int w2 = warp_id();
    raw = s.xchg[w2][src_lane & 31];
    sync_group(s.warps[w2], warp_width());
    T r;
    std::memcpy(&r, &raw, sizeof(T));
    return r;
}

} // namespace hostsim

// ---- the CUDA built-ins the kernels use -----------------------------------------------------------
// NOTE: threadIdx is a global that the scheduler rewrites on every resume, so it is valid again as soon
// as a synchronising call returns.
static inline void __syncthreads() {
    hostsim::sync_group(hostsim::st().block, (int)blockDim.x);
}
static inline void __threadfence() {}
static inline int atomicAdd(int *p, int v) { // one thread runs at a time
    const int old = *p;
    *p += v;
    return old;
}
static inline void __syncwarp(unsigned = 0xffffffffu) {
    hostsim::sync_group(hostsim::st().warps[hostsim::warp_id()], hostsim::warp_width());
}
static inline unsigned __ballot_sync(unsigned, int pred) {
    unsigned out = 0;
    // 32 one-bit exchanges would be slow: exchange the predicate once, read all slots
    hostsim::State &s = hostsim::st();
    const int w = hostsim::warp_id();
    s.xchg[w][hostsim::lane_id()] = pred ? 1ull : 0ull;
    hostsim::sync_group(s.warps[w], hostsim::warp_width());
    const int w2 = hostsim::warp_id();
    for (int l = 0; l < hostsim::warp_width(); l++) out |= s.xchg[w2][l] ? (1u << l) : 0u;
    hostsim::sync_group(s.warps[w2], hostsim::warp_width());
    return out;
}
static inline int __any_sync(unsigned m, int pred) { return __ballot_sync(m, pred) != 0u; }
static inline int __all_sync(unsigned m, int pred) {
    const unsigned full = hostsim::warp_width() == 32 ? 0xffffffffu : ((1u << hostsim::warp_width()) - 1u);
    return __ballot_sync(m, pred) == full;
}
template <class T> static inline T __shfl_sync(unsigned, T v, int src) { return hostsim::warp_exchange(v, src); }
template <class T> static inline T __shfl_xor_sync(unsigned, T v, int m) {
    return hostsim::warp_exchange(v, hostsim::lane_id() ^ m);
}
template <class T> static inline T __shfl_up_sync(unsigned, T v, unsigned d) {
    const int l = hostsim::lane_id();
    const T r = hostsim::warp_exchange(v, l >= (int)d ? l - (int)d : l);
    return r;
}
template <class T> static inline T __shfl_down_sync(unsigned, T v, unsigned d) {
    const int l = hostsim::lane_id();
    return hostsim::warp_exchange(v, l + (int)d < 32 ? l + (int)d : l);
}
static inline int __double2hiint(double x) {
    unsigned long long u;
    std::memcpy(&u, &x, 8);
    return (int)(u >> 32);
}
static inline int __double2loint(double x) {
    unsigned long long u;
    std::memcpy(&u, &x, 8);
    return (int)(u & 0xffffffffull);
}
static inline double __hiloint2double(int hi, int lo) {
    const unsigned long long u = ((unsigned long long)(unsigned)hi << 32) | (unsigned)lo;
    double x;
    std::memcpy(&x, &u, 8);
    return x;
}
static inline double __longlong_as_double(long long v) {
    double x;
    std::memcpy(&x, &v, 8);
    return x;
}
static inline long long __double_as_longlong(double x) {
    long long v;
    std::memcpy(&v, &x, 8);
    return v;
}
static inline int __popc(unsigned x) { return __builtin_popcount(x); }
static inline int __clz(int x) { return x == 0 ? 32 : __builtin_clz((unsigned)x); }
static inline int __ffs(int x) { return __builtin_ffs(x); }
static inline long long clock64() { return 0; }
static inline void sincospi(double x, double *s, double *c) { // the device generator of rep_kernel (unused in z mode)
    *s = std::sin(M_PI * x);
    *c = std::cos(M_PI * x);
}
using std::max;
using std::min;
