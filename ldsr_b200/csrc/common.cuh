// common.cuh -- device-side tables, PTX helpers (mbarrier + TMA bulk copy) shared by the kernels.
#pragma once
#include <cstdint>
#ifndef LDSR_HOST_SIM
#include <cuda_runtime.h>
// shared memory declarations inside a kernel (tests/host_simt/ re-defines them to run the kernel
// source on the CPU; see LDSR_HOST_SIM below)
#define LDSR_DYN_SMEM(name) extern __shared__ __align__(128) unsigned char name[]
#define LDSR_STATIC_SMEM(type, name) __shared__ type name
#else
// TEST BUILD ONLY (tests/host_simt/host_simt.h): the kernels' source compiled by g++ and run by a
// coroutine-per-thread emulator.  Never part of the product library.
#define LDSR_DYN_SMEM(name) unsigned char *const name = ::hostsim::dyn_smem()
#define LDSR_STATIC_SMEM(type, name) static type name
// the atomics of the quantile selection (aux_kernels.cuh): one emulated thread runs at a time
static inline unsigned atomicAdd(unsigned *p, unsigned v) {
    const unsigned old = *p;
    *p += v;
    return old;
}
static inline unsigned long long atomicAdd(unsigned long long *p, unsigned long long v) {
    const unsigned long long old = *p;
    *p += v;
    return old;
}
static inline unsigned long long atomicMin(unsigned long long *p, unsigned long long v) {
    const unsigned long long old = *p;
    *p = v < old ? v : old;
    return old;
}
static inline unsigned long long atomicMax(unsigned long long *p, unsigned long long v) {
    const unsigned long long old = *p;
    *p = v > old ? v : old;
    return old;
}
#endif

// Plan-consistency checks inside the kernels (compute-sanitizer is not available on the GPU pool): always on in
// the CPU emulation (tests/host_simt), on the device only in a -DLDSR_DEBUG_CHECKS build (tools/gpu_jobs/
// debug_checks.sh runs the GPU test suite against it).  They assert, once per task, that everything the shared-
// memory carve-up was sized from on the host (units, observed-unit steps, series length, aliased scratch) holds
// for what the kernel derives on the device -- every index used afterwards is bounded by these.
#if defined(LDSR_HOST_SIM)
#define LDSR_CHECK(cond)                                                                          \
    do {                                                                                          \
        if (!(cond)) {                                                                            \
            std::fprintf(stderr, "LDSR_CHECK failed: %s (%s:%d)\n", #cond, __FILE__, __LINE__);   \
            std::abort();                                                                         \
        }                                                                                         \
    } while (0)
#elif defined(LDSR_DEBUG_CHECKS)
#include <cstdio>
#define LDSR_CHECK(cond)                                                                                          \
    do {                                                                                                          \
        if (!(cond)) {                                                                                            \
            printf("LDSR_CHECK failed: %s (%s:%d) block %d thread %d\n", #cond, __FILE__, __LINE__, (int)blockIdx.x, \
                   (int)threadIdx.x);                                                                             \
            __trap();                                                                                             \
        }                                                                                                         \
    } while (0)
#else
#define LDSR_CHECK(cond) \
    do {                 \
    } while (0)
#endif

namespace ldsr {

constexpr unsigned FULL = 0xffffffffu;
constexpr double LOG_2PI = 1.8378770664093454835606594728112; // log(2*pi), pi as in EM.cpp:3

// One (y,u,v) triple, packed in HBM as a "blob" that one TMA bulk copy moves into shared memory:
//   [ y : Ty doubles | u : T*PQ doubles, time-major, rows >= p zero | v : T*PQ (absent if same_uv) ]
// PQ is the plan-wide padded input width (template parameter of the kernels).
struct SeriesDev {
    int T;
    int p, q;            // lengths of B and D in the caller's theta
    int has_u, has_v;    // 0 = the reference's matrix(0) sentinel (EM.cpp:71,77,157,189)
    int same_uv;         // v is bit-identical to u: staged once
    int y_off, u_off, v_off; // offsets inside the blob, in doubles
    int blob_doubles;    // multiple of 2 (16-byte granularity of cp.async.bulk)
    long long blob_off;  // offset of the blob in the blob arena, in doubles (even)
    long long sconst_off; // -> TuuInv[PQ*PQ] in the constants arena
    int fit_begin, fit_end; // this series' contiguous range in the (internally sorted) fit table
    int uwin_off;        // -> this series' window Gram blocks sum_{t in window} u_t u_t' in the uwin arena
                         //    ([window][PQ*PQ] doubles, windows of SPLIT_UW steps; em_split_kernel.cuh)
};

// per-group constants (theta-independent M-step blocks, EM.cpp:158,161 restricted to the group's
// observed steps): [ Syy, n_obs, Syv[PQ], wy[PQ] = SvvInv*Syv, SvvInv[PQ*PQ] ]
__host__ __device__ inline int gconst_stride(int pq) { return 2 + 2 * pq + pq * pq; }

#ifndef LDSR_HOST_SIM
__device__ __forceinline__ unsigned smem_u32(const void *p) {
    return static_cast<unsigned>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() {
    // make the initialised barrier visible to the async (TMA) proxy
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
// TMA 1-D bulk copy global -> shared, completion signalled on an mbarrier (SASS: UBLKCP).
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, unsigned bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst_smem)),
                 "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
    unsigned ok;
    do {
        asm volatile("{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
                     "selp.u32 %0, 1, 0, p;\n\t}"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
    } while (!ok);
}

#else
// emulation: *bar counts completed phases; a wait on parity p returns once phase p has completed
__device__ __forceinline__ void mbar_init(uint64_t *bar, unsigned) { *bar = 0; }
__device__ __forceinline__ void fence_mbar_init() {}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *, unsigned) {}
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src_gmem, unsigned bytes, uint64_t *) {
    std::memcpy(dst_smem, src_gmem, bytes);
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, unsigned parity) {
    while (((*(volatile uint64_t *)bar) & 1u) == parity) ::hostsim::yield();
}
#endif

// Control block (ints) of em_split_kernel's ranked task assignment, zeroed before every launch by compact_kernel:
// [0] SMs seen, [1] CTAs that have done their share, [2 + smid] CTAs arrived on the SM, [2 + 1024 + smid] 1 + rank of the SM,
// [2 + 2048 + smid] CTAs of the SM that have done their share
constexpr int SHARE_CTL_SMS = 0, SHARE_CTL_FINISHED = 1, SHARE_CTL_SLOT = 2, SHARE_MAX_SMID = 1024,
              SHARE_CTL_RANK = SHARE_CTL_SLOT + SHARE_MAX_SMID, SHARE_CTL_DONE = SHARE_CTL_RANK + SHARE_MAX_SMID,
              SHARE_CTL_LEN = SHARE_CTL_DONE + SHARE_MAX_SMID;

// ---- hand-over of a fit's state between CTAs of one (co-resident) launch (em_split_kernel.cuh, task loop)
#ifndef LDSR_HOST_SIM
template <class T> __device__ __forceinline__ T ld_l2(const T *p) { return __ldcg(p); } // L1 is not coherent across SMs
__device__ __forceinline__ void flag_raise(int *flag, int value) {
    asm volatile("st.release.gpu.global.s32 [%0], %1;" ::"l"(flag), "r"(value) : "memory");
}
__device__ __forceinline__ void flag_wait(const int *flag, int value) {
    int v;
    for (;;) {
        asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(flag) : "memory");
        if (v == value) break;
        __nanosleep(200);
    }
}
__device__ __forceinline__ int ld_acquire(const int *p) {
    int v;
    asm volatile("ld.acquire.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ int ld_relaxed(const int *p) {
    int v;
    asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void share_trap() { __trap(); }
__device__ __forceinline__ unsigned sm_id(int /*slots_per_sm*/) {
    unsigned v;
    asm("mov.u32 %0, %%smid;" : "=r"(v));
    return v;
}
#else
template <class T> __device__ __forceinline__ T ld_l2(const T *p) { return *p; }
__device__ __forceinline__ int ld_acquire(const int *p) { return *p; }
__device__ __forceinline__ int ld_relaxed(const int *p) { return *p; }
// the emulated grid fills "SMs" of slots_per_sm CTAs in launch order: CTA b sits on SM b mod (grid / slots_per_sm)
__device__ __forceinline__ unsigned sm_id(int slots_per_sm) { return blockIdx.x % (gridDim.x / slots_per_sm); }
__device__ __forceinline__ void share_trap() { LDSR_CHECK(!"CTAs are not two per SM"); }
__device__ __forceinline__ void flag_raise(int *flag, int value) { *flag = value; }
// the emulator runs one CTA at a time, the harness the highest CTA first: the producer has always finished
__device__ __forceinline__ void flag_wait(const int *flag, int value) { LDSR_CHECK(*flag == value); }
#endif

// Stage `bytes` (multiple of 16) from global to shared with TMA bulk copies issued by one thread.
// Pieces of <= 32 KB keep each transaction well inside the mbarrier tx-count range.
__device__ __forceinline__ void stage_blob(void *dst_smem, const void *src_gmem, unsigned bytes, uint64_t *bar) {
    mbar_arrive_expect_tx(bar, bytes);
    const unsigned PIECE = 32768u;
    for (unsigned off = 0; off < bytes; off += PIECE) {
        unsigned n = bytes - off < PIECE ? bytes - off : PIECE;
        bulk_g2s(static_cast<char *>(dst_smem) + off, static_cast<const char *>(src_gmem) + off, n, bar);
    }
#ifdef LDSR_HOST_SIM
    *bar += 1; // all bytes have landed: the phase completes
#endif
}

} // namespace ldsr
