// kernels_inst.cu -- compiled once per supported padded width: nvcc -DLDSR_PQ=<n>.
// A wide PQ takes minutes to compile (fully unrolled PQ x PQ bodies), so the build may cut the
// translation unit into parts, one nvcc process each: -DLDSR_PART=0 (table + single-step kernels),
// 1, 2, 3 (lane-per-fit EM kernel, MODE 0 / 1 / 2), 4 (time-split EM kernel), 5 (wide-input EM kernel,
// PQ >= WIDE_MIN_PQ; also the small-batch scan kernel, PQ <= SCAN_MAX_PQ).  -DLDSR_NO_PART=k compiles everything but part k; without either macro everything
// is in one unit.
#include "kernel_table.h"

#ifndef LDSR_PQ
#error "compile with -DLDSR_PQ=<n>"
#endif
#ifdef LDSR_PART
#define LDSR_HAS_PART(k) (LDSR_PART == (k))
#elif defined(LDSR_NO_PART)
#define LDSR_HAS_PART(k) (LDSR_NO_PART != (k))
#else
#define LDSR_HAS_PART(k) 1
#endif

namespace ldsr {

constexpr int PQ = LDSR_PQ;
constexpr int MINB = split_minb_for(PQ);
constexpr int MINB_WIDE = 2;

// launchers: explicit specialisations, defined in the part that owns the kernel
template <int PQV, int MODE> cudaError_t chunk_prepare(size_t smem_bytes);
template <int PQV, int MODE> cudaError_t chunk_launch(const EmParams &, int, size_t, cudaStream_t);
template <int PQV, int WIDE> cudaError_t split_prepare(size_t smem_bytes);
template <int PQV, int WIDE> cudaError_t split_launch(const SplitParams &, int, size_t, cudaStream_t);
#define LDSR_DECLARE_CHUNK(M)                                                                      \
    template <> cudaError_t chunk_prepare<PQ, M>(size_t);                                          \
    template <> cudaError_t chunk_launch<PQ, M>(const EmParams &, int, size_t, cudaStream_t);
LDSR_DECLARE_CHUNK(0)
LDSR_DECLARE_CHUNK(1)
LDSR_DECLARE_CHUNK(2)
template <> cudaError_t split_prepare<PQ, 0>(size_t);
template <> cudaError_t split_prepare<PQ, 1>(size_t);
template <> cudaError_t split_launch<PQ, 0>(const SplitParams &, int, size_t, cudaStream_t);
template <> cudaError_t split_launch<PQ, 1>(const SplitParams &, int, size_t, cudaStream_t);
template <int PQV> int split_resident(size_t smem_bytes);
template <> int split_resident<PQ>(size_t);

#define LDSR_DEFINE_CHUNK(M)                                                                       \
    template <> cudaError_t chunk_prepare<PQ, M>(size_t smem_bytes) {                              \
        if (M == 0) return cudaSuccess;                                                            \
        return cudaFuncSetAttribute(em_chunk_kernel<PQ, EM_SEG, EM_WARPS, M>,                      \
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes); \
    }                                                                                              \
    template <> cudaError_t chunk_launch<PQ, M>(const EmParams &p, int n_tasks, size_t smem_bytes, \
                                                cudaStream_t st) {                                 \
        em_chunk_kernel<PQ, EM_SEG, EM_WARPS, M><<<n_tasks, EM_WARPS * 32, M == 0 ? 0 : smem_bytes, st>>>(p); \
        return cudaGetLastError();                                                                 \
    }
#if LDSR_HAS_PART(1)
LDSR_DEFINE_CHUNK(0)
#endif
#if LDSR_HAS_PART(2)
LDSR_DEFINE_CHUNK(1)
#endif
#if LDSR_HAS_PART(3)
LDSR_DEFINE_CHUNK(2)
#endif

#if LDSR_HAS_PART(4)
template <> cudaError_t split_prepare<PQ, 0>(size_t smem_bytes) {
    return cudaFuncSetAttribute(em_split_kernel<PQ, SPLIT_NW, MINB, SPLIT_MSEG, SPLIT_UW>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
}
template <> cudaError_t split_launch<PQ, 0>(const SplitParams &p, int n_tasks, size_t smem_bytes, cudaStream_t st) {
    em_split_kernel<PQ, SPLIT_NW, MINB, SPLIT_MSEG, SPLIT_UW><<<n_tasks, SPLIT_NW * 32, smem_bytes, st>>>(p);
    return cudaGetLastError();
}
// the same kernel compiled for two CTAs per SM (255 registers); identical when MINB is already 2
template <> cudaError_t split_prepare<PQ, 1>(size_t smem_bytes) {
    return cudaFuncSetAttribute(em_split_kernel<PQ, SPLIT_NW, MINB_WIDE, SPLIT_MSEG, SPLIT_UW>,
                                cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
}
template <> cudaError_t split_launch<PQ, 1>(const SplitParams &p, int n_tasks, size_t smem_bytes, cudaStream_t st) {
    if (p.flags) {
        // CTAs wait for one another (iteration-level task sharing): the grid must be co-resident, which a
        // cooperative launch guarantees (it fails instead of dead-locking when the grid does not fit)
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3((unsigned)n_tasks);
        cfg.blockDim = dim3(SPLIT_NW * 32);
        cfg.dynamicSmemBytes = smem_bytes;
        cfg.stream = st;
        cudaLaunchAttribute at;
        at.id = cudaLaunchAttributeCooperative;
        at.val.cooperative = 1;
        cfg.attrs = &at;
        cfg.numAttrs = 1;
        return cudaLaunchKernelEx(&cfg, em_split_kernel<PQ, SPLIT_NW, MINB_WIDE, SPLIT_MSEG, SPLIT_UW>, p);
    }
    em_split_kernel<PQ, SPLIT_NW, MINB_WIDE, SPLIT_MSEG, SPLIT_UW><<<n_tasks, SPLIT_NW * 32, smem_bytes, st>>>(p);
    return cudaGetLastError();
}
template <> int split_resident<PQ>(size_t smem_bytes) {
    int n = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&n, em_split_kernel<PQ, SPLIT_NW, MINB_WIDE, SPLIT_MSEG, SPLIT_UW>,
                                                      SPLIT_NW * 32, smem_bytes) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}
#endif

// wide-input kernel
template <int PQV> cudaError_t wide_prepare(size_t smem_bytes);
template <int PQV> cudaError_t wide_launch(const WideParams &, int, size_t, cudaStream_t);
template <> cudaError_t wide_prepare<PQ>(size_t);
template <> cudaError_t wide_launch<PQ>(const WideParams &, int, size_t, cudaStream_t);
#if LDSR_HAS_PART(5)
template <int PQV, bool HAVE> struct WideLaunch { // widths below WIDE_MIN_PQ have no wide-input kernel
    static cudaError_t prepare(size_t) { return cudaErrorNotSupported; }
    static cudaError_t launch(const WideParams &, int, size_t, cudaStream_t) { return cudaErrorNotSupported; }
};
template <int PQV> struct WideLaunch<PQV, true> {
    static cudaError_t prepare(size_t smem_bytes) {
        return cudaFuncSetAttribute(em_wide_kernel<PQV, WIDE_NW, WIDE_MSEG, SPLIT_UW>,
                                    cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_bytes);
    }
    static cudaError_t launch(const WideParams &p, int n_tasks, size_t smem_bytes, cudaStream_t st) {
        em_wide_kernel<PQV, WIDE_NW, WIDE_MSEG, SPLIT_UW><<<n_tasks, WIDE_NW * 32, smem_bytes, st>>>(p);
        return cudaGetLastError();
    }
};
template <> cudaError_t wide_prepare<PQ>(size_t smem_bytes) {
    return WideLaunch<PQ, (PQ >= WIDE_MIN_PQ)>::prepare(smem_bytes);
}
template <> cudaError_t wide_launch<PQ>(const WideParams &p, int n_tasks, size_t smem_bytes, cudaStream_t st) {
    return WideLaunch<PQ, (PQ >= WIDE_MIN_PQ)>::launch(p, n_tasks, smem_bytes, st);
}
#endif

// small-batch scan kernel
template <int PQV> cudaError_t scan_launch(const EmParams &, int, int, cudaStream_t);
template <> cudaError_t scan_launch<PQ>(const EmParams &, int, int, cudaStream_t);
template <int PQV> cudaError_t scan_traj_launch(const EmParams &, int, cudaStream_t);
template <> cudaError_t scan_traj_launch<PQ>(const EmParams &, int, cudaStream_t);
#if LDSR_HAS_PART(5)
template <int PQV, bool HAVE> struct ScanLaunch { // widths above SCAN_MAX_PQ have no scan kernel
    static cudaError_t launch(const EmParams &, int, int, cudaStream_t) { return cudaErrorNotSupported; }
    static cudaError_t traj(const EmParams &, int, cudaStream_t) { return cudaErrorNotSupported; }
};
template <int PQV> struct ScanLaunch<PQV, true> {
    // EMIT mode: the smoothed trajectories of p.n_jobs winners, one CTA each
    static cudaError_t traj(const EmParams &p, int steps_per_thread, cudaStream_t st) {
        const int threads = (((p.max_seg + steps_per_thread - 1) / steps_per_thread + 31) / 32) * 32;
        if (steps_per_thread == 2) {
            em_scan_kernel<PQV, 2, true><<<p.n_jobs, threads, 0, st>>>(p);
        } else if (steps_per_thread == 4) {
            if constexpr (PQV <= 4)
                em_scan_kernel<PQV, 4, true><<<p.n_jobs, threads, 0, st>>>(p);
            else
                return cudaErrorNotSupported;
        } else {
            return cudaErrorNotSupported;
        }
        return cudaGetLastError();
    }
    static cudaError_t launch(const EmParams &p, int n_tasks, int steps_per_thread, cudaStream_t st) {
        // one thread per `steps_per_thread` steps, whole warps
        const int threads = (((p.max_seg + steps_per_thread - 1) / steps_per_thread + 31) / 32) * 32;
        if (steps_per_thread == 2) {
            em_scan_kernel<PQV, 2><<<n_tasks, threads, 0, st>>>(p);
        } else if (steps_per_thread == 4) {
            if constexpr (PQV <= 4) {
                // p.mode = 1: more than two fits per SM (plan_em): the build for three CTAs per SM, if the block fits it
                if (p.mode == 1 && threads <= 128)
                    em_scan_kernel<PQV, 4, false, true><<<n_tasks, threads, 0, st>>>(p);
                else
                    em_scan_kernel<PQV, 4><<<n_tasks, threads, 0, st>>>(p);
            } else {
                return cudaErrorNotSupported; // wide inputs: two steps per thread only (registers)
            }
        } else {
            return cudaErrorNotSupported;
        }
        return cudaGetLastError();
    }
};
template <> cudaError_t scan_launch<PQ>(const EmParams &p, int n_tasks, int warps, cudaStream_t st) {
    return ScanLaunch<PQ, (PQ <= SCAN_MAX_PQ)>::launch(p, n_tasks, warps, st);
}
template <> cudaError_t scan_traj_launch<PQ>(const EmParams &p, int steps_per_thread, cudaStream_t st) {
    return ScanLaunch<PQ, (PQ <= SCAN_MAX_PQ)>::traj(p, steps_per_thread, st);
}
#endif

#if LDSR_HAS_PART(0)
namespace {

cudaError_t em_prepare(size_t smem_bytes) {
    cudaError_t e = chunk_prepare<PQ, 1>(smem_bytes);
    return e != cudaSuccess ? e : chunk_prepare<PQ, 2>(smem_bytes);
}
cudaError_t em_chunk(const EmParams &p, int n_tasks, size_t smem_bytes, cudaStream_t st) {
    if (p.mode == 2) return chunk_launch<PQ, 2>(p, n_tasks, smem_bytes, st);
    if (p.mode == 1) return chunk_launch<PQ, 1>(p, n_tasks, smem_bytes, st);
    return chunk_launch<PQ, 0>(p, n_tasks, smem_bytes, st);
}
cudaError_t em_split_prepare(size_t smem_bytes) {
    cudaError_t e = split_prepare<PQ, 0>(smem_bytes);
    return e != cudaSuccess ? e : split_prepare<PQ, 1>(smem_bytes);
}
cudaError_t em_split(const SplitParams &p, int n_tasks, size_t smem_bytes, cudaStream_t st) {
    return split_launch<PQ, 0>(p, n_tasks, smem_bytes, st);
}
cudaError_t em_split_wide(const SplitParams &p, int n_tasks, size_t smem_bytes, cudaStream_t st) {
    return split_launch<PQ, 1>(p, n_tasks, smem_bytes, st);
}
int em_split_resident(size_t smem_bytes) { return split_resident<PQ>(smem_bytes); }
cudaError_t em_wide_prepare(size_t smem_bytes) { return wide_prepare<PQ>(smem_bytes); }
cudaError_t em_wide(const WideParams &p, int n_tasks, size_t smem_bytes, cudaStream_t st) {
    return wide_launch<PQ>(p, n_tasks, smem_bytes, st);
}
cudaError_t em_scan(const EmParams &p, int n_tasks, int warps, cudaStream_t st) {
    return scan_launch<PQ>(p, n_tasks, warps, st);
}
cudaError_t em_scan_traj(const EmParams &p, int steps_per_thread, cudaStream_t st) {
    return scan_traj_launch<PQ>(p, steps_per_thread, st);
}
cudaError_t smoother(const SmootherParams &p, cudaStream_t st) {
    smoother_kernel<PQ><<<(p.n_jobs + 63) / 64, 64, 0, st>>>(p);
    return cudaGetLastError();
}
cudaError_t smoother_coef(const SmootherParams &p, cudaStream_t st) {
    smoother_kernel<PQ, true><<<(p.n_jobs + 63) / 64, 64, 0, st>>>(p);
    return cudaGetLastError();
}
cudaError_t mstep(const MstepParams &p, cudaStream_t st) {
    mstep_kernel<PQ><<<(p.n_fits + 63) / 64, 64, 0, st>>>(p);
    return cudaGetLastError();
}
cudaError_t propagate(const SmootherParams &p, cudaStream_t st) {
    propagate_kernel<PQ><<<(p.n_jobs + 63) / 64, 64, 0, st>>>(p);
    return cudaGetLastError();
}
cudaError_t rep(const RepParams &p, cudaStream_t st) {
    const size_t smem = rep_smem_bytes(p.z != nullptr);
    // above the 48 KB default: opt in (per device; a cheap call, repeated rather than cached per device)
    cudaError_t e = cudaFuncSetAttribute(rep_kernel<PQ>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)rep_smem_bytes(true));
    if (e != cudaSuccess) return e;
    const int per_cta = REP_WARPS * 32;
    rep_kernel<PQ><<<(p.n_reps + per_cta - 1) / per_cta, per_cta, smem, st>>>(p);
    return cudaGetLastError();
}

const KernelTable table = {PQ,
                           em_prepare,
                           em_chunk,
                           SPLIT_NW,
                           MINB,
                           SPLIT_MSEG,
                           SPLIT_UW,
                           em_split_prepare,
                           em_split,
                           em_split_wide,
                           em_split_resident,
                           PQ >= WIDE_MIN_PQ ? WIDE_NW : 0,
                           WIDE_MSEG,
                           em_wide_prepare,
                           em_wide,
                           PQ <= SCAN_MAX_PQ ? SCAN_L : 0,
                           em_scan,
                           em_scan_traj,
                           smoother,
                           smoother_coef,
                           mstep,
                           propagate,
                           rep};

} // namespace

#define LDSR_CAT2(a, b) a##b
#define LDSR_CAT(a, b) LDSR_CAT2(a, b)
const KernelTable *LDSR_CAT(kernel_table_pq, LDSR_PQ)() { return &table; }
#endif

} // namespace ldsr
