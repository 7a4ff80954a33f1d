// kernel_table.h -- host-visible launchers of the per-PQ kernel instantiations.
// Each supported padded input width PQ is compiled as its own translation unit
// (kernels_inst.cu with -DLDSR_PQ=n) and exposes one table of launch functions.
#pragma once
#include "aux_kernels.cuh"
#include "em_kernel.cuh"
#include "em_split_kernel.cuh"
#include "em_wide_kernel.cuh"
#include "em_scan_kernel.cuh"

namespace ldsr {

#ifndef LDSR_SEG
#define LDSR_SEG 8
#endif
constexpr int EM_SEG = LDSR_SEG; // steps per checkpoint segment (divides 32)
constexpr int EM_WARPS = 4; // warps per CTA (one per SM sub-partition)
// time-split kernel: warps per CTA and the CTAs/SM the register budget is set for
// (65536 regs / (NW*32*MINB): 4 warps x 3 CTAs -> 170 registers per thread)
#ifndef LDSR_SPLIT_NW
#define LDSR_SPLIT_NW 4
#endif
constexpr int SPLIT_NW = LDSR_SPLIT_NW;
#ifndef LDSR_SPLIT_MSEG
#define LDSR_SPLIT_MSEG 4
#endif
#ifndef LDSR_SPLIT_UW
#define LDSR_SPLIT_UW 32
#endif
constexpr int SPLIT_MSEG = LDSR_SPLIT_MSEG; // steps per M unit (observed somewhere in the CTA)
constexpr int SPLIT_UW = LDSR_SPLIT_UW;     // steps per U unit (unobserved by every fit of the CTA)
constexpr int split_minb_for(int pq) {
#ifdef LDSR_SPLIT_MINB
    return LDSR_SPLIT_MINB;
#else
    return pq <= 4 ? 3 : 2;
#endif
}

// wide-input kernel (em_wide_kernel.cuh): compiled for PQ >= WIDE_MIN_PQ, one CTA of WIDE_NW warps per SM
constexpr int WIDE_MIN_PQ = 5;
#ifndef LDSR_WIDE_NW
#define LDSR_WIDE_NW 8
#endif
constexpr int WIDE_NW = LDSR_WIDE_NW;
constexpr int WIDE_MSEG = 8;

// small-batch scan kernel (em_scan_kernel.cuh): one CTA per fit, SCAN_L steps per thread; compiled for PQ <= SCAN_MAX_PQ
constexpr int SCAN_MAX_PQ = 10;
constexpr int SCAN_L = 4; // steps per thread for width <= 4 (T <= 1024); wider inputs take 2 (T <= 512, v == u)

struct KernelTable {
    int pq;
    cudaError_t (*em_prepare)(size_t smem_bytes); // opt in to > 48 KB dynamic shared memory
    cudaError_t (*em_chunk)(const EmParams &, int n_tasks, size_t smem_bytes, cudaStream_t);
    // time-split kernel (em_split_kernel.cuh): warps per CTA, CTAs per SM it is compiled for
    int split_nw, split_minb, split_mseg, split_uw;
    cudaError_t (*em_split_prepare)(size_t smem_bytes);
    cudaError_t (*em_split)(const SplitParams &, int n_tasks, size_t smem_bytes, cudaStream_t);
    // the same kernel compiled for 2 CTAs/SM (255 registers): 9 % faster per launch when the batch
    // needs no more than two CTAs per SM; the same function as em_split when split_minb == 2
    // With SplitParams.flags the launch is cooperative (the CTAs hand tasks over to one another).
    cudaError_t (*em_split_wide)(const SplitParams &, int n_tasks, size_t smem_bytes, cudaStream_t);
    int (*em_split_resident)(size_t smem_bytes); // CTAs of em_split_wide one SM holds at once (0: unknown)
    // wide-input kernel: wide_nw == 0 when this width has none (PQ < WIDE_MIN_PQ)
    int wide_nw, wide_mseg;
    cudaError_t (*em_wide_prepare)(size_t smem_bytes);
    cudaError_t (*em_wide)(const WideParams &, int n_tasks, size_t smem_bytes, cudaStream_t);
    // small-batch scan kernel: scan_l == 0 when this width has none (PQ > SCAN_MAX_PQ); series up to
    // scan_l * 32 * SCAN_MAX_WARPS steps.  Launched with 2 or 4 steps per thread; EmParams.max_seg carries
    // the longest series of the plan (the block is sized from it).
    int scan_l;
    cudaError_t (*em_scan)(const EmParams &, int n_tasks, int steps_per_thread, cudaStream_t);
    // the same kernel's E-step once, writing the smoothed trajectories of EmParams.n_jobs (group, fit) pairs
    cudaError_t (*em_scan_traj)(const EmParams &, int steps_per_thread, cudaStream_t);
    cudaError_t (*smoother)(const SmootherParams &, cudaStream_t);
    cudaError_t (*smoother_coef)(const SmootherParams &, cudaStream_t); // its backward-sampling coefficient mode
    cudaError_t (*mstep)(const MstepParams &, cudaStream_t);
    cudaError_t (*propagate)(const SmootherParams &, cudaStream_t);
    cudaError_t (*rep)(const RepParams &, cudaStream_t);
};

const KernelTable *kernel_table_for(int pq_needed); // smallest instantiation with pq >= pq_needed

} // namespace ldsr
