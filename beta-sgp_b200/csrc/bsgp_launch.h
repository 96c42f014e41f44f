// Host-side launch helpers shared by the translation units of libbsgp.
#pragma once
#include <cuda_runtime.h>
#include <string.h>

#include "bsgp_device.cuh"

namespace bsgp {

template <typename T> struct SolveArgs;
struct RowArgs;

struct LaunchCfg {
    int grid, threads, G;
    size_t smem;
    cudaStream_t stream;
    int minb = 1;          // CTAs per SM the kernel variant is compiled for (solve kernel only)
};

// The dynamic shared-memory attribute is per function, not per plan: plans of different shapes share the
// kernels, so every launch (re)states the limit it needs.
static inline cudaError_t prepare_func(const void* func, const LaunchCfg& lc) {
    cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)lc.smem);
    if (e != cudaSuccess) return e;
    if (lc.G > 8) e = cudaFuncSetAttribute(func, cudaFuncAttributeNonPortableClusterSizeAllowed, 1);
    return e;
}

static inline void fill_cfg(cudaLaunchConfig_t* cfg, cudaLaunchAttribute* at, const LaunchCfg& lc, int grid) {
    memset(cfg, 0, sizeof *cfg);
    cfg->gridDim = dim3(grid); cfg->blockDim = dim3(lc.threads); cfg->dynamicSmemBytes = lc.smem; cfg->stream = lc.stream;
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = lc.G; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg->attrs = at; cfg->numAttrs = 1;
}

static inline cudaError_t launch_clustered(const void* func, const LaunchCfg& lc, void** args) {
    cudaError_t e = prepare_func(func, lc);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute at[1];
    fill_cfg(&cfg, at, lc, lc.grid);
    return cudaLaunchKernelExC(&cfg, func, args);
}

// how many clusters of this configuration can be resident at once
static inline cudaError_t query_clusters(const void* func, const LaunchCfg& lc, int num_sms, int* out) {
    cudaError_t e = prepare_func(func, lc);
    if (e != cudaSuccess) return e;
    if (lc.G == 1) {
        int nb = 0;
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, func, lc.threads, lc.smem);
        *out = nb * num_sms;
        return e;
    }
    cudaLaunchConfig_t cfg;
    cudaLaunchAttribute at[1];
    fill_cfg(&cfg, at, lc, lc.G * num_sms);
    int n = 0;
    e = cudaOccupancyMaxActiveClusters(&n, func, &cfg);
    *out = n;
    return e;
}

// rows: NULL, or a mixed batch (the ROWS kernels, bsgp_solve_kernel.cuh).  Defined in bsgp_solve_f64.cu / bsgp_solve_f32.cu (MK = false) and bsgp_solve_f64_padded.cu / bsgp_solve_f32_padded.cu (MK = true)
template <typename T, bool MK> cudaError_t launch_solve(const LaunchCfg& lc, const SolveArgs<T>& a, const SmemPlan& sp, size_t tf_stride,
                                                  const RowArgs* rows);
template <typename T, bool MK> cudaError_t query_solve_clusters(const LaunchCfg& lc, int num_sms, int* out);
// split: the plan has an axis of split transforms (bsgp_conv.cuh), run by the frame kernels of SplitCtx
template <typename T, bool MK> cudaError_t launch_frame(const LaunchCfg& lc, const SolveArgs<T>& a, const SmemPlan& sp, size_t tf_stride, double* gpart,
                                                  const RowArgs* rows, bool split);
template <typename T, bool MK> cudaError_t query_frame_ctas(const LaunchCfg& lc, int* per_sm, bool split);

}  // namespace bsgp
