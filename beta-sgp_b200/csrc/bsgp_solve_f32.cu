// f32 instantiation of the persistent solve kernels, circular operator.
#include "bsgp_solve_kernel.cuh"

namespace bsgp {
template cudaError_t launch_solve<float, false>(const LaunchCfg&, const SolveArgs<float>&, const SmemPlan&, size_t, const RowArgs*);
template cudaError_t query_solve_clusters<float, false>(const LaunchCfg&, int, int*);
template cudaError_t launch_frame<float, false>(const LaunchCfg&, const SolveArgs<float>&, const SmemPlan&, size_t, double*, const RowArgs*, bool);
template cudaError_t query_frame_ctas<float, false>(const LaunchCfg&, int*, bool);
}  // namespace bsgp
