// f64 instantiation of the persistent solve kernels, circular operator.
#include "bsgp_solve_kernel.cuh"

namespace bsgp {
template cudaError_t launch_solve<double, false>(const LaunchCfg&, const SolveArgs<double>&, const SmemPlan&, size_t, const RowArgs*);
template cudaError_t query_solve_clusters<double, false>(const LaunchCfg&, int, int*);
template cudaError_t launch_frame<double, false>(const LaunchCfg&, const SolveArgs<double>&, const SmemPlan&, size_t, double*, const RowArgs*, bool);
template cudaError_t query_frame_ctas<double, false>(const LaunchCfg&, int*, bool);
}  // namespace bsgp
