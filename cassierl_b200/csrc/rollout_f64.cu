// fp64 instantiation of the fused rollout kernel (parity build), see rollout_kernels.cuh
#include "rollout_launch.cuh"
namespace cassie {
template cudaError_t launch_rollout<double>(const ModelPair<double>&, const BatchView<double>&, const RolloutArgs&, cudaStream_t);
template cudaError_t launch_discounted_returns<double>(const void*, const uint8_t*, const void*, double, int, int, void*, cudaStream_t);
template cudaError_t launch_baseline_moments<double>(const BaselineArgs&, cudaStream_t);
template cudaError_t launch_advantages<double>(const BaselineArgs&, cudaStream_t);
// the 3-D observation (cassie3d_api.cu)
template cudaError_t launch_baseline_moments<double, kMaxFeat3d, kMomentsPerThread3d>(const BaselineArgs&, cudaStream_t);
template cudaError_t launch_advantages<double, kMaxFeat3d>(const BaselineArgs&, cudaStream_t);
}
