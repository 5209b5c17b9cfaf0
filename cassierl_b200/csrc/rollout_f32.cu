// fp32 instantiation of the fused rollout kernel (policy MLP + env step), see rollout_kernels.cuh
#include "rollout_launch.cuh"
namespace cassie {
template cudaError_t launch_rollout<float>(const ModelPair<float>&, const BatchView<float>&, const RolloutArgs&, cudaStream_t);
template cudaError_t launch_discounted_returns<float>(const void*, const uint8_t*, const void*, double, int, int, void*, cudaStream_t);
template cudaError_t launch_baseline_moments<float>(const BaselineArgs&, cudaStream_t);
template cudaError_t launch_advantages<float>(const BaselineArgs&, cudaStream_t);
// the 3-D observation (cassie3d_api.cu)
template cudaError_t launch_baseline_moments<float, kMaxFeat3d, kMomentsPerThread3d>(const BaselineArgs&, cudaStream_t);
template cudaError_t launch_advantages<float, kMaxFeat3d>(const BaselineArgs&, cudaStream_t);
}
