// Host-side arguments of the fused rollout launch (rollout_kernels.cuh) and the sampler-side launches that the planar
// (cassie2d_api.cu) and the 3-D (cassie3d_api.cu) C-ABI share
#pragma once
#include <cstdint>
#include <cuda_runtime.h>
namespace cassie {
struct RolloutArgs {
  int task, mode, n_substeps, T_steps, max_path_length, flags, normalize;
  uint64_t seed;
  uint32_t env0;
  const void* params;
  void* obs; void* act; void* mean; void* rew; uint8_t* done;
  double act_lo[7], act_hi[7];
};
// arguments of the baseline-moment / advantage launches (rollout_kernels.cuh)
struct BaselineArgs {
  const void* obs; const void* rew; const void* ret; const uint8_t* done; const int32_t* start; int32_t* idx;
  const void* coeffs; void* adv; void* value; double* moments; int odim, T_steps, n; double gamma, lambda;
};

// the sampler-side launches for the 3-D observation (cassie3d_api.cu; instantiated in rollout_f32.cu / rollout_f64.cu
// next to the planar ones, which batch_state.h declares): MAXF = feature capacity (D = 2 odim + 4 <= MAXF), EPT = packed
// moment entries per thread (D (D + 1) / 2 + D <= 256 EPT).  The 45-real observation of tree_env.cuh: D = 94, 4559 entries.
constexpr int kMaxFeat3d = 2 * 45 + 4, kMomentsPerThread3d = 18;
static_assert(kMaxFeat3d * (kMaxFeat3d + 1) / 2 + kMaxFeat3d <= 256 * kMomentsPerThread3d, "3-D moments per thread");
template <typename T>
cudaError_t launch_discounted_returns(const void* rew, const uint8_t* done, const void* tail, double gamma, int T_steps, int n,
                                      void* ret, cudaStream_t s);
template <typename T, int MAXF, int EPT>
cudaError_t launch_baseline_moments(const BaselineArgs& a, cudaStream_t s);
template <typename T, int MAXF>
cudaError_t launch_advantages(const BaselineArgs& a, cudaStream_t s);
}  // namespace cassie
