// Policy side of the 3-D fused rollout (Cassie3dBatchRollout, k_tree_rollout_step in tree_kernels.cuh): what rllab's
// sampler does between two env steps -- GaussianMLPPolicy.get_action on the observation, then NormalizedEnv's action map
// -- as the prologue of a policy step.  Tile-cooperative like tree_env.cuh, so the rollout kernel and the one-lane CPU
// harness (tests/host_harness/rollout3d_harness.cpp) run the same code.
//
//   obs   the 45-real observation of the env's current state (tree_env.cuh), frames recomputed for it
//   mean  tanh MLP 45 -> 32 -> 32 -> nu, linear head; rllab's flat parameters W1 b1 W2 b2 W3 b3 log_std, W stored [in][out]
//   raw   mean + exp(log_std) eps, eps standard normal (the kernel draws it from Philox, the harness injects it)
//   env action  normalize: lb + (raw + 1) / 2 (ub - lb), clipped to [lb, ub]; else raw clipped
//
// Lane j of the tile owns hidden units j, j + LANES, ... and action slots j, j + LANES, ...; every unit is one lane's
// serial dot product in input order, so no value is reduced across lanes and the result does not depend on LANES or on
// the env's CTA mates.  The weights (11.2 KB in fp32) are read through the read-only path, shared by every tile via L1:
// lane j reads W[i][j], a tile reads whole lines.  The observation and hidden layers are staged in the constraint
// Jacobian's storage (J), dead between simulator steps, so the per-env shared block stays the env step's.
#pragma once
#include "tree_env.cuh"

namespace cassie {
namespace tree {

constexpr int kPolicyHidden3d = 32;   // hidden_sizes=(32, 32), as the planar policy
constexpr int kPolicyAct3d = 10;      // the ten motors
constexpr int kPolicyParams3d = kObsDim3d * kPolicyHidden3d + kPolicyHidden3d + kPolicyHidden3d * kPolicyHidden3d +
                                kPolicyHidden3d + kPolicyHidden3d * kPolicyAct3d + kPolicyAct3d + kPolicyAct3d;   // 2868
static_assert(kPolicyAct3d <= kMaxAct, "action slots");

// the prologue's staging inside s.J
template <typename T>
struct PolicyStage {
  T obs[kObsDim3d], h1[kPolicyHidden3d], h2[kPolicyHidden3d], mean[kPolicyAct3d], raw[kPolicyAct3d];
};
template <typename T, typename SC>
TREE_FN PolicyStage<T>& policy_stage(SC& s) {
  static_assert(sizeof(PolicyStage<T>) <= sizeof(SC::J), "the policy staging must fit in the Jacobian's storage");
  return *reinterpret_cast<PolicyStage<T>*>(s.J);
}

template <typename T>
TREE_FN T ro_load(const T* p) {
#if defined(__CUDA_ARCH__)
  return __ldg(p);
#else
  return *p;
#endif
}

// a * b rounded on its own, never contracted into an FMA: the action map then rounds as an elementwise restatement
// (PyTorch, numpy) of lb + (a + 1) / 2 (ub - lb) does, so that replaying the recorded actions through EnvStep reproduces
// a rollout bit for bit
template <typename T>
TREE_FN T mul_rn(T a, T b) {
#if defined(__CUDA_ARCH__)
  if constexpr (sizeof(T) == 8) return __dmul_rn(a, b);
  else return __fmul_rn(a, b);
#else
  return a * b;
#endif
}

// y[j] = tanh(b[j] + sum_i x[i] W[i][j]) for the tile's hidden units
template <int NIN, int LANES, typename T>
TREE_FN void dense_tanh(const Tile<LANES>& tl, const T* x, const T* __restrict__ W, const T* __restrict__ b, T* y) {
  for (int j = tl.lane; j < kPolicyHidden3d; j += LANES) {
    T acc = ro_load(b + j);
#pragma unroll 8
    for (int i = 0; i < NIN; i++) acc += x[i] * ro_load(W + i * kPolicyHidden3d + j);
    y[j] = tanh(acc);
  }
  tl.sync();
}

// The prologue of one policy step of one env: observation into the staging, policy forward, noise (eps(a) = the standard
// normal of action slot a), action map.  Leaves obs / mean / raw in policy_stage(s) and the env action in s.target and
// s.ctrl (the torque mode's controls; the PD mode overwrites s.ctrl before every simulator step).  lo / hi = the box.
template <int LANES, typename T, typename SC, typename Eps>
TREE_FN void policy_prologue(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s, const T* __restrict__ params, const T* lo,
                             const T* hi, int normalize, Eps eps) {
  PolicyStage<T>& ps = policy_stage<T>(s);
  T f[6];
  frames(tl, m, s);
  feet(m, s, f);
  for (int j = tl.lane; j < kObsDim3d; j += LANES) ps.obs[j] = obs_slot(m, s, f, j);
  tl.sync();
  const T* W1 = params;
  const T* b1 = W1 + kObsDim3d * kPolicyHidden3d;
  const T* W2 = b1 + kPolicyHidden3d;
  const T* b2 = W2 + kPolicyHidden3d * kPolicyHidden3d;
  const T* W3 = b2 + kPolicyHidden3d;
  const T* b3 = W3 + kPolicyHidden3d * kPolicyAct3d;
  const T* lstd = b3 + kPolicyAct3d;
  dense_tanh<kObsDim3d>(tl, ps.obs, W1, b1, ps.h1);
  dense_tanh<kPolicyHidden3d>(tl, ps.h1, W2, b2, ps.h2);
  for (int a = tl.lane; a < kPolicyAct3d; a += LANES) {
    T mu = ro_load(b3 + a);
#pragma unroll 8
    for (int i = 0; i < kPolicyHidden3d; i++) mu += ps.h2[i] * ro_load(W3 + i * kPolicyAct3d + a);
    const T raw = mu + exp(ro_load(lstd + a)) * eps(a);
    T x = raw;
    if (normalize) x = lo[a] + mul_rn(mul_rn(raw + (T)1, (T)0.5), hi[a] - lo[a]);
    x = x < lo[a] ? lo[a] : (x > hi[a] ? hi[a] : x);
    ps.mean[a] = mu;
    ps.raw[a] = raw;
    s.target[a] = x;
    s.ctrl[a] = x;
  }
  tl.sync();
}

// the action box of the rollout (host side, from the flattened model): the motors' ctrlrange in kActTorque, the range of
// each motor's joint in kActPd
inline void action_box(const TreeModel<double>& m, int mode, double* lo, double* hi) {
  for (int a = 0; a < m.nu; a++) {
    const int d = m.act_dof[a];
    lo[a] = mode == kActPd ? m.range[d][0] : m.act_lo[a];
    hi[a] = mode == kActPd ? m.range[d][1] : m.act_hi[a];
  }
}

// the rollout's done code of an env done code: 1 fell / 2 diverged -> 1 (terminated), 3 time limit -> 2 (cut at
// max_path_length): the planar rollout's path-buffer codes
TREE_HD int path_done(int env_done) { return env_done == 3 ? 2 : (env_done != 0 ? 1 : 0); }

}  // namespace tree
}  // namespace cassie
