// Policy side of the 3-D fused rollout (Cassie3dBatchRollout, k_tree_rollout_step in tree_kernels.cuh): what rllab's
// sampler does between two env steps -- GaussianMLPPolicy.get_action on the observation, then NormalizedEnv's action map
// -- as the prologue of a policy step.  Tile-cooperative like tree_env.cuh, so the rollout kernel and the one-lane CPU
// harness (tests/host_harness/rollout3d_harness.cpp) run the same code.
//
//   obs   the 45-real observation of the env's current state (tree_env.cuh), frames recomputed for it
//   mean  tanh MLP 45 -> h1 -> ... -> hL -> nu, linear head (hidden_sizes = (h1, ..., hL), 1 <= L <= 4, 1 <= h <= 256);
//         rllab's flat parameters W1 b1 ... W(L+1) b(L+1) log_std, W stored [in][out]
//   raw   mean + exp(log_std) eps, eps standard normal (the kernel draws it from Philox, the harness injects it)
//   env action  normalize: lb + (raw + 1) / 2 (ub - lb), clipped to [lb, ub]; else raw clipped
//
// Lane j of the tile owns the units j, j + LANES, ... of every layer and action slots j, j + LANES, ...; every unit is
// one lane's serial dot product in input order, so no value is reduced across lanes and the result does not depend on
// LANES, on the env's CTA mates or on the hidden sizes of other layers.  The widths are runtime values: one kernel body
// serves every shape.  The weights (11.2 KB in fp32 at (32, 32), 94 KB at (128, 128)) are read through the read-only
// path, shared by every tile via L1 / L2: lane j reads W[i][j], a tile reads whole lines.  The observation and the hidden
// layers are staged in the constraint Jacobian's storage (J), dead between simulator steps, the hidden layers
// ping-ponging between two buffers of the widest layer, so the per-env shared block stays the env step's at any depth.
#pragma once
#include "tree_env.cuh"

namespace cassie {
namespace tree {

constexpr int kPolicyHidden3d = 32;     // the default hidden_sizes=(32, 32), as the planar policy
constexpr int kPolicyAct3d = 10;        // the ten motors
constexpr int kPolicyMaxLayers3d = 4;   // hidden layers
constexpr int kPolicyMaxWidth3d = 256;  // units per hidden layer
constexpr int kPolicyParams3d = kObsDim3d * kPolicyHidden3d + kPolicyHidden3d + kPolicyHidden3d * kPolicyHidden3d +
                                kPolicyHidden3d + kPolicyHidden3d * kPolicyAct3d + kPolicyAct3d + kPolicyAct3d;   // 2868
static_assert(kPolicyAct3d <= kMaxAct, "action slots");

// rllab's GaussianMLPPolicy(hidden_sizes=(width[0], ..., width[n_hidden - 1])) on the 45-real observation
struct PolicyShape3d {
  int n_hidden;
  int width[kPolicyMaxLayers3d];
};
TREE_HD PolicyShape3d default_policy3d() { return PolicyShape3d{2, {kPolicyHidden3d, kPolicyHidden3d, 0, 0}}; }

// the length of the flat parameter vector of a shape (2868 at the default)
TREE_HD int policy_params3d(const PolicyShape3d& p) {
  int n = 0, in = kObsDim3d;
  for (int l = 0; l < p.n_hidden; l++) {
    n += in * p.width[l] + p.width[l];
    in = p.width[l];
  }
  return n + in * kPolicyAct3d + 2 * kPolicyAct3d;
}

// the prologue's staging inside s.J
template <typename T>
struct PolicyStage {
  T obs[kObsDim3d], h[2][kPolicyMaxWidth3d], mean[kPolicyAct3d], raw[kPolicyAct3d];
};
template <typename T, typename SC>
TREE_FN PolicyStage<T>& policy_stage(SC& s) {
  // the fast pass's scratch has the smallest J: 577 reals of staging in 32 x 21
  static_assert(sizeof(PolicyStage<T>) <= sizeof(EnvScratch<T, kFastRows, kFastCon>::J),
                "the policy staging must fit in the fast pass's Jacobian storage");
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

// y[j] = tanh(b[j] + sum_i x[i] W[i][j]) for the tile's units j < nout, W [nin][nout]
template <int LANES, typename T>
TREE_FN void dense_tanh(const Tile<LANES>& tl, int nin, int nout, const T* x, const T* __restrict__ W,
                        const T* __restrict__ b, T* y) {
  for (int j = tl.lane; j < nout; j += LANES) {
    T acc = ro_load(b + j);
#pragma unroll 8
    for (int i = 0; i < nin; i++) acc += x[i] * ro_load(W + i * nout + j);
    y[j] = tanh(acc);
  }
  tl.sync();
}

// The prologue of one policy step of one env: observation into the staging, policy forward, noise (eps(a) = the standard
// normal of action slot a), action map.  Leaves obs / mean / raw in policy_stage(s) and the env action in s.target and
// s.ctrl (the torque mode's controls; the PD mode overwrites s.ctrl before every simulator step).  lo / hi = the box.
// `shape` must be valid (the C-ABI checks it: 1 to kPolicyMaxLayers3d layers of 1 to kPolicyMaxWidth3d units).
template <int LANES, typename T, typename SC, typename Eps>
TREE_FN void policy_prologue(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s, const T* __restrict__ params, const T* lo,
                             const T* hi, int normalize, Eps eps, const PolicyShape3d& shape = default_policy3d()) {
  PolicyStage<T>& ps = policy_stage<T>(s);
  T f[6];
  frames(tl, m, s);
  feet(m, s, f);
  for (int j = tl.lane; j < kObsDim3d; j += LANES) ps.obs[j] = obs_slot(m, s, f, j);
  tl.sync();
  const T* p = params;   // W1 b1 W2 b2 ... W(L+1) b(L+1) log_std
  const T* x = ps.obs;
  int nin = kObsDim3d;
  for (int l = 0; l < shape.n_hidden; l++) {
    const int nout = shape.width[l];
    T* y = ps.h[l & 1];
    dense_tanh(tl, nin, nout, x, p, p + nin * nout, y);
    p += nin * nout + nout;
    x = y;
    nin = nout;
  }
  const T* bh = p + nin * kPolicyAct3d;
  const T* lstd = bh + kPolicyAct3d;
  for (int a = tl.lane; a < kPolicyAct3d; a += LANES) {
    T mu = ro_load(bh + a);
#pragma unroll 8
    for (int i = 0; i < nin; i++) mu += x[i] * ro_load(p + i * kPolicyAct3d + a);
    const T raw = mu + exp(ro_load(lstd + a)) * eps(a);
    T v = raw;
    if (normalize) v = lo[a] + mul_rn(mul_rn(raw + (T)1, (T)0.5), hi[a] - lo[a]);
    v = v < lo[a] ? lo[a] : (v > hi[a] ? hi[a] : v);
    ps.mean[a] = mu;
    ps.raw[a] = raw;
    s.target[a] = v;
    s.ctrl[a] = v;
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
