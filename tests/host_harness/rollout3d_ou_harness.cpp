// TEST INFRASTRUCTURE: the deterministic policy kind of the 3-D rollout's prologue (cassierl_b200/csrc/tree_rollout.cuh,
// kPolicyOu3d: DeterministicMLPPolicy + OUStrategy) compiled for the CPU as a one-lane tile in the fast pass's scratch,
// so that tests/test_rollout3d_ou_host.py can check the forward, the OU step and the action map against numpy without a
// GPU.  fp64 only.  States are in MuJoCo's order; eps and the prior OU state are injected.
#include <string>
#include "../../cassierl_b200/csrc/mjcf_flatten.h"
#include "../../cassierl_b200/csrc/tree_rollout.cuh"

using namespace cassie;
using namespace cassie::tree;

typedef EnvScratch<double, kFastRows, kFastCon> FastScratch;
static TreeModel<double> g_m;
static std::string g_err;
static FastScratch g_s;

static PolicyShape3d shape_of(int n_hidden, const int* sizes) {
  PolicyShape3d p = {n_hidden, {0, 0, 0, 0}};
  for (int l = 0; l < n_hidden; l++) p.width[l] = sizes[l];
  return p;
}

extern "C" {
const char* roh_error() { return g_err.c_str(); }
int roh_load(const char* path) { return flatten_tree_file(path, &g_m, &g_err) ? 0 : -1; }
void roh_box(int mode, double* lo, double* hi) { action_box(g_m, mode, lo, hi); }
// the deterministic parameter count of a shape (no log_std)
int roh_params(int n_hidden, const int* sizes) { return policy_params3d(shape_of(n_hidden, sizes), kPolicyOu3d); }
// one deterministic prologue from the state (q, qd) and the OU state x_prev: obs [45], mean / raw / env action / x_next
// [nu].  x_next may alias x_prev; the kernel advances the state in place.
void roh_prologue(int mode, int normalize, int n_hidden, const int* sizes, const double* q, const double* qd,
                  const double* params, const double* eps, double mu, double theta, double sigma, const double* x_prev,
                  int path_start, double* obs, double* mean, double* raw, double* env_act, double* x_next) {
  const Tile<1> tl = Tile<1>::make();
  const TreeModel<double>& m = g_m;
  for (int i = 0; i < 7; i++) g_s.q[i] = q[i];
  for (int d = 6; d < m.nv; d++) g_s.q[d + 1] = q[m.user_dof[d] + 1];
  for (int d = 0; d < m.nv; d++) g_s.qd[d] = qd[m.user_dof[d]];
  double lo[kMaxAct], hi[kMaxAct];
  roh_box(mode, lo, hi);
  double x[kMaxAct];
  for (int a = 0; a < m.nu; a++) x[a] = x_prev[a];
  const int32_t ep_len = path_start ? 0 : 1;
  const OuStep3d<double> ou = {mu, theta, sigma, x, &ep_len, true};
  policy_prologue(tl, m, g_s, params, lo, hi, normalize, [&](int a) { return eps[a]; }, shape_of(n_hidden, sizes),
                  kPolicyOu3d, ou);
  const PolicyStage<double>& ps = policy_stage<double>(g_s);
  for (int j = 0; j < kObsDim3d; j++) obs[j] = ps.obs[j];
  for (int a = 0; a < m.nu; a++) { mean[a] = ps.mean[a]; raw[a] = ps.raw[a]; env_act[a] = g_s.target[a]; x_next[a] = x[a]; }
}
}
