// TEST INFRASTRUCTURE: the policy prologue of the 3-D rollout (cassierl_b200/csrc/tree_rollout.cuh) at any hidden_sizes,
// compiled for the CPU as a one-lane tile in the fast pass's scratch (the smallest constraint-Jacobian storage), so that
// tests/test_rollout3d_mlp_host.py can check the forward and the action map against numpy without a GPU.  fp64 only.
// States are in MuJoCo's order; eps is injected instead of drawn.
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
const char* rmh_error() { return g_err.c_str(); }
int rmh_load(const char* path) { return flatten_tree_file(path, &g_m, &g_err) ? 0 : -1; }
// the action box of Cassie3dBatchRollout: mode 0 the motors' ctrlrange, mode 1 the range of each motor's joint
void rmh_box(int mode, double* lo, double* hi) { action_box(g_m, mode, lo, hi); }
int rmh_params(int n_hidden, const int* sizes) { return policy_params3d(shape_of(n_hidden, sizes)); }
// reals of the prologue's staging, and of the fast pass's constraint-Jacobian storage it lives in
int rmh_stage_reals() { return (int)(sizeof(PolicyStage<double>) / sizeof(double)); }
int rmh_fast_j_reals() { return (int)(sizeof(FastScratch::J) / sizeof(double)); }
// the prologue of one policy step from the state (q, qd): obs [45], mean / raw / env action [nu]
void rmh_prologue(int mode, int normalize, int n_hidden, const int* sizes, const double* q, const double* qd,
                  const double* params, const double* eps, double* obs, double* mean, double* raw, double* env_act) {
  const Tile<1> tl = Tile<1>::make();
  const TreeModel<double>& m = g_m;
  for (int i = 0; i < 7; i++) g_s.q[i] = q[i];
  for (int d = 6; d < m.nv; d++) g_s.q[d + 1] = q[m.user_dof[d] + 1];
  for (int d = 0; d < m.nv; d++) g_s.qd[d] = qd[m.user_dof[d]];
  double lo[kMaxAct], hi[kMaxAct];
  rmh_box(mode, lo, hi);
  policy_prologue(tl, m, g_s, params, lo, hi, normalize, [&](int a) { return eps[a]; }, shape_of(n_hidden, sizes));
  const PolicyStage<double>& ps = policy_stage<double>(g_s);
  for (int j = 0; j < kObsDim3d; j++) obs[j] = ps.obs[j];
  for (int a = 0; a < m.nu; a++) { mean[a] = ps.mean[a]; raw[a] = ps.raw[a]; env_act[a] = g_s.target[a]; }
}
}
