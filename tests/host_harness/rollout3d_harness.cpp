// TEST INFRASTRUCTURE: the policy prologue of the 3-D rollout (cassierl_b200/csrc/tree_rollout.cuh) compiled for the CPU
// as a one-lane tile, so that tests/test_rollout3d_host.py can check the observation, the policy forward and the action
// map against numpy without a GPU.  fp64 only.  States are in MuJoCo's order; eps is injected instead of drawn.
#include <string>
#include "../../cassierl_b200/csrc/mjcf_flatten.h"
#include "../../cassierl_b200/csrc/tree_rollout.cuh"

using namespace cassie;
using namespace cassie::tree;

static TreeModel<double> g_m;
static std::string g_err;
static EnvScratch<double> g_s;

extern "C" {
const char* rh_error() { return g_err.c_str(); }
int rh_load(const char* path) { return flatten_tree_file(path, &g_m, &g_err) ? 0 : -1; }
int rh_params() { return kPolicyParams3d; }
// the action box of Cassie3dBatchRollout: mode 0 the motors' ctrlrange, mode 1 the range of each motor's joint
void rh_box(int mode, double* lo, double* hi) { action_box(g_m, mode, lo, hi); }
int rh_path_done(int env_done) { return path_done(env_done); }
// the prologue of one policy step from the state (q, qd): obs [45], mean / raw / env action [nu]
void rh_prologue(int mode, int normalize, const double* q, const double* qd, const double* params, const double* eps,
                 double* obs, double* mean, double* raw, double* env_act) {
  const Tile<1> tl = Tile<1>::make();
  const TreeModel<double>& m = g_m;
  for (int i = 0; i < 7; i++) g_s.q[i] = q[i];
  for (int d = 6; d < m.nv; d++) g_s.q[d + 1] = q[m.user_dof[d] + 1];
  for (int d = 0; d < m.nv; d++) g_s.qd[d] = qd[m.user_dof[d]];
  double lo[kMaxAct], hi[kMaxAct];
  rh_box(mode, lo, hi);
  policy_prologue(tl, m, g_s, params, lo, hi, normalize, [&](int a) { return eps[a]; });
  const PolicyStage<double>& ps = policy_stage<double>(g_s);
  for (int j = 0; j < kObsDim3d; j++) obs[j] = ps.obs[j];
  for (int a = 0; a < m.nu; a++) { mean[a] = ps.mean[a]; raw[a] = ps.raw[a]; env_act[a] = g_s.target[a]; }
}
}
