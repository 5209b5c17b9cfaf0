// TEST INFRASTRUCTURE: the 3-D stand env (cassierl_b200/csrc/tree_env.cuh) on the tree engine, compiled for the CPU as
// a one-lane tile, so that tests/test_env3d_host.py can check the frame pass, the PD action space, the observation and
// the reward against the oracle and a numpy restatement without a GPU.  fp64 only.  States are in MuJoCo's order.
#include <cstring>
#include <string>
#include "../../cassierl_b200/csrc/mjcf_flatten.h"
#include "../../cassierl_b200/csrc/tree_env.cuh"

using namespace cassie;
using namespace cassie::tree;

static TreeModel<double> g_m;
static std::string g_err;
static Scratch<double> g_s;

static void load_state(const double* q, const double* qd, const double* warm) {
  const TreeModel<double>& m = g_m;
  for (int i = 0; i < 7; i++) g_s.q[i] = q[i];
  for (int d = 6; d < m.nv; d++) g_s.q[d + 1] = q[m.user_dof[d] + 1];
  for (int d = 0; d < m.nv; d++) { g_s.qd[d] = qd[m.user_dof[d]]; g_s.warm[d] = warm ? warm[m.user_dof[d]] : 0.0; }
}
static void store_state(double* q, double* qd, double* warm) {
  const TreeModel<double>& m = g_m;
  for (int i = 0; i < 7; i++) q[i] = g_s.q[i];
  for (int d = 6; d < m.nv; d++) q[m.user_dof[d] + 1] = g_s.q[d + 1];
  for (int d = 0; d < m.nv; d++) { qd[m.user_dof[d]] = g_s.qd[d]; warm[m.user_dof[d]] = g_s.warm[d]; }
}

extern "C" {
const char* te_error() { return g_err.c_str(); }
int te_load(const char* path) { return flatten_tree_file(path, &g_m, &g_err) ? 0 : -1; }
void te_defaults(double* kp, double* kd) {
  for (int a = 0; a < g_m.nu; a++) { kp[a] = kDefaultKp; kd[a] = kDefaultKd; }
}
// the four foot sites minus the pelvis position (world axes) at pose q, from the frame pass alone: out [4][3]
void te_sites(const double* q, double* out) {
  static const double zero[kMaxDof] = {0};
  const Tile<1> tl = Tile<1>::make();
  load_state(q, zero, nullptr);   // velocities are not read by the frame pass
  frames(tl, g_m, g_s);
  for (int k = 0; k < kNumFootSites; k++) site_rel(g_m, g_s, k, out + 3 * k);
}
// the observation of the state (q, qd) (Cassie3dBatchObserve)
void te_observe(const double* q, const double* qd, double* obs) {
  const Tile<1> tl = Tile<1>::make();
  load_state(q, qd, nullptr);
  double f[6];
  observe(tl, g_m, g_s, obs, f);
}
// one EnvStep of one env (the body of k_tree_env_step at full capacity): n_sub simulator steps with the action `act`
// (mode 0: torques, 1: PD targets), then the epilogue.  (q, qd, warm) and *len are updated in place; returns done
int te_env_step(int mode, double* q, double* qd, double* warm, const double* act, const double* kp, const double* kd,
                int n_sub, int max_path_length, int flags, const double* reset_q, const double* reset_qd, int* len,
                double* obs, double* reward) {
  const Tile<1> tl = Tile<1>::make();
  load_state(q, qd, warm);
  double target[kMaxAct];
  for (int a = 0; a < g_m.nu; a++) target[a] = g_s.ctrl[a] = act[a];
  TreeStats st = {0, 0, 0, 0};
  for (int k = 0; k < n_sub; k++) {
    if (mode == kActPd) pd_controls(tl, g_m, g_s, target, kp, kd);
    tree_step(tl, g_m, g_s, g_s.ctrl, &st);
  }
  const EnvResult r = env_finish(tl, g_m, g_s, target, flags, max_path_length, reset_q, reset_qd, *len, obs, reward);
  store_state(q, qd, warm);
  *len = r.len;
  return r.done;
}
}
