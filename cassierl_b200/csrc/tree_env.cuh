// Stand-task env of the 3-D tree engine (include/cassie3d.h, Cassie3dBatchEnvStep): the PD action space, the 45-real
// observation, the reward and the termination rule.  Tile-cooperative like tree_engine.cuh, so the step kernels
// (tree_kernels.cuh) and the one-lane CPU harness (tests/host_harness/tree_env_harness.cpp) run the same code.
//
// The 3-D model has no reference environment; this carries the planar stand task (cassie_stand2d.py:119-133) over:
//   obs    [0] pelvis height qpos[2], [1..4] pelvis quaternion qpos[3:7], [5..18] the 14 hinge angles qpos[7:21],
//          [19..38] qvel[0:20] (MuJoCo convention), [39..41] / [42..44] left / right foot minus pelvis, world axes;
//          a foot is the mean of its front and rear contact site
//   reward 1 - 2 (0.9 - z)^2 - 2 |c|^2 - 0.001 |a|^2, c = horizontal offset of the feet midpoint from the pelvis,
//          a = the action as given (targets or torques, before clamping); 0 for a diverged env
//   done   2 diverged (not finite or beyond 1e10), else 1 fell (z < 0.5), else 3 time limit (episode length reached
//          max_path_length > 0), else 0
// Observation, reward and done are taken from the state after the last substep, with the frames recomputed for it
// (the frames in Scratch after tree_step belong to the start of that substep).
#pragma once
#include "tree_engine.cuh"

namespace cassie {
namespace tree {

constexpr int kObsDim3d = 45;
constexpr double kStandHeight = 0.9, kFallHeight = 0.5, kDivergedBound = 1e10;
enum EnvFlags3d { kEnvAutoReset = 1, kEnvTerminalObs = 8 };   // CASSIE3D_AUTO_RESET, CASSIE3D_TERMINAL_OBS
enum ActionMode3d { kActTorque = 0, kActPd = 1 };             // CASSIE3D_MODE_TORQUE, CASSIE3D_MODE_PD
constexpr double kDefaultKp = 10.0, kDefaultKd = 5.0;          // ctrl units, Cassie2d.cpp:96-112

// PD law of one simulator step, ahead of tree_step: ctrl_a = kp_a (target_a - q_j(a)) - kd_a qd_j(a), j(a) = the
// motor's joint (tree_step then clamps to ctrlrange as for torques)
template <int LANES, typename T, typename SC>
TREE_FN void pd_controls(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s, const T* target, const T* kp, const T* kd) {
  for (int a = tl.lane; a < m.nu; a += LANES) {
    const int d = m.act_dof[a];
    s.ctrl[a] = kp[a] * (target[a] - s.q[d + 1]) - kd[a] * s.qd[d];
  }
  tl.sync();
}

// the frame pass of dynamics() alone (mj_kinematics): link frames of the state in s.q, no velocities, inertias or forces
template <int LANES, typename T, typename SC>
TREE_FN void frames(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s) {
  for (int lev = 0; lev < m.nlevels; lev++) {
    for (int l = m.level_off[lev] + tl.lane; l < m.level_off[lev + 1]; l += LANES) {
      T an[3], ax[3];
      link_frame(m, s, l, an, ax);
    }
    tl.sync();
  }
}

// foot-site position minus pelvis position, world axes (every lane computes it; the frames are current)
template <typename T, typename SC>
TREE_FN void site_rel(const TreeModel<T>& m, const SC& s, int k, T* p) {
  const int l = m.site_link[k];
  mulv(p, s.xmat[l], m.site_pos[k]);
  for (int i = 0; i < 3; i++) p[i] += s.xpos[l][i];
}

// left foot [0..2], right foot [3..5]: mean of the front and rear contact sites, minus the pelvis position
template <typename T, typename SC>
TREE_FN void feet(const TreeModel<T>& m, const SC& s, T* f) {
  for (int side = 0; side < 2; side++) {
    T a[3], b[3];
    site_rel(m, s, 2 * side, a);
    site_rel(m, s, 2 * side + 1, b);
    for (int i = 0; i < 3; i++) f[3 * side + i] = (T)0.5 * (a[i] + b[i]);
  }
}

// slot j of the observation (MuJoCo order; the engine's depth order is internal)
template <typename T, typename SC>
TREE_FN T obs_slot(const TreeModel<T>& m, const SC& s, const T* f, int j) {
  if (j < 5) return s.q[2 + j];                          // height, quaternion
  if (j < 19) return s.q[m.dof_of_user[j + 1] + 1];      // hinge qpos[7 + i] = user dof 6 + i
  if (j < 39) return s.qd[m.dof_of_user[j - 19]];
  return f[j - 39];
}

// frames of the current state, then its observation (obs = this env's row); returns the feet
template <int LANES, typename T, typename SC>
TREE_FN void observe(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s, T* obs, T* f) {
  frames(tl, m, s);
  feet(m, s, f);
  for (int j = tl.lane; j < kObsDim3d; j += LANES) obs[j] = obs_slot(m, s, f, j);
}

template <typename T>
TREE_FN T stand_reward(T z, const T* f, const T* act, int nu) {
  const T cx = (T)0.5 * (f[0] + f[3]), cy = (T)0.5 * (f[1] + f[4]), dz = (T)kStandHeight - z;
  T a2 = 0;
  for (int a = 0; a < nu; a++) a2 += act[a] * act[a];
  return 1 - 2 * dz * dz - 2 * (cx * cx + cy * cy) - (T)0.001 * a2;
}

// not finite, or beyond 1e10 (the planar state_diverged; MuJoCo's mj_checkPos / mj_checkVel)
template <typename T, typename SC>
TREE_FN bool env_diverged(const TreeModel<T>& m, const SC& s) {
  bool bad = false;
  for (int i = 0; i < m.nq; i++) bad = bad || !(s.q[i] < (T)kDivergedBound && s.q[i] > (T)-kDivergedBound);
  for (int i = 0; i < m.nv; i++) bad = bad || !(s.qd[i] < (T)kDivergedBound && s.qd[i] > (T)-kDivergedBound);
  return bad;
}

// s.q, s.qd <- the reset state (MuJoCo order, as the handle keeps it); warm start cleared
template <int LANES, typename T, typename SC>
TREE_FN void load_reset(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s, const T* rq, const T* rqd) {
  for (int i = tl.lane; i < 7; i += LANES) s.q[i] = rq[i];
  for (int d = 6 + tl.lane; d < m.nv; d += LANES) s.q[d + 1] = rq[m.user_dof[d] + 1];
  for (int d = tl.lane; d < m.nv; d += LANES) { s.qd[d] = rqd[m.user_dof[d]]; s.warm[d] = 0; }
  tl.sync();
}

// the env kernels' per-env scratch: the step's, plus the action as given (PD targets survive all substeps in it)
template <typename T, int ROWS = kMaxRows, int CON = kMaxCon>
struct EnvScratch : Scratch<T, ROWS, CON> {
  T target[kMaxAct];
};

struct EnvResult { int done, len; bool reset; };

// The epilogue of one env after the last substep of an EnvStep: reward (every lane holds it), done code, episode length
// (len = the length before this step), reset of a done env (auto-reset) or a diverged one (always), observation into
// obs (this env's row): the reset state's for a reset env unless kEnvTerminalObs asks for the terminal one -- never the
// terminal one of a diverged env, which is not finite.
template <int LANES, typename T, typename SC>
TREE_FN EnvResult env_finish(const Tile<LANES>& tl, const TreeModel<T>& m, SC& s, const T* act, int flags,
                             int max_path_length, const T* reset_q, const T* reset_qd, int len, T* obs, T* reward) {
  EnvResult r;
  const bool bad = env_diverged(m, s);
  r.len = len + 1;
  r.done = bad ? 2 : (s.q[2] < (T)kFallHeight ? 1 : (max_path_length > 0 && r.len >= max_path_length ? 3 : 0));
  r.reset = bad || (r.done != 0 && (flags & kEnvAutoReset));
  const bool terminal_obs = !r.reset || ((flags & kEnvTerminalObs) && !bad);
  T f[6];
  frames(tl, m, s);
  feet(m, s, f);
  *reward = bad ? (T)0 : stand_reward(s.q[2], f, act, m.nu);
  if (terminal_obs)
    for (int j = tl.lane; j < kObsDim3d; j += LANES) obs[j] = obs_slot(m, s, f, j);
  if (r.reset) {
    tl.sync();                                 // every lane is done reading the terminal state
    load_reset(tl, m, s, reset_q, reset_qd);
    r.len = 0;
    if (!terminal_obs) observe(tl, m, s, obs, f);
  }
  return r;
}

}  // namespace tree
}  // namespace cassie
