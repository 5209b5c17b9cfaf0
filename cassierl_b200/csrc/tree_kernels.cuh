// CUDA kernels of the 3-D tree engine (tree_engine.cuh): one env per tile of LANES lanes, the env's whole scratch block in
// shared memory, all substeps of a policy step fused in one launch, termination + auto-reset in the same kernel.
// State in HBM is row-major per env ([n][nq], [n][nv]: a tile reads its env's row with consecutive lanes -> coalesced),
// in MuJoCo's dof order (file order); the engine's depth order is internal (TreeModel::user_dof).
#pragma once
#include <cstdint>
#include <cstdlib>
#include <cuda_runtime.h>
#include "rollout_philox.cuh"
#include "tree_engine.cuh"
#include "tree_env.cuh"
#include "tree_rollout.cuh"

namespace cassie {
void count_launch();
namespace tree {

constexpr int kTreeMaxBlock = 384;

template <typename T>
struct TreeBatchView {
  int n;
  T* qpos;        // [n][nq]
  T* qvel;        // [n][nv]
  T* warm;        // [n][nv]  qacc_warmstart
  int32_t* stats; // [n][4]: constraint rows, contacts, PGS sweeps of the last step; contacts dropped (cumulative)
  int32_t* resets; // [n] auto-resets so far
  int32_t* order;  // [n] tile slot -> env: envs binned by the row count of their last step (k_tree_bin_*), or nullptr
  int32_t* bins;   // [2 * kTreeBins] histogram / cursors of that binning
  int32_t* resume; // [n] substeps of the current launch an env has completed (two-pass scheme, k_tree_step)
};
constexpr int kTreeBins = 64;

struct TreeStepArgs {
  const void* action;   // real [n][nu], held for n_sub simulator steps; nullptr = zero controls
  int n_sub;
  double z_done;        // > 0: done when the base height qpos[2] < z_done (cassie_stand2d.py:131-133) or the state is not finite
  int auto_reset;       // done envs are put back to the reset state (zero warm start) inside the kernel
  uint8_t* done;        // [n] or nullptr
  const void* reset_q;  // real [nq] device
  const void* reset_qd; // real [nv] device
};

// MODE 0: single pass with this capacity (surplus rows / contacts are dropped and counted).
// MODE 1: fast pass: an env whose step needs more than ROWS rows / CON contacts stops BEFORE that step (state untouched),
//         is stored as it is and leaves the number of substeps it completed in v.resume[e].
// MODE 2: continuation pass with the full capacity: only envs with resume[e] < n_sub run, from that substep on.
// An env's result is therefore the full-capacity result whatever pass computed it (tests/test_gpu_tree.py).
template <typename T, int LANES, int ROWS, int CON, int MODE>
__global__ void __launch_bounds__(kTreeMaxBlock)
k_tree_step(const __grid_constant__ TreeModel<T> m, const TreeBatchView<T> v, const T* __restrict__ action, int n_sub, T z_done,
            int auto_reset, uint8_t* __restrict__ done, const T* __restrict__ reset_q, const T* __restrict__ reset_qd,
            int step_barrier) {
  // the model (5.9 KB in fp32) is a __grid_constant__ kernel parameter: it lives in the constant bank, is read with
  // tile-uniform addresses, and costs no shared memory (shared memory is what bounds the resident envs per SM)
  typedef Scratch<T, ROWS, CON> SC;
  extern __shared__ __align__(16) unsigned char tree_smem[];
  const Tile<LANES> tl = Tile<LANES>::make();
  const int tile_in_block = (int)threadIdx.x / LANES, tiles_per_block = (int)blockDim.x / LANES;
  const int e_raw = (int)blockIdx.x * tiles_per_block + tile_in_block;
  const bool active = e_raw < v.n;           // surplus tiles shadow the last env (they take part in the CTA barriers) and store nothing
  const int slot = active ? e_raw : v.n - 1;
  // the tiles of a CTA run in lock step, so a CTA is as slow as its env with the most constraint rows: slots are handed
  // out in the order of the last step's row counts (envs of similar cost share a CTA); results do not depend on it
  const int e = v.order ? v.order[slot] : slot;
  int k0 = 0;
  if (MODE == 2) {                           // no CTA barrier in this pass: tiles without work leave at once
    k0 = v.resume[e];
    if (!active || k0 >= n_sub) return;
  }
  SC& s = *reinterpret_cast<SC*>(tree_smem + (size_t)tile_in_block * sizeof(SC));
  const int nq = m.nq, nv = m.nv, nu = m.nu;
  const T* gq = v.qpos + (size_t)e * nq;
  const T* gv = v.qvel + (size_t)e * nv;
  const T* gw = v.warm + (size_t)e * nv;
  for (int i = tl.lane; i < 7; i += LANES) s.q[i] = gq[i];
  for (int d = 6 + tl.lane; d < nv; d += LANES) s.q[d + 1] = gq[m.user_dof[d] + 1];
  for (int d = tl.lane; d < nv; d += LANES) { s.qd[d] = gv[m.user_dof[d]]; s.warm[d] = gw[m.user_dof[d]]; }
  for (int a = tl.lane; a < nu; a += LANES) s.ctrl[a] = action ? action[(size_t)e * nu + a] : (T)0;
  if (tl.lane == 0) { s.n_dropped = 0; s.overflow = 0; }
  tl.sync();
  TreeStats st = {0, 0, 0, 0};
  int k_done = n_sub;
  bool alive = true;
  for (int k = k0; k < n_sub; k++) {
    // lock step of the CTA's tiles: the once-per-step code is ~10 k straight-line instructions, and tiles that run through
    // it together share the instruction-cache fills (+15 %, profiles/r2v_sweep.txt; CASSIE3D_STEP_BARRIER=0 turns it off)
    if (MODE != 2 && step_barrier > 0 && k % step_barrier == 0) __syncthreads();   // every step_barrier-th simulator step
    if (alive && !tree_step(tl, m, s, s.ctrl, &st, MODE == 1)) { alive = false; k_done = k; }
  }
  // termination (every lane evaluates it on the shared state) and auto-reset -- not for an env that is handed on
  bool bad = false;
  for (int i = 0; i < nq; i++) bad = bad || !isfinite(s.q[i]);
  for (int i = 0; i < nv; i++) bad = bad || !isfinite(s.qd[i]);
  const bool fell = z_done > 0 && s.q[2] < z_done;
  const bool is_done = alive && (bad || fell);
  tl.sync();
  if (is_done && auto_reset) {
    for (int i = tl.lane; i < 7; i += LANES) s.q[i] = reset_q[i];
    for (int d = 6 + tl.lane; d < nv; d += LANES) s.q[d + 1] = reset_q[m.user_dof[d] + 1];
    for (int d = tl.lane; d < nv; d += LANES) { s.qd[d] = reset_qd[m.user_dof[d]]; s.warm[d] = 0; }
    tl.sync();
  }
  if (!active) return;
  T* oq = v.qpos + (size_t)e * nq;
  T* ov = v.qvel + (size_t)e * nv;
  T* ow = v.warm + (size_t)e * nv;
  for (int i = tl.lane; i < 7; i += LANES) oq[i] = s.q[i];
  for (int d = 6 + tl.lane; d < nv; d += LANES) oq[m.user_dof[d] + 1] = s.q[d + 1];
  for (int d = tl.lane; d < nv; d += LANES) { ov[m.user_dof[d]] = s.qd[d]; ow[m.user_dof[d]] = s.warm[d]; }
  if (tl.lane == 0) {
    if (MODE != 0) v.resume[e] = k_done;
    if (alive) {
      if (done) done[e] = bad ? 2 : (fell ? 1 : 0);
      if (n_sub > k0) {
        v.stats[4 * e + 0] = st.nefc; v.stats[4 * e + 1] = st.ncon; v.stats[4 * e + 2] = st.sweeps;
        v.stats[4 * e + 3] += st.dropped;
      }
      if (is_done && auto_reset) v.resets[e] += 1;
    }
  }
}

// What the env variant of the step kernel (k_tree_env_step, Cassie3dBatchEnvStep) adds: the action space, the
// stand task's epilogue (tree_env.cuh) and its outputs.  A __grid_constant__ parameter: the gains are read from the
// constant bank with tile-uniform addresses.
template <typename T>
struct TreeEnvParams {
  T kp[kMaxAct], kd[kMaxAct];   // PD gains of the handle
  int mode;                     // kActTorque: the action is the controls; kActPd: PD targets, the law runs every substep
  int flags;                    // kEnvAutoReset, kEnvTerminalObs
  int max_path_length;          // > 0: done = 3 when the episode length reaches it
  T* obs;                       // [n][kObsDim3d]
  T* reward;                    // [n]
  int32_t* ep_len;              // [n] policy steps since the env's last reset
};

// Cassie3dBatchEnvStep: the passes of k_tree_step (same MODEs, same physics) with the env's action space -- in kActPd the
// PD law runs ahead of every substep on the targets kept in s.target, which the continuation pass re-reads from `action`
// -- and, instead of the z_done rule, the stand task's epilogue (tree_env.cuh).  The epilogue runs in the pass that
// completes the env's last substep, so exactly once per env and call.  A separate kernel, so that k_tree_step is
// compiled exactly as without the env.
template <typename T, int LANES, int ROWS, int CON, int MODE>
__global__ void __launch_bounds__(kTreeMaxBlock)
k_tree_env_step(const __grid_constant__ TreeModel<T> m, const TreeBatchView<T> v, const __grid_constant__ TreeEnvParams<T> env,
                const T* __restrict__ action, int n_sub, uint8_t* __restrict__ done, const T* __restrict__ reset_q,
                const T* __restrict__ reset_qd, int step_barrier) {
  typedef EnvScratch<T, ROWS, CON> SC;
  extern __shared__ __align__(16) unsigned char tree_smem[];
  const Tile<LANES> tl = Tile<LANES>::make();
  const int tile_in_block = (int)threadIdx.x / LANES, tiles_per_block = (int)blockDim.x / LANES;
  const int e_raw = (int)blockIdx.x * tiles_per_block + tile_in_block;
  const bool active = e_raw < v.n;
  const int e = active ? e_raw : v.n - 1;
  int k0 = 0;
  if (MODE == 2) {
    k0 = v.resume[e];
    if (!active || k0 >= n_sub) return;
  }
  SC& s = *reinterpret_cast<SC*>(tree_smem + (size_t)tile_in_block * sizeof(SC));
  const int nq = m.nq, nv = m.nv, nu = m.nu;
  const T* gq = v.qpos + (size_t)e * nq;
  const T* gv = v.qvel + (size_t)e * nv;
  const T* gw = v.warm + (size_t)e * nv;
  for (int i = tl.lane; i < 7; i += LANES) s.q[i] = gq[i];
  for (int d = 6 + tl.lane; d < nv; d += LANES) s.q[d + 1] = gq[m.user_dof[d] + 1];
  for (int d = tl.lane; d < nv; d += LANES) { s.qd[d] = gv[m.user_dof[d]]; s.warm[d] = gw[m.user_dof[d]]; }
  for (int a = tl.lane; a < nu; a += LANES) s.target[a] = s.ctrl[a] = action[(size_t)e * nu + a];
  if (tl.lane == 0) { s.n_dropped = 0; s.overflow = 0; }
  tl.sync();
  TreeStats st = {0, 0, 0, 0};
  int k_done = n_sub;
  bool alive = true;
  const bool pd = env.mode == kActPd;
  for (int k = k0; k < n_sub; k++) {
    if (MODE != 2 && step_barrier > 0 && k % step_barrier == 0) __syncthreads();
    if (!alive) continue;
    if (pd) pd_controls(tl, m, s, s.target, env.kp, env.kd);
    if (!tree_step(tl, m, s, s.ctrl, &st, MODE == 1)) { alive = false; k_done = k; }
  }
  if (!active) return;                       // no CTA barrier follows
  EnvResult r = {0, 0, false};
  if (alive) {                               // not for an env that is handed on
    T rew;
    r = env_finish(tl, m, s, s.target, env.flags, env.max_path_length, reset_q, reset_qd, env.ep_len[e],
                   env.obs + (size_t)e * kObsDim3d, &rew);
    if (tl.lane == 0) { env.reward[e] = rew; env.ep_len[e] = r.len; }
  }
  T* oq = v.qpos + (size_t)e * nq;
  T* ov = v.qvel + (size_t)e * nv;
  T* ow = v.warm + (size_t)e * nv;
  for (int i = tl.lane; i < 7; i += LANES) oq[i] = s.q[i];
  for (int d = 6 + tl.lane; d < nv; d += LANES) oq[m.user_dof[d] + 1] = s.q[d + 1];
  for (int d = tl.lane; d < nv; d += LANES) { ov[m.user_dof[d]] = s.qd[d]; ow[m.user_dof[d]] = s.warm[d]; }
  if (tl.lane == 0) {
    if (MODE != 0) v.resume[e] = k_done;
    if (alive) {
      done[e] = (uint8_t)r.done;
      if (n_sub > k0) {
        v.stats[4 * e + 0] = st.nefc; v.stats[4 * e + 1] = st.ncon; v.stats[4 * e + 2] = st.sweeps;
        v.stats[4 * e + 3] += st.dropped;
      }
      if (r.reset) v.resets[e] += 1;
    }
  }
}

// What the rollout variant of the env kernel (k_tree_rollout_step, Cassie3dBatchRollout) adds: the policy, the noise
// keys, the action box and the path buffers of ONE policy step (the host offsets them to row k of the [T][n][.] buffers).
template <typename T>
struct TreeRolloutParams {
  T lo[kMaxAct], hi[kMaxAct];   // action box: ctrlrange (torque mode) or the motors' joint ranges (PD mode)
  const T* params;              // [policy_params3d(shape)] GaussianMLPPolicy.flat
  PolicyShape3d shape;          // hidden_sizes
  int normalize;                // NormalizedEnv's affine map before the clip
  uint64_t seed;
  uint32_t env0;                // global id of this batch's env 0
  int32_t* policy_step;         // [n] Philox step counter, advanced by every finished policy step
  T* act_env;                   // [n][nu] the mapped, clipped action (the continuation pass reads it)
  T* obs;                       // [n][kObsDim3d] row k: the observation the policy saw
  T* act;                       // [n][nu] raw policy output
  T* mean;                      // [n][nu]
  T* rew;                       // [n]
  uint8_t* done;                // [n] path codes: 1 terminated, 2 cut at max_path_length
};

// One policy step of Cassie3dBatchRollout: the passes of k_tree_env_step (same MODEs, physics and stand-task epilogue,
// auto-reset always on), with the policy's prologue (tree_rollout.cuh) in MODE 0 / 1 instead of an action from the host.
// The continuation pass re-reads the env action from ro.act_env.  The epilogue writes the path row: reward (its action
// term on the env action), the done code in path codes, and advances policy_step.  A separate kernel, so that
// k_tree_step and k_tree_env_step compile exactly as without it.
template <typename T, int LANES, int ROWS, int CON, int MODE>
__global__ void __launch_bounds__(kTreeMaxBlock)
k_tree_rollout_step(const __grid_constant__ TreeModel<T> m, const TreeBatchView<T> v, const __grid_constant__ TreeEnvParams<T> env,
                    const __grid_constant__ TreeRolloutParams<T> ro, int n_sub, const T* __restrict__ reset_q,
                    const T* __restrict__ reset_qd, int step_barrier) {
  typedef EnvScratch<T, ROWS, CON> SC;
  extern __shared__ __align__(16) unsigned char tree_smem[];
  const Tile<LANES> tl = Tile<LANES>::make();
  const int tile_in_block = (int)threadIdx.x / LANES, tiles_per_block = (int)blockDim.x / LANES;
  const int e_raw = (int)blockIdx.x * tiles_per_block + tile_in_block;
  const bool active = e_raw < v.n;
  const int e = active ? e_raw : v.n - 1;
  int k0 = 0;
  if (MODE == 2) {
    k0 = v.resume[e];
    if (!active || k0 >= n_sub) return;
  }
  SC& s = *reinterpret_cast<SC*>(tree_smem + (size_t)tile_in_block * sizeof(SC));
  const int nq = m.nq, nv = m.nv, nu = m.nu;
  const T* gq = v.qpos + (size_t)e * nq;
  const T* gv = v.qvel + (size_t)e * nv;
  const T* gw = v.warm + (size_t)e * nv;
  for (int i = tl.lane; i < 7; i += LANES) s.q[i] = gq[i];
  for (int d = 6 + tl.lane; d < nv; d += LANES) s.q[d + 1] = gq[m.user_dof[d] + 1];
  for (int d = tl.lane; d < nv; d += LANES) { s.qd[d] = gv[m.user_dof[d]]; s.warm[d] = gw[m.user_dof[d]]; }
  if (MODE == 2)
    for (int a = tl.lane; a < nu; a += LANES) s.target[a] = s.ctrl[a] = ro.act_env[(size_t)e * nu + a];
  if (tl.lane == 0) { s.n_dropped = 0; s.overflow = 0; }
  tl.sync();
  if (MODE != 2) {
    const uint32_t gid = ro.env0 + (uint32_t)e, pstep = (uint32_t)ro.policy_step[e];
    policy_prologue(tl, m, s, ro.params, ro.lo, ro.hi, ro.normalize,
                    [&](int a) { return normal_slot<T>(ro.seed, gid, pstep, a); }, ro.shape);
    if (active) {
      const PolicyStage<T>& ps = policy_stage<T>(s);
      for (int j = tl.lane; j < kObsDim3d; j += LANES) ro.obs[(size_t)e * kObsDim3d + j] = ps.obs[j];
      for (int a = tl.lane; a < nu; a += LANES) {
        const size_t i = (size_t)e * nu + a;
        ro.act[i] = ps.raw[a];
        ro.mean[i] = ps.mean[a];
        ro.act_env[i] = s.target[a];
      }
    }
  }
  TreeStats st = {0, 0, 0, 0};
  int k_done = n_sub;
  bool alive = true;
  const bool pd = env.mode == kActPd;
  for (int k = k0; k < n_sub; k++) {
    if (MODE != 2 && step_barrier > 0 && k % step_barrier == 0) __syncthreads();
    if (!alive) continue;
    if (pd) pd_controls(tl, m, s, s.target, env.kp, env.kd);
    if (!tree_step(tl, m, s, s.ctrl, &st, MODE == 1)) { alive = false; k_done = k; }
  }
  if (!active) return;                       // no CTA barrier follows
  EnvResult r = {0, 0, false};
  if (alive) {                               // not for an env that is handed on
    T rew;
    // the observation env_finish leaves goes to the staging: the next prologue observes the state again
    r = env_finish(tl, m, s, s.target, kEnvAutoReset, env.max_path_length, reset_q, reset_qd, env.ep_len[e],
                   policy_stage<T>(s).obs, &rew);
    if (tl.lane == 0) { ro.rew[e] = rew; env.ep_len[e] = r.len; }
  }
  T* oq = v.qpos + (size_t)e * nq;
  T* ov = v.qvel + (size_t)e * nv;
  T* ow = v.warm + (size_t)e * nv;
  for (int i = tl.lane; i < 7; i += LANES) oq[i] = s.q[i];
  for (int d = 6 + tl.lane; d < nv; d += LANES) oq[m.user_dof[d] + 1] = s.q[d + 1];
  for (int d = tl.lane; d < nv; d += LANES) { ov[m.user_dof[d]] = s.qd[d]; ow[m.user_dof[d]] = s.warm[d]; }
  if (tl.lane == 0) {
    if (MODE != 0) v.resume[e] = k_done;
    if (alive) {
      ro.done[e] = (uint8_t)path_done(r.done);
      ro.policy_step[e] += 1;
      if (n_sub > k0) {
        v.stats[4 * e + 0] = st.nefc; v.stats[4 * e + 1] = st.ncon; v.stats[4 * e + 2] = st.sweeps;
        v.stats[4 * e + 3] += st.dropped;
      }
      if (r.reset) v.resets[e] += 1;
    }
  }
}

// ---- binning of the envs by the constraint-row count of their last step (a counting sort in three tiny launches)
static __global__ void k_tree_bin_hist(int n, const int32_t* __restrict__ stats, int32_t* __restrict__ bins) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  int key = stats[4 * e];
  key = key < 0 ? 0 : (key >= kTreeBins ? kTreeBins - 1 : key);
  atomicAdd(&bins[key], 1);
}
static __global__ void k_tree_bin_scan(int32_t* __restrict__ bins) {   // one thread: exclusive prefix into the cursors, histogram cleared
  int acc = 0;
  for (int k = 0; k < kTreeBins; k++) { bins[kTreeBins + k] = acc; acc += bins[k]; bins[k] = 0; }
}
static __global__ void k_tree_bin_scatter(int n, const int32_t* __restrict__ stats, int32_t* __restrict__ bins, int32_t* __restrict__ order) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n) return;
  int key = stats[4 * e];
  key = key < 0 ? 0 : (key >= kTreeBins ? kTreeBins - 1 : key);
  order[atomicAdd(&bins[kTreeBins + key], 1)] = e;
}

// qpos / qvel of selected envs <- one state (reset); warm start cleared
template <typename T>
__global__ void k_tree_set_all(TreeBatchView<T> v, int nq, int nv, const T* __restrict__ q, const T* __restrict__ qd,
                               const uint8_t* __restrict__ mask) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= v.n || (mask && !mask[e])) return;
  for (int i = 0; i < nq; i++) v.qpos[(size_t)e * nq + i] = q[i];
  for (int i = 0; i < nv; i++) { v.qvel[(size_t)e * nv + i] = qd[i]; v.warm[(size_t)e * nv + i] = 0; }
}

// the env observation of every env's current state, without stepping (Cassie3dBatchObserve / EnvReset): a tile of
// kObsLanes lanes per env, the frame pass on a small shared block (state and frames only)
template <typename T>
struct FrameScratch {
  T q[kMaxDof + 1], qd[kMaxDof];
  T xpos[kMaxLinks][3], xmat[kMaxLinks][9];
};
constexpr int kObsLanes = 8, kObsTiles = 16;

template <typename T>
__global__ void __launch_bounds__(kObsLanes * kObsTiles)
k_tree_observe(const __grid_constant__ TreeModel<T> m, const TreeBatchView<T> v, T* __restrict__ obs) {
  __shared__ FrameScratch<T> sm[kObsTiles];
  const Tile<kObsLanes> tl = Tile<kObsLanes>::make();
  const int t = (int)threadIdx.x / kObsLanes, e = (int)blockIdx.x * kObsTiles + t;
  if (e >= v.n) return;                      // whole tiles leave: only tile barriers follow
  FrameScratch<T>& s = sm[t];
  const T* gq = v.qpos + (size_t)e * m.nq;
  const T* gv = v.qvel + (size_t)e * m.nv;
  for (int i = tl.lane; i < 7; i += kObsLanes) s.q[i] = gq[i];
  for (int d = 6 + tl.lane; d < m.nv; d += kObsLanes) s.q[d + 1] = gq[m.user_dof[d] + 1];
  for (int d = tl.lane; d < m.nv; d += kObsLanes) s.qd[d] = gv[m.user_dof[d]];
  tl.sync();
  T f[6];
  observe(tl, m, s, obs + (size_t)e * kObsDim3d, f);
}

// episode lengths of the selected envs (mask nullptr: all) <- 0
static __global__ void k_tree_zero_len(int n, const uint8_t* __restrict__ mask, int32_t* __restrict__ ep_len) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < n && (!mask || mask[e])) ep_len[e] = 0;
}

template <typename T>
struct TreeLaunch {
  static cudaError_t step(const TreeModel<T>& m, const TreeBatchView<T>& v, const TreeStepArgs& a, int lanes, cudaStream_t s);
  static cudaError_t set_all(const TreeBatchView<T>& v, int nq, int nv, const T* q, const T* qd, const uint8_t* mask, cudaStream_t s);
  // EnvStep: a.action (required), a.n_sub, a.done, a.reset_q / reset_qd are used; z_done / auto_reset are the env's rule
  static cudaError_t env_step(const TreeModel<T>& m, const TreeBatchView<T>& v, const TreeStepArgs& a, const TreeEnvParams<T>& env,
                              int lanes, cudaStream_t s);
  static cudaError_t observe(const TreeModel<T>& m, const TreeBatchView<T>& v, T* obs, cudaStream_t s);
  // one policy step of Rollout: a.n_sub, a.reset_q / reset_qd are used
  static cudaError_t rollout_step(const TreeModel<T>& m, const TreeBatchView<T>& v, const TreeStepArgs& a, const TreeEnvParams<T>& env,
                                  const TreeRolloutParams<T>& ro, int lanes, cudaStream_t s);
};

// tiles (envs) per CTA of one kernel instantiation: shared memory is the resource (one Scratch block per env).  Two
// resident CTAs per SM with as many tiles each as fit; the tiles of a CTA run in lock step and share their
// instruction-cache fills (profiles/r2aa_tree_sweep_v7.txt).  CASSIE3D_TILES overrides.  Whole warps only.
template <typename K>
inline int tree_tiles(K kernel, size_t scratch_bytes, int lanes, int want) {
  int dev = 0, smem_sm = 0, smem_blk = 0;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
  cudaDeviceGetAttribute(&smem_blk, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev);
  const int per_warp = 32 / lanes;
  int t = want > 0 ? want : (smem_sm / 2 - 1024) / (int)scratch_bytes;
  const int cap_blk = smem_blk / (int)scratch_bytes, cap_thr = kTreeMaxBlock / lanes;
  if (t > cap_blk) t = cap_blk;
  if (t > cap_thr) t = cap_thr;
  t = t / per_warp * per_warp;
  if (t < per_warp) t = per_warp;
  if ((size_t)t * scratch_bytes > (size_t)smem_blk) return -1;
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)((size_t)t * scratch_bytes));
  cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
  return t;
}

template <typename T, int LANES>
inline cudaError_t launch_tree_step(const TreeModel<T>& m, const TreeBatchView<T>& v, const TreeStepArgs& a, cudaStream_t s) {
  typedef Scratch<T, kFastRows, kFastCon> Fast;
  typedef Scratch<T, kMaxRows, kMaxCon> Full;
  static const int env_tiles = [] { const char* e = getenv("CASSIE3D_TILES"); return e ? atoi(e) : 0; }();
  static const int step_barrier = [] { const char* e = getenv("CASSIE3D_STEP_BARRIER"); return e ? atoi(e) : 1; }();
  static const int sort_envs = [] { const char* e = getenv("CASSIE3D_SORT"); return e ? atoi(e) : 0; }();   // measured +1 %: off by default (profiles/r2ac_tree_lockstep.txt)
  // CASSIE3D_TWO_PASS=0: one pass with the full capacity (the round-2 v8 kernel); default: fast capacity first, the rare
  // env that needs more rows continues in a full-capacity pass (profiles/r2al_two_pass.txt)
  static const int two_pass = [] { const char* e = getenv("CASSIE3D_TWO_PASS"); return e ? atoi(e) : 1; }();
  static const int t_single = tree_tiles(k_tree_step<T, LANES, kMaxRows, kMaxCon, 0>, sizeof(Full), LANES, env_tiles);
  static const int t_fast = tree_tiles(k_tree_step<T, LANES, kFastRows, kFastCon, 1>, sizeof(Fast), LANES, env_tiles);
  static const int t_cont = tree_tiles(k_tree_step<T, LANES, kMaxRows, kMaxCon, 2>, sizeof(Full), LANES, 32 / LANES);   // one warp per CTA: idle tiles leave at once
  if (t_single < 0 || t_fast < 0 || t_cont < 0) return cudaErrorInvalidConfiguration;
  TreeBatchView<T> vv = v;
  const int tiles0 = two_pass ? t_fast : t_single;
  if (sort_envs && step_barrier && v.order && v.bins && tiles0 > 1) {
    k_tree_bin_hist<<<(v.n + 255) / 256, 256, 0, s>>>(v.n, v.stats, v.bins);
    k_tree_bin_scan<<<1, 1, 0, s>>>(v.bins);
    k_tree_bin_scatter<<<(v.n + 255) / 256, 256, 0, s>>>(v.n, v.stats, v.bins, v.order);
    count_launch(); count_launch(); count_launch();
  } else
    vv.order = nullptr;
  const T* act = (const T*)a.action;
  const T *rq = (const T*)a.reset_q, *rv = (const T*)a.reset_qd;
  if (!two_pass) {
    k_tree_step<T, LANES, kMaxRows, kMaxCon, 0><<<(unsigned)((v.n + t_single - 1) / t_single), t_single * LANES, (size_t)t_single * sizeof(Full), s>>>(
        m, vv, act, a.n_sub, (T)a.z_done, a.auto_reset, a.done, rq, rv, step_barrier);
    count_launch();
    return cudaGetLastError();
  }
  k_tree_step<T, LANES, kFastRows, kFastCon, 1><<<(unsigned)((v.n + t_fast - 1) / t_fast), t_fast * LANES, (size_t)t_fast * sizeof(Fast), s>>>(
      m, vv, act, a.n_sub, (T)a.z_done, a.auto_reset, a.done, rq, rv, step_barrier);
  count_launch();
  vv.order = nullptr;
  k_tree_step<T, LANES, kMaxRows, kMaxCon, 2><<<(unsigned)((v.n + t_cont - 1) / t_cont), t_cont * LANES, (size_t)t_cont * sizeof(Full), s>>>(
      m, vv, act, a.n_sub, (T)a.z_done, a.auto_reset, a.done, rq, rv, 0);
  count_launch();
  return cudaGetLastError();
}

inline int tree_knob(const char* name, int dflt) {
  const char* e = getenv(name);
  return e ? atoi(e) : dflt;
}

// the passes of launch_tree_step (same knobs, no env sorting) on the env kernels
template <typename T, int LANES>
inline cudaError_t launch_tree_env_step(const TreeModel<T>& m, const TreeBatchView<T>& v, const TreeStepArgs& a,
                                        const TreeEnvParams<T>& env, cudaStream_t s) {
  typedef EnvScratch<T, kFastRows, kFastCon> Fast;
  typedef EnvScratch<T, kMaxRows, kMaxCon> Full;
  static const int env_tiles = tree_knob("CASSIE3D_TILES", 0);
  static const int step_barrier = tree_knob("CASSIE3D_STEP_BARRIER", 1);
  static const int two_pass = tree_knob("CASSIE3D_TWO_PASS", 1);
  static const int t_single = tree_tiles(k_tree_env_step<T, LANES, kMaxRows, kMaxCon, 0>, sizeof(Full), LANES, env_tiles);
  static const int t_fast = tree_tiles(k_tree_env_step<T, LANES, kFastRows, kFastCon, 1>, sizeof(Fast), LANES, env_tiles);
  static const int t_cont = tree_tiles(k_tree_env_step<T, LANES, kMaxRows, kMaxCon, 2>, sizeof(Full), LANES, 32 / LANES);
  if (t_single < 0 || t_fast < 0 || t_cont < 0) return cudaErrorInvalidConfiguration;
  TreeBatchView<T> vv = v;
  vv.order = nullptr;
  const T* act = (const T*)a.action;
  const T *rq = (const T*)a.reset_q, *rv = (const T*)a.reset_qd;
  if (!two_pass) {
    k_tree_env_step<T, LANES, kMaxRows, kMaxCon, 0><<<(unsigned)((v.n + t_single - 1) / t_single), t_single * LANES, (size_t)t_single * sizeof(Full), s>>>(
        m, vv, env, act, a.n_sub, a.done, rq, rv, step_barrier);
    count_launch();
    return cudaGetLastError();
  }
  k_tree_env_step<T, LANES, kFastRows, kFastCon, 1><<<(unsigned)((v.n + t_fast - 1) / t_fast), t_fast * LANES, (size_t)t_fast * sizeof(Fast), s>>>(
      m, vv, env, act, a.n_sub, a.done, rq, rv, step_barrier);
  count_launch();
  k_tree_env_step<T, LANES, kMaxRows, kMaxCon, 2><<<(unsigned)((v.n + t_cont - 1) / t_cont), t_cont * LANES, (size_t)t_cont * sizeof(Full), s>>>(
      m, vv, env, act, a.n_sub, a.done, rq, rv, 0);
  count_launch();
  return cudaGetLastError();
}

// the passes of launch_tree_env_step (same knobs, same tiles per CTA: the rollout's per-env block is EnvScratch) on the
// rollout kernel, for one policy step
template <typename T, int LANES>
inline cudaError_t launch_tree_rollout_step(const TreeModel<T>& m, const TreeBatchView<T>& v, const TreeStepArgs& a,
                                            const TreeEnvParams<T>& env, const TreeRolloutParams<T>& ro, cudaStream_t s) {
  typedef EnvScratch<T, kFastRows, kFastCon> Fast;
  typedef EnvScratch<T, kMaxRows, kMaxCon> Full;
  static const int env_tiles = tree_knob("CASSIE3D_TILES", 0);
  static const int step_barrier = tree_knob("CASSIE3D_STEP_BARRIER", 1);
  static const int two_pass = tree_knob("CASSIE3D_TWO_PASS", 1);
  static const int t_single = tree_tiles(k_tree_rollout_step<T, LANES, kMaxRows, kMaxCon, 0>, sizeof(Full), LANES, env_tiles);
  static const int t_fast = tree_tiles(k_tree_rollout_step<T, LANES, kFastRows, kFastCon, 1>, sizeof(Fast), LANES, env_tiles);
  static const int t_cont = tree_tiles(k_tree_rollout_step<T, LANES, kMaxRows, kMaxCon, 2>, sizeof(Full), LANES, 32 / LANES);
  if (t_single < 0 || t_fast < 0 || t_cont < 0) return cudaErrorInvalidConfiguration;
  TreeBatchView<T> vv = v;
  vv.order = nullptr;
  const T *rq = (const T*)a.reset_q, *rv = (const T*)a.reset_qd;
  if (!two_pass) {
    k_tree_rollout_step<T, LANES, kMaxRows, kMaxCon, 0><<<(unsigned)((v.n + t_single - 1) / t_single), t_single * LANES, (size_t)t_single * sizeof(Full), s>>>(
        m, vv, env, ro, a.n_sub, rq, rv, step_barrier);
    count_launch();
    return cudaGetLastError();
  }
  k_tree_rollout_step<T, LANES, kFastRows, kFastCon, 1><<<(unsigned)((v.n + t_fast - 1) / t_fast), t_fast * LANES, (size_t)t_fast * sizeof(Fast), s>>>(
      m, vv, env, ro, a.n_sub, rq, rv, step_barrier);
  count_launch();
  k_tree_rollout_step<T, LANES, kMaxRows, kMaxCon, 2><<<(unsigned)((v.n + t_cont - 1) / t_cont), t_cont * LANES, (size_t)t_cont * sizeof(Full), s>>>(
      m, vv, env, ro, a.n_sub, rq, rv, 0);
  count_launch();
  return cudaGetLastError();
}

#define CASSIE_TREE_INSTANTIATE(T)                                                                                         \
  template <>                                                                                                              \
  cudaError_t TreeLaunch<T>::step(const TreeModel<T>& dm, const TreeBatchView<T>& v, const TreeStepArgs& a, int lanes,     \
                                  cudaStream_t s) {                                                                        \
    if (lanes == 8) return launch_tree_step<T, 8>(dm, v, a, s);                                                            \
    if (lanes == 16) return launch_tree_step<T, 16>(dm, v, a, s);                                                          \
    if (lanes == 32) return launch_tree_step<T, 32>(dm, v, a, s);                                                          \
    return cudaErrorInvalidValue;                                                                                          \
  }                                                                                                                        \
  template <>                                                                                                              \
  cudaError_t TreeLaunch<T>::set_all(const TreeBatchView<T>& v, int nq, int nv, const T* q, const T* qd,                   \
                                     const uint8_t* mask, cudaStream_t s) {                                                \
    k_tree_set_all<T><<<(v.n + 127) / 128, 128, 0, s>>>(v, nq, nv, q, qd, mask);                                           \
    count_launch();                                                                                                        \
    return cudaGetLastError();                                                                                             \
  }                                                                                                                        \
  template <>                                                                                                              \
  cudaError_t TreeLaunch<T>::env_step(const TreeModel<T>& dm, const TreeBatchView<T>& v, const TreeStepArgs& a,            \
                                      const TreeEnvParams<T>& env, int lanes, cudaStream_t s) {                            \
    if (lanes == 8) return launch_tree_env_step<T, 8>(dm, v, a, env, s);                                                   \
    if (lanes == 16) return launch_tree_env_step<T, 16>(dm, v, a, env, s);                                                 \
    if (lanes == 32) return launch_tree_env_step<T, 32>(dm, v, a, env, s);                                                 \
    return cudaErrorInvalidValue;                                                                                          \
  }                                                                                                                        \
  template <>                                                                                                              \
  cudaError_t TreeLaunch<T>::observe(const TreeModel<T>& dm, const TreeBatchView<T>& v, T* obs, cudaStream_t s) {          \
    k_tree_observe<T><<<(v.n + kObsTiles - 1) / kObsTiles, kObsLanes * kObsTiles, 0, s>>>(dm, v, obs);                     \
    count_launch();                                                                                                        \
    return cudaGetLastError();                                                                                             \
  }                                                                                                                        \
  template <>                                                                                                              \
  cudaError_t TreeLaunch<T>::rollout_step(const TreeModel<T>& dm, const TreeBatchView<T>& v, const TreeStepArgs& a,        \
                                          const TreeEnvParams<T>& env, const TreeRolloutParams<T>& ro, int lanes,          \
                                          cudaStream_t s) {                                                                \
    if (lanes == 8) return launch_tree_rollout_step<T, 8>(dm, v, a, env, ro, s);                                           \
    if (lanes == 16) return launch_tree_rollout_step<T, 16>(dm, v, a, env, ro, s);                                         \
    if (lanes == 32) return launch_tree_rollout_step<T, 32>(dm, v, a, env, ro, s);                                         \
    return cudaErrorInvalidValue;                                                                                          \
  }

}  // namespace tree
}  // namespace cassie
