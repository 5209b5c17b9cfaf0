/* C-ABI of the batched 3-D Cassie step path (libcassie2d.so, same shared library as include/cassie2d.h).
 *
 * The reference ships NO library for its 3-D model: model/cassie3d_stiff.xml:1-192 is only ever loaded by MuJoCo's own
 * viewer (SURVEY.md section 8(d) config 4: "No reference library exists for 3-D"; 8(f) row 2: "also a 3-D RobotInterface
 * (none exists)").  These entry points are therefore the batch analogue of what src/Cassie2d/Cassie2d.cpp:15-27 exports
 * for the planar model, restricted to what BASELINE.json configs[3] needs: torque actions (the ten motors of
 * cassie3d_stiff.xml:180-191), mj_step semantics (cassie3d_stiff.xml:5), done when the pelvis height drops below a
 * threshold (rule borrowed from rllab/envs/cassie_stand2d.py:131-133), auto-reset to a standing pose.
 *
 * Conventions: plain pointers and sizes only; device pointers unless a name ends in Host; `real` = float (precision 32)
 * or double (precision 64); qpos [n][nq] and qvel [n][nv] row-major per env in MuJoCo's order (free joint: position,
 * quaternion w x y z; then the hinges in file order); every call is asynchronous on `stream` and returns 0 or -1 with
 * Cassie3dGetLastError(); nothing aborts.  There is no CPU fallback: Create fails without a CUDA device.
 */
#ifndef CASSIE3D_H_
#define CASSIE3D_H_
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct Cassie3dBatch Cassie3dBatch;

const char* Cassie3dGetLastError(void);
/* xml_path NULL: the packaged physics-only rendition of cassie3d_stiff.xml (cassierl_b200/model/). */
Cassie3dBatch* Cassie3dBatchCreate(const char* xml_path, int n_envs, int device, int precision);
void Cassie3dBatchDestroy(Cassie3dBatch* h);
/* out[0..5] = nq, nv, nu, constraint-row capacity, contact capacity (per env and step; what exceeds them is dropped in
 * MuJoCo's pair order and counted in the stats), bytes of shared memory per env of the first pass (the step runs a small
 * capacity first and finishes the rare env that needs more in a full-capacity continuation launch: same results) */
int Cassie3dBatchSizes(Cassie3dBatch* h, int32_t* out);
/* lanes per env of the step kernel: 8, 16 or 32 (default: env CASSIE3D_LANES, else 32) */
int Cassie3dBatchSetLanes(Cassie3dBatch* h, int lanes);
/* the state done envs are reset to, and the state SetAll writes (host doubles, qpos[nq], qvel[nv]); the default is
 * the standing pose of Cassie2d.cpp:56-58 carried over to the 3-D joints (abduction = yaw = 0) */
int Cassie3dBatchSetResetState(Cassie3dBatch* h, const double* qpos, const double* qvel);
int Cassie3dBatchGetResetState(Cassie3dBatch* h, double* qpos, double* qvel);
/* every env (mask NULL) or the envs with mask[e] != 0 <- the reset state; warm start and episode length cleared */
int Cassie3dBatchResetAll(Cassie3dBatch* h, const uint8_t* mask, void* stream);
/* whole-batch state I/O, real [n][nq] / [n][nv]; SetState clears the warm start and the episode lengths */
int Cassie3dBatchSetState(Cassie3dBatch* h, const void* qpos, const void* qvel, void* stream);
int Cassie3dBatchGetState(Cassie3dBatch* h, void* qpos, void* qvel, void* stream);
int Cassie3dBatchGetWarmStart(Cassie3dBatch* h, void* qacc_warmstart, void* stream);
int Cassie3dBatchSetWarmStart(Cassie3dBatch* h, const void* qacc_warmstart, void* stream);
/* n_substeps x mj_step with the controls `action` (real [n][nu], clamped to ctrlrange; NULL = zero) held.  z_done > 0:
 * done[e] = 1 when qpos[2] < z_done after the last substep, 2 when the state is not finite; with auto_reset such envs
 * restart from the reset state inside the same launch.  done may be NULL. */
int Cassie3dBatchStep(Cassie3dBatch* h, const void* action, int n_substeps, double z_done, int auto_reset, uint8_t* done,
                      void* stream);
/* the same with HOST buffers (pinned or pageable): action in, qpos / qvel / done out; copies and the synchronisation
 * are inside the call -- the end-to-end path of bench3d */
int Cassie3dBatchStepHost(Cassie3dBatch* h, const void* action, int n_substeps, double z_done, int auto_reset,
                          void* qpos_out, void* qvel_out, uint8_t* done_out);
/* int32 [n][4]: constraint rows, contacts, PGS sweeps of the last step; contacts dropped for capacity so far */
int Cassie3dBatchGetStats(Cassie3dBatch* h, int32_t* stats, void* stream);
/* int32 [n]: auto-resets so far */
int Cassie3dBatchGetResets(Cassie3dBatch* h, int32_t* resets, void* stream);

/* ---- stand-task environment (the planar Cassie2dBatchEnvStep's counterpart; the 3-D model has no reference env, so the
 * task is a design carried over from rllab/envs/cassie_stand2d.py:119-133, DESIGN.md section 11).
 *
 * action real [n][nu], motors in file order (abduction, yaw, hip, knee, toe per leg, left leg first):
 *   CASSIE3D_MODE_TORQUE  the controls, held for the n_substeps simulator steps (clamped to ctrlrange)
 *   CASSIE3D_MODE_PD      joint targets [rad]; before EVERY simulator step u = kp (target - q) - kd qd on each motor's
 *                         joint, then clamped to ctrlrange.  Gains per handle, default kp = 10, kd = 5 (Cassie2d.cpp:96-112)
 * obs real [n][CASSIE3D_OBS_DIM] of the state after the last simulator step: [0] pelvis height, [1..4] pelvis quaternion
 *   w x y z, [5..18] the 14 hinge angles, [19..38] qvel (linear velocity in world axes, angular velocity in pelvis axes,
 *   hinge rates), [39..41] left and [42..44] right foot minus pelvis position in world axes (a foot is the mean of its
 *   *_contact_front and *_contact_rear sites)
 * reward real [n] = 1 - 2 (0.9 - z)^2 - 2 |c|^2 - 0.001 |action|^2, z = pelvis height, c = horizontal offset of the feet
 *   midpoint from the pelvis; 0 for a diverged env
 * done uint8 [n]: 2 the state is not finite or beyond 1e10 (the env is then always reset), else 1 pelvis below 0.5 m,
 *   else 3 the episode length reached max_path_length > 0, else 0
 * flags: CASSIE3D_AUTO_RESET: done envs restart from the reset state inside the call (warm start cleared), and the
 *   observation returned is the reset state's unless CASSIE3D_TERMINAL_OBS asks for the terminal one (a diverged env
 *   always returns the reset state's).  Episode length: +1 per EnvStep, 0 after every reset (EnvReset, ResetAll,
 *   SetState, auto-reset). */
enum { CASSIE3D_MODE_TORQUE = 0, CASSIE3D_MODE_PD = 1 };
enum { CASSIE3D_AUTO_RESET = 1, CASSIE3D_TERMINAL_OBS = 8 };
enum { CASSIE3D_OBS_DIM = 45 };
/* host doubles, [nu] each */
int Cassie3dBatchSetPdGains(Cassie3dBatch* h, const double* kp, const double* kd);
/* n_substeps >= 1 simulator steps of every env, then observation, reward, done; obs / reward / done are required */
int Cassie3dBatchEnvStep(Cassie3dBatch* h, int mode, const void* action, int n_substeps, int max_path_length, int flags,
                         void* obs, void* reward, uint8_t* done, void* stream);
/* the same with HOST buffers: action in, obs / reward / done out (each may be NULL); copies and the synchronisation are
 * inside the call */
int Cassie3dBatchEnvStepHost(Cassie3dBatch* h, int mode, const void* action, int n_substeps, int max_path_length, int flags,
                             void* obs, void* reward, uint8_t* done);
/* ResetAll(mask) (NULL = every env), then the observation of EVERY env into obs (obs may be NULL) */
int Cassie3dBatchEnvReset(Cassie3dBatch* h, const uint8_t* mask, void* obs, void* stream);
/* the observation of the current state of every env, without stepping (e.g. after SetState) */
int Cassie3dBatchObserve(Cassie3dBatch* h, void* obs, void* stream);
/* int32 [n]: EnvStep calls since each env's last reset */
int Cassie3dBatchGetEpisodeLengths(Cassie3dBatch* h, int32_t* ep_len, void* stream);

/* ---- rollout collection on the stand-task env (the planar Cassie2dBatchRollout's counterpart): rllab's BatchSampler
 * with GaussianMLPPolicy(hidden_sizes) and normalize(env), n_policy_steps policy steps of every env, enqueued on
 * `stream` without a host synchronisation (one or two launches per policy step).
 *
 * Per env and policy step k: obs[k] = the observation of the current state; mean[k] = tanh MLP 45 -> h1 -> ... -> hL ->
 * 10 with a linear head, hidden_sizes = (h1, ..., hL) (host int32 [n_hidden]), 1 <= L <= CASSIE3D_POLICY_MAX_LAYERS,
 * 1 <= h <= CASSIE3D_POLICY_MAX_WIDTH; params_dev = rllab's flat vector W1 b1 W2 b2 ... W(L+1) b(L+1) log_std (real,
 * W stored [in][out]), n_params = its length, sum over layers of (in + 1) out, plus 10; action[k] = mean + exp(log_std)
 * * eps, the raw policy output rllab stores; the env action = lb + (action + 1) / 2 (ub - lb) clipped to [lb, ub] with
 * normalize != 0, else action clipped; then n_substeps >= 1 simulator steps and the EnvStep epilogue with auto-reset:
 * reward[k] (its action term on the env action), done[k] in path codes 1 = terminated (fell or diverged; a diverged env's
 * reward is 0), 2 = cut because the episode length reached max_path_length > 0, else 0.  Episodes continue across calls;
 * the episode lengths are EnvStep's (GetEpisodeLengths).
 *
 * Buffers (device): obs real [T][n][CASSIE3D_OBS_DIM], action / mean real [T][n][nu], reward real [T][n], done uint8
 * [T][n], T = n_policy_steps.
 * Action box [lb, ub] (Cassie3dBatchActionBox), from the model: CASSIE3D_MODE_TORQUE the motors' ctrlrange,
 * CASSIE3D_MODE_PD the range of each motor's joint.
 * Noise: eps of action a = Box-Muller on Philox4x32-10 with key = seed (low word first) and counter {first_global_env +
 * e, step, a / 4, 0}, step = the env's rollout policy-step counter (0 at Create, advanced by Rollout only, never reset):
 * actions 0..7 are the two pairs of blocks 0 and 1 as in the planar rollout, actions 8 and 9 the first pair of block 2.
 * A batch holding global envs [first_global_env, first_global_env + n) therefore draws what one large batch would, and
 * the noise does not depend on hidden_sizes.
 * Returns -1 (Cassie3dGetLastError) for a null pointer, an unknown mode, n_substeps < 1, max_path_length <= 0, a shape
 * outside the limits or an n_params that is not the shape's. */
enum { CASSIE3D_POLICY_MAX_LAYERS = 4, CASSIE3D_POLICY_MAX_WIDTH = 256 };
int Cassie3dBatchRolloutMlp(Cassie3dBatch* h, int mode, int n_hidden, const int32_t* hidden_sizes, const void* params_dev,
                            int n_params, int n_policy_steps, int n_substeps, int max_path_length, int normalize,
                            unsigned long long seed, unsigned int first_global_env, void* obs_dev, void* action_dev,
                            void* mean_dev, void* reward_dev, uint8_t* done_dev, void* stream);
/* RolloutMlp with hidden_sizes = (32, 32), the reference's TRPO launcher's: CASSIE3D_POLICY_PARAMS entries */
enum { CASSIE3D_POLICY_PARAMS = 2868 };
int Cassie3dBatchRollout(Cassie3dBatch* h, int mode, const void* params_dev, int n_params, int n_policy_steps,
                         int n_substeps, int max_path_length, int normalize, unsigned long long seed,
                         unsigned int first_global_env, void* obs_dev, void* action_dev, void* mean_dev,
                         void* reward_dev, uint8_t* done_dev, void* stream);
/* RolloutMlp with DDPG's sampler: rllab's DeterministicMLPPolicy(hidden_sizes) explored by OUStrategy(mu, theta, sigma).
 *
 * Per env and policy step k: mean[k] = tanh(b + x W) of a relu MLP 45 -> h1 -> ... -> hL -> 10 (same shape limits);
 * params_dev = W1 b1 ... W(L+1) b(L+1) with NO log_std, n_params = the sum over layers of (in + 1) out.  OU state x
 * (real [n][nu], kept in the handle across calls): at a path start (the env's episode length is 0: after Create,
 * ResetAll, SetState, EnvReset or an auto-reset) x = ou_mu, as rllab's es.reset() after env.reset(); then
 * x += ou_theta (ou_mu - x) + ou_sigma eps, eps the same standard normal of (seed, global env, step, action) RolloutMlp
 * draws.  action[k] = clip(mean + x, -1, 1) with normalize != 0 (the box of normalize(env)), else clip(mean + x, lb, ub):
 * the clipped exploratory action rllab's DDPG stores in its pool; the env action is mapped from it as in RolloutMlp.
 * Every finished policy step advances x once.  The state is zero at Create and is not touched by the other calls, so a
 * path already under way at the first RolloutOU call (e.g. run by RolloutMlp or EnvStep before) starts from x = 0, not
 * mu.  Buffers, reward, done and the noise counter are RolloutMlp's.
 * Returns -1 as RolloutMlp does, and for an n_params that is not the deterministic count (a Gaussian vector with its
 * log_std included), a non-finite ou_mu, ou_theta or ou_sigma, or ou_sigma < 0. */
int Cassie3dBatchRolloutOU(Cassie3dBatch* h, int mode, int n_hidden, const int32_t* hidden_sizes, const void* params_dev,
                           int n_params, double ou_mu, double ou_theta, double ou_sigma, int n_policy_steps,
                           int n_substeps, int max_path_length, int normalize, unsigned long long seed,
                           unsigned int first_global_env, void* obs_dev, void* action_dev, void* mean_dev,
                           void* reward_dev, uint8_t* done_dev, void* stream);
/* host doubles [nu]: the action box Rollout maps into and clips to in `mode` */
int Cassie3dBatchActionBox(Cassie3dBatch* h, int mode, double* lo, double* hi);
/* sampler side of rllab's process_samples on Rollout's [T][n] buffers, as the planar calls of the same names:
 * returns[k] = reward[k] + gamma returns[k + 1] within a path, the last unfinished path bootstrapped with tail_dev
 * (real [n], NULL = 0) */
int Cassie3dBatchDiscountedReturns(Cassie3dBatch* h, const void* reward_dev, const uint8_t* done_dev, const void* tail_dev,
                                   double gamma, int n_policy_steps, void* returns_dev, void* stream);
/* LinearFeatureBaseline normal equations: features [clip(o, -10, 10), clip(o)^2, al, al^2, al^3, 1], al = step in path
 * / 100 (D = 94); path_start_dev (int32 [n], may be NULL = 0) = the in-path index of each env's first sample,
 * path_index_dev (int32 [T][n]) receives every sample's; moments_dev (double, D (D + 1) / 2 + D) = the packed upper
 * triangle of F'F row by row, then F'y */
int Cassie3dBatchBaselineMoments(Cassie3dBatch* h, const void* obs_dev, const void* returns_dev, const uint8_t* done_dev,
                                 const int32_t* path_start_dev, int n_policy_steps, int32_t* path_index_dev,
                                 double* moments_dev, void* stream);
/* baseline values (values_dev may be NULL) and GAE advantages [T][n] with the coefficients coeffs_dev (real [D]) */
int Cassie3dBatchAdvantages(Cassie3dBatch* h, const void* obs_dev, const void* reward_dev, const uint8_t* done_dev,
                            const int32_t* path_index_dev, const void* coeffs_dev, double gamma, double gae_lambda,
                            int n_policy_steps, void* advantages_dev, void* values_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif
