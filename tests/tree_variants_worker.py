"""Worker of tests/test_gpu_tree_variants.py: runs one seeded scenario through the 3-D tree engine's Step and EnvStep
launches for precision 32 and 64 and lanes 8, 16 and 32, and saves what every launch returns to an .npz file.

The launch knobs of the tree kernels (CASSIE3D_TWO_PASS, CASSIE3D_SORT, CASSIE3D_STEP_BARRIER, CASSIE3D_TILES) are read
once per process, so the test starts this worker once per setting and compares the files.

    python tests/tree_variants_worker.py OUT.npz
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.dirname(HERE), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from conftest import TORQUE_HIGH_3D, LEG_POSE_3D, lying3d, pose3d  # noqa: E402
from test_env3d_host import PD_HIGH, PD_LOW  # noqa: E402

N = 101                                          # prime: the last CTA has idle tiles at every tile count
LYING = (0, 23, 24, 39, 40, 55, 56, N - 1)       # 33-36 rows: handed on to the continuation pass; at CTA boundaries
AIR = (3, 11, 30, 47, 70, 88)                    # tumbling in the air
LOW = (5, 19, 33, 61, 77, 95)                    # rolled and spinning below the fall height
NAN_ENV = 17
SUB = 10
# Step launches: (name, z_done, auto_reset, n_sub)
STEPS = (("s1", 0.5, True, SUB), ("s2", 0.5, True, SUB), ("s3", 0.5, True, SUB), ("one_step", 0.0, True, 1))
# EnvStep launches: (name, mode, flags, max_path_length, n_sub); mode 1 PD, 0 torque; flags 1 auto-reset, 8 terminal obs
ENVS = (("e1", 1, 1, 2, SUB), ("e2", 1, 1, 2, SUB), ("e3", 1, 1, 2, SUB), ("t1", 0, 1 | 8, 0, SUB), ("t2", 0, 1 | 8, 0, SUB),
        ("one_env", 1, 0, 0, 1))
STEP_MODE = {s[0]: s[1:] for s in STEPS}
ENV_MODE = {s[0]: s[1:] for s in ENVS}
LAUNCHES = ["s1", "s2", "s3", "e1", "e2", "e3", "t1", "t2", "one_step", "one_env"]
# launches that start from the scenario (SetState, which also zeroes the warm start and the episode lengths).  s1
# leaves mixed row counts; under CASSIE3D_SORT=1 they order the envs of s2, which starts from the scenario again, so
# that the sorted launch hands the lying robots on to the continuation pass.  one_step / one_env: one substep from
# the scenario, what the fp32 build of the single-pass kernels is compared on.
RESTART = {"s1", "s2", "e1", "t1", "one_step", "one_env"}


def quat_yaw_roll(yaw, roll):
    """the quaternion product yaw (about z) * roll (about x)"""
    cy, sy, cr, sr = np.cos(yaw / 2), np.sin(yaw / 2), np.cos(roll / 2), np.sin(roll / 2)
    return np.array([cy * cr, cy * sr, sy * sr, sy * cr])


def asymmetric_reset():
    """a reset state that shows a wrong dof mapping: left and right legs differ (inside the joint ranges), yawed and
    slightly rolled pelvis off the origin, twenty distinct non-zero velocities"""
    q = pose3d(0.95)
    q[0:2] = [0.8, -0.6]
    q[3:7] = quat_yaw_roll(0.7, 0.05)
    q[7:14] = np.array(LEG_POSE_3D) + [0.08, -0.05, 0.10, -0.08, 0.06, -0.05, 0.02]
    q[14:21] = np.array(LEG_POSE_3D) + [-0.04, 0.07, -0.06, 0.05, -0.03, 0.08, -0.03]
    v = 0.02 * (1 + np.arange(20)) * (-1.0) ** np.arange(20)
    return q, v


def scenario(seed=0):
    """initial qpos, qvel of the N envs and the actions of every launch"""
    rng = np.random.default_rng(seed)
    q = np.tile(pose3d(0.945), (N, 1))
    q[:, 7:] += rng.normal(size=(N, 14)) * 0.03
    for e in range(N):
        q[e, 3:7] = quat_yaw_roll(rng.uniform(-np.pi, np.pi), rng.normal() * 0.05)
    q[:, 0:2] = rng.normal(size=(N, 2)) * 3.0
    v = rng.normal(size=(N, 20)) * 0.05
    for e in AIR:
        q[e, 2] = 2.0
        qu = rng.normal(size=4); q[e, 3:7] = qu / np.linalg.norm(qu)
        v[e] = rng.normal(size=20) * 0.5
    for e in LOW:
        q[e, 2] = 0.6; q[e, 3:7] = quat_yaw_roll(rng.uniform(-np.pi, np.pi), 1.2)
        v[e, 3:6] += rng.normal(size=3) * 2.0
    kinds = [(0.10, "x", 1.5708, False), (0.14, "y", -1.5708, True), (0.12, "x", 1.5708, True), (0.06, "y", 1.5708, False)]
    for i, e in enumerate(LYING):
        q[e] = lying3d(*kinds[i % 4][:3], straight=kinds[i % 4][3]); v[e] = 0
    q[NAN_ENV, 9] = np.nan
    acts = {}
    for name in LAUNCHES:
        pd = name in ENV_MODE and ENV_MODE[name][0] == 1
        acts[name] = rng.uniform(PD_LOW, PD_HIGH, (N, 10)) if pd else rng.uniform(-1, 1, (N, 10)) * TORQUE_HIGH_3D
    return q, v, acts


def run(prec, lanes, out):
    import torch
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    q0, v0, acts = scenario()
    env = Cassie3dBatchEnv(N, precision=prec, lanes=lanes)
    b = env.batch
    b.set_reset_state(*asymmetric_reset())
    pre = "p%d_l%d_" % (prec, lanes)

    def record(name, done, obs=None, rew=None):
        q, v = b.state()
        torch.cuda.synchronize()
        rec = dict(q=q, v=v, w=b.warm_start(), stats=b.stats(), resets=b.resets(), done=done)
        if obs is not None:
            rec.update(obs=obs, rew=rew, len=env.episode_lengths())
        for k, x in rec.items():
            out[pre + name + "_" + k] = x.cpu().numpy().copy()

    for name in LAUNCHES:
        if name in RESTART:
            b.set_state(q0, v0)
        a = torch.tensor(acts[name], dtype=b.dtype, device=b.device)
        if name in STEP_MODE:
            z, auto, n_sub = STEP_MODE[name]
            done = torch.empty(N, dtype=torch.uint8, device=b.device)
            record(name, b.step(a, n=n_sub, z_done=z, auto_reset=auto, done=done))
        else:
            env.mode, env.flags, env.max_path_length, n_sub = ENV_MODE[name]   # the env's action space and flags per launch
            obs, rew, done = env.step(a, n=n_sub)
            record(name, done, obs, rew)
    env.terminate()


if __name__ == "__main__":
    out = {}
    for prec in (32, 64):
        for lanes in (8, 16, 32):
            run(prec, lanes, out)
    np.savez(sys.argv[1], **out)
