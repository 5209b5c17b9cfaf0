"""3-D stand env (cassierl_b200/csrc/tree_env.cuh) on the CPU: the device code compiled as a one-lane tile
(tests/host_harness/tree_env_harness.cpp) against the fp64 oracle and a numpy restatement of the observation and reward
(include/cassie3d.h, DESIGN.md section 11).  The numpy / oracle restatement here is also what tests/test_gpu_env3d.py
checks the kernels against."""
import ctypes as ct
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, pose3d

FOOT_SITES = ("left_contact_front", "left_contact_rear", "right_contact_front", "right_contact_rear")
PD_LOW = np.radians([-15.0, -22.5, -50.0, -164.0, -140.0] * 2)
PD_HIGH = np.radians([22.5, 22.5, 80.0, -37.0, -30.0] * 2)
KP, KD = np.full(10, 10.0), np.full(10, 5.0)


def _stale(target, deps):
    return not os.path.exists(target) or any(os.path.getmtime(d) > os.path.getmtime(target) for d in deps)


class EnvHarness:
    def __init__(self, path, xml):
        self.L = ct.CDLL(path)
        self.L.te_error.restype = ct.c_char_p
        assert self.L.te_load(xml.encode()) == 0, self.L.te_error()
        self.kp, self.kd = np.zeros(10), np.zeros(10)
        self.L.te_defaults(self.p(self.kp), self.p(self.kd))

    @staticmethod
    def p(a):
        assert a.dtype == np.float64 and a.flags.c_contiguous
        return a.ctypes.data_as(ct.POINTER(ct.c_double))

    def sites(self, q):
        out = np.zeros((4, 3))
        self.L.te_sites(self.p(np.ascontiguousarray(q, np.float64)), self.p(out))
        return out

    def observe(self, q, v):
        o = np.zeros(45)
        self.L.te_observe(self.p(np.ascontiguousarray(q, np.float64)), self.p(np.ascontiguousarray(v, np.float64)), self.p(o))
        return o

    def env_step(self, mode, q, v, w, act, n_sub=10, max_path_length=0, flags=0, length=0, reset=None, kp=None, kd=None):
        """one EnvStep of one env, (q, v, w) in place; returns done, new length, obs, reward"""
        rq, rv = reset if reset is not None else (pose3d(), np.zeros(20))
        obs, rew, ln = np.zeros(45), ct.c_double(), ct.c_int(int(length))
        done = self.L.te_env_step(int(mode), self.p(q), self.p(v), self.p(w), self.p(np.ascontiguousarray(act, np.float64)),
                                  self.p(self.kp if kp is None else np.ascontiguousarray(kp, np.float64)),
                                  self.p(self.kd if kd is None else np.ascontiguousarray(kd, np.float64)),
                                  int(n_sub), int(max_path_length), int(flags), self.p(np.ascontiguousarray(rq, np.float64)),
                                  self.p(np.ascontiguousarray(rv, np.float64)), ct.byref(ln), self.p(obs), ct.byref(rew))
        return done, ln.value, obs, rew.value


@pytest.fixture(scope="module")
def env_harness(oracle):
    src = os.path.join(ROOT, "tests", "host_harness", "tree_env_harness.cpp")
    csrc = os.path.join(ROOT, "cassierl_b200", "csrc")
    out = os.path.join(ROOT, "tests", "_build", "libtree_env_harness.so")
    deps = [src] + [os.path.join(csrc, f) for f in ("tree_env.cuh", "tree_engine.cuh", "tree_model.h", "mjcf_flatten.cpp", "mjcf_flatten.h")]
    if _stale(out, deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", out, src, os.path.join(csrc, "mjcf_flatten.cpp")])
    return EnvHarness(out, oracle.model3d_path())


# ------------------------------------------------------------------ the restatement (oracle kinematics + numpy)
def site_ids(m):
    names = [s["name"] for s in m.spec["sites"]]
    return [names.index(n) for n in FOOT_SITES]


def motor_index(m):
    """qpos / qvel index of each motor's joint (MuJoCo order)"""
    dof = np.array([m.joint_dof[a["joint"]] for a in m.spec["actuators"]])
    return dof + 1, dof


def oracle_sites(oracle, m, q):
    d = oracle.Data(m)
    d.set_state(q, np.zeros(m.nv)); d.forward()
    return np.array([d.site_pos(s) - q[:3] for s in site_ids(m)])


def obs_np(q, v, sites):
    feet = np.concatenate([sites[0:2].mean(axis=0), sites[2:4].mean(axis=0)])
    return np.concatenate([q[2:7], q[7:21], v, feet])


def reward_np(obs, act):
    c = 0.5 * (obs[39:41] + obs[42:44])
    return 1.0 - 2.0 * (0.9 - obs[0]) ** 2 - 2.0 * (c @ c) - 0.001 * np.sum(np.square(act))


def pd_step(d, target, qi, vi, kp=KP, kd=KD):
    q, v = d.state()
    d.step(kp * (target - q[qi]) - kd * v[vi])


def random_poses(n, seed):
    """standing-range joints, random (tumbled) pelvis orientations and positions"""
    rng = np.random.default_rng(seed)
    q = np.tile(pose3d(), (n, 1))
    q[:, 0:3] = rng.normal(size=(n, 3))
    qu = rng.normal(size=(n, 4)); q[:, 3:7] = qu / np.linalg.norm(qu, axis=1, keepdims=True)
    q[:, 7:] += rng.normal(size=(n, 14)) * 0.3
    return q


# ------------------------------------------------------------------ tests
def test_foot_sites_flattened(oracle, omodel3d):
    """the four contact sites are the 3rd..6th sites of cassie3d_stiff.xml, two per toe"""
    assert site_ids(omodel3d) == [2, 3, 4, 5]


def test_foot_sites_vs_oracle(oracle, omodel3d, env_harness):
    """the env's frame pass (no inertia, no forces) puts the foot sites where the oracle's forward kinematics does, at 64
    random poses with tumbled pelvis orientations"""
    worst = 0.0
    for q in random_poses(64, 0):
        worst = max(worst, np.abs(env_harness.sites(q) - oracle_sites(oracle, omodel3d, q)).max())
    assert worst < 1e-12, worst


def test_pd_trajectory_vs_oracle(oracle, omodel3d, env_harness):
    """the PD action space against an oracle loop applying the same law before every Data.step, random targets over the
    whole joint ranges held 10 steps (one EnvStep each), fp64:
    - 400 free-running simulator steps of a tumbling robot in the air (connects and leg-leg checks, no floor): 1e-10;
    - 400 simulator steps standing on the floor, every EnvStep started from the oracle's state and warm start: 1e-9.
    Free-running on the floor is not compared: sustained multi-contact standing amplifies the step's own last-bit
    differences from the oracle (PGS with its tolerance exit) by orders of magnitude within a few hundred steps."""
    qi, vi = motor_index(omodel3d)
    rng = np.random.default_rng(1)
    targets = rng.uniform(PD_LOW, PD_HIGH, (40, 10))
    q = pose3d(3.0); qu = rng.normal(size=4); q[3:7] = qu / np.linalg.norm(qu)
    v, w = rng.normal(size=20) * 0.5, np.zeros(20)
    d = oracle.Data(omodel3d); d.set_state(q, v)
    air = 0.0
    for k in range(40):
        assert env_harness.env_step(1, q, v, w, targets[k])[0] == 0
        for _ in range(10):
            pd_step(d, targets[k], qi, vi)
        qo, vo = d.state()
        air = max(air, np.abs(q - qo).max(), np.abs(v - vo).max() / max(1.0, np.abs(vo).max()))
    d = oracle.Data(omodel3d); d.set_state(pose3d(), np.zeros(20))
    ground = 0.0
    for k in range(40):
        q, v = (x.copy() for x in d.state()); w = d.warmstart().copy()
        env_harness.env_step(1, q, v, w, targets[k])
        for _ in range(10):
            pd_step(d, targets[k], qi, vi)
        qo, vo = d.state()
        ground = max(ground, np.abs(q - qo).max(), np.abs(v - vo).max() / max(1.0, np.abs(vo).max()))
    assert qo[2] > 0.8 and d.efc()["J"].shape[0] >= 12            # still standing, on its toes
    assert air < 1e-10 and ground < 1e-9, (air, ground)


def test_observation_and_reward_vs_numpy(oracle, omodel3d, env_harness):
    """the 45-d observation of a state (Observe) and the observation + reward after an EnvStep, against the numpy
    restatement with the oracle's site positions"""
    rng = np.random.default_rng(2)
    worst = 0.0
    for q in random_poses(16, 3):
        v = rng.normal(size=20)
        o = env_harness.observe(q, v)
        worst = max(worst, np.abs(o - obs_np(q, v, oracle_sites(oracle, omodel3d, q))).max())
    assert worst < 1e-12, worst
    qi, vi = motor_index(omodel3d)
    worst = 0.0
    for k in range(8):
        q, v, w = pose3d(0.95), rng.normal(size=20) * 0.1, np.zeros(20)
        act = rng.uniform(PD_LOW, PD_HIGH)
        done, ln, o, r = env_harness.env_step(1, q, v, w, act, n_sub=5, length=k)
        assert done == 0 and ln == k + 1
        ref = obs_np(q, v, oracle_sites(oracle, omodel3d, q))
        worst = max(worst, np.abs(o - ref).max(), abs(r - reward_np(ref, act)))
    assert worst < 1e-12, worst


def test_done_codes_and_reset(env_harness):
    """fell (1), time limit (3), diverged (2: reward 0, always reset, finite observation) and the episode length"""
    eh = env_harness
    rq, rv = pose3d(0.939), np.zeros(20)
    obs_reset = eh.observe(rq, rv)
    # time limit without auto-reset: done 3, the terminal state stays
    q, v, w = pose3d(0.95), np.zeros(20), np.zeros(20)
    done, ln, o, _ = eh.env_step(1, q, v, w, pose3d()[[7, 8, 9, 10, 12, 14, 15, 16, 17, 19]], n_sub=2, max_path_length=5, length=4,
                                 reset=(rq, rv))
    assert (done, ln) == (3, 5) and q[2] > 0.9
    # fell with auto-reset: the reset state's observation, or the terminal one with TERMINAL_OBS
    for flags in (1, 9):
        q, v, w = pose3d(0.3), np.zeros(20), np.ones(20)
        done, ln, o, r = eh.env_step(0, q, v, w, np.zeros(10), n_sub=1, max_path_length=5, length=4, flags=flags, reset=(rq, rv))
        assert (done, ln) == (1, 0) and np.array_equal(q, rq) and not w.any()
        assert np.array_equal(o, obs_reset) if flags == 1 else abs(o[0] - 0.3) < 0.01
    # diverged, without auto-reset: reset anyway, reward 0, finite observation of the reset state
    q, v, w = pose3d(), np.zeros(20), np.ones(20)
    q[9] = np.nan
    done, ln, o, r = eh.env_step(1, q, v, w, np.zeros(10), n_sub=1, length=3, flags=8, reset=(rq, rv))
    assert (done, ln, r) == (2, 0, 0.0) and np.array_equal(o, obs_reset) and np.array_equal(q, rq) and not w.any()
    q, v, w = pose3d(), np.zeros(20), np.zeros(20)
    v[4] = 2e10
    assert eh.env_step(0, q, v, w, np.zeros(10), n_sub=1, reset=(rq, rv))[0] == 2
