"""The policy prologue of the 3-D rollout (cassierl_b200/csrc/tree_rollout.cuh) on the CPU: the device code compiled as
a one-lane tile (tests/host_harness/rollout3d_harness.cpp), fp64, against a numpy restatement of rllab's
GaussianMLPPolicy forward and NormalizedEnv's action map, with the noise injected."""
import ctypes as ct
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, TORQUE_HIGH_3D, pose3d
from test_env3d_host import PD_HIGH, PD_LOW, obs_np, oracle_sites

N_PARAMS = 45 * 32 + 32 + 32 * 32 + 32 + 32 * 10 + 10 + 10


def _stale(target, deps):
    return not os.path.exists(target) or any(os.path.getmtime(d) > os.path.getmtime(target) for d in deps)


class RolloutHarness:
    def __init__(self, path, xml):
        self.L = ct.CDLL(path)
        self.L.rh_error.restype = ct.c_char_p
        assert self.L.rh_load(xml.encode()) == 0, self.L.rh_error()

    @staticmethod
    def p(a):
        assert a.dtype == np.float64 and a.flags.c_contiguous
        return a.ctypes.data_as(ct.POINTER(ct.c_double))

    def box(self, mode):
        lo, hi = np.zeros(10), np.zeros(10)
        self.L.rh_box(int(mode), self.p(lo), self.p(hi))
        return lo, hi

    def prologue(self, mode, normalize, q, v, params, eps):
        obs, mean, raw, act = np.zeros(45), np.zeros(10), np.zeros(10), np.zeros(10)
        c = lambda x: np.ascontiguousarray(x, np.float64)
        self.L.rh_prologue(int(mode), int(normalize), self.p(c(q)), self.p(c(v)), self.p(c(params)), self.p(c(eps)),
                           self.p(obs), self.p(mean), self.p(raw), self.p(act))
        return obs, mean, raw, act


@pytest.fixture(scope="module")
def rollout_harness(oracle):
    src = os.path.join(ROOT, "tests", "host_harness", "rollout3d_harness.cpp")
    csrc = os.path.join(ROOT, "cassierl_b200", "csrc")
    out = os.path.join(ROOT, "tests", "_build", "librollout3d_harness.so")
    deps = [src] + [os.path.join(csrc, f) for f in ("tree_rollout.cuh", "tree_env.cuh", "tree_engine.cuh", "tree_model.h",
                                                     "mjcf_flatten.cpp", "mjcf_flatten.h")]
    if _stale(out, deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", out, src, os.path.join(csrc, "mjcf_flatten.cpp")])
    return RolloutHarness(out, oracle.model3d_path())


def random_params(rng, log_std):
    """a GaussianMLPPolicy.flat with non-zero biases (rllab initialises them to zero) and the given log_std"""
    parts = []
    for fi, fo in ((45, 32), (32, 32), (32, 10)):
        parts += [rng.uniform(-1, 1, (fi, fo)) * np.sqrt(6.0 / (fi + fo)), rng.normal(size=fo) * 0.3]
    parts.append(np.full(10, log_std))
    flat = np.concatenate([x.reshape(-1) for x in parts])
    assert flat.size == N_PARAMS
    return flat


def mean_np(flat, obs):
    """GaussianMLPPolicy's mean: W [in][out], y = x W + b, tanh hidden layers, linear head"""
    sizes = [(45, 32), (32,), (32, 32), (32,), (32, 10), (10,), (10,)]
    parts, k = [], 0
    for s in sizes:
        n = int(np.prod(s)); parts.append(flat[k:k + n].reshape(s)); k += n
    W1, b1, W2, b2, W3, b3, log_std = parts
    h = np.tanh(obs @ W1 + b1)
    h = np.tanh(h @ W2 + b2)
    return h @ W3 + b3, log_std


def test_parameter_count_and_path_codes(rollout_harness):
    assert rollout_harness.L.rh_params() == N_PARAMS == 2868
    assert [rollout_harness.L.rh_path_done(d) for d in range(4)] == [0, 1, 1, 2]


def test_action_box_from_the_model(rollout_harness):
    """torque mode: the motors' ctrlrange; PD mode: each motor's joint range -- what Cassie3dBatchEnv.action_space states"""
    lo, hi = rollout_harness.box(0)
    assert np.array_equal(lo, -TORQUE_HIGH_3D) and np.array_equal(hi, TORQUE_HIGH_3D)
    lo, hi = rollout_harness.box(1)
    assert np.abs(lo - PD_LOW).max() < 1e-12 and np.abs(hi - PD_HIGH).max() < 1e-12


def test_policy_forward_vs_numpy(oracle, omodel3d, rollout_harness):
    """observation (against the oracle's sites), mean and raw action of the prologue against numpy, 1e-12, at random
    standing-range states and random parameters"""
    rng = np.random.default_rng(5)
    worst_obs = worst = 0.0
    for i in range(16):
        q = pose3d(0.9 + 0.1 * rng.random())
        qu = np.array([1.0, 0, 0, 0]) + rng.normal(size=4) * 0.2
        q[3:7] = qu / np.linalg.norm(qu)
        q[7:] += rng.normal(size=14) * 0.2
        v = rng.normal(size=20)
        flat, eps = random_params(rng, rng.normal() * 0.5), rng.normal(size=10)
        obs, mean, raw, _ = rollout_harness.prologue(i % 2, 1, q, v, flat, eps)
        worst_obs = max(worst_obs, np.abs(obs - obs_np(q, v, oracle_sites(oracle, omodel3d, q))).max())
        want, log_std = mean_np(flat, obs)                  # on the harness's own observation
        worst = max(worst, np.abs(mean - want).max(), np.abs(raw - (want + np.exp(log_std) * eps)).max())
    assert worst_obs < 1e-12 and worst < 1e-12, (worst_obs, worst)


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("normalize", [0, 1])
def test_action_map_and_clip_vs_numpy(rollout_harness, mode, normalize):
    """NormalizedEnv's lb + (a + 1) / 2 (ub - lb) then the clip to [lb, ub] (normalize), or the clip alone, with fixed
    eps; log_std = 1 so that both bounds are hit"""
    rng = np.random.default_rng(10 + 2 * mode + normalize)
    lo, hi = rollout_harness.box(mode)
    scale = 1.0 if normalize else 0.5 * (hi - lo).max()
    clipped = 0
    worst = 0.0
    for _ in range(16):
        flat = random_params(rng, np.log(scale))
        eps = rng.normal(size=10) * 1.5
        q, v = pose3d(0.95), rng.normal(size=20) * 0.1
        _, _, raw, act = rollout_harness.prologue(mode, normalize, q, v, flat, eps)
        x = lo + (raw + 1.0) * 0.5 * (hi - lo) if normalize else raw
        want = np.clip(x, lo, hi)
        worst = max(worst, np.abs(act - want).max())
        clipped += int(np.sum((act == lo) | (act == hi)))
        assert np.all(act >= lo) and np.all(act <= hi)
    assert worst < 1e-12, worst
    assert 0 < clipped < 16 * 10, clipped
