"""The 3-D rollout's policy prologue at any hidden_sizes (cassierl_b200/csrc/tree_rollout.cuh) on the CPU: the device code
compiled as a one-lane tile in the fast pass's scratch (tests/host_harness/rollout3d_mlp_harness.cpp), fp64, against a
numpy restatement of rllab's GaussianMLPPolicy forward and NormalizedEnv's action map, with the noise injected; and
GaussianMLPPolicy's parameter layout and initialiser."""
import ctypes as ct
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT, pose3d

SHAPES = [(32, 32), (64, 64), (128, 128), (256, 256), (100, 50, 25), (256,), (8, 8, 8, 8)]


def _stale(target, deps):
    return not os.path.exists(target) or any(os.path.getmtime(d) > os.path.getmtime(target) for d in deps)


class MlpHarness:
    def __init__(self, path, xml):
        self.L = ct.CDLL(path)
        self.L.rmh_error.restype = ct.c_char_p
        assert self.L.rmh_load(xml.encode()) == 0, self.L.rmh_error()

    @staticmethod
    def p(a):
        assert a.dtype == np.float64 and a.flags.c_contiguous
        return a.ctypes.data_as(ct.POINTER(ct.c_double))

    @staticmethod
    def sizes(shape):
        return len(shape), (ct.c_int * len(shape))(*shape)

    def params(self, shape):
        return self.L.rmh_params(*self.sizes(shape))

    def prologue(self, mode, normalize, shape, q, v, params, eps):
        obs, mean, raw, act = np.zeros(45), np.zeros(10), np.zeros(10), np.zeros(10)
        c = lambda x: np.ascontiguousarray(x, np.float64)
        self.L.rmh_prologue(int(mode), int(normalize), *self.sizes(shape), self.p(c(q)), self.p(c(v)), self.p(c(params)),
                            self.p(c(eps)), self.p(obs), self.p(mean), self.p(raw), self.p(act))
        return obs, mean, raw, act

    def box(self, mode):
        lo, hi = np.zeros(10), np.zeros(10)
        self.L.rmh_box(int(mode), self.p(lo), self.p(hi))
        return lo, hi


@pytest.fixture(scope="module")
def mlp_harness(oracle):
    src = os.path.join(ROOT, "tests", "host_harness", "rollout3d_mlp_harness.cpp")
    csrc = os.path.join(ROOT, "cassierl_b200", "csrc")
    out = os.path.join(ROOT, "tests", "_build", "librollout3d_mlp_harness.so")
    deps = [src] + [os.path.join(csrc, f) for f in ("tree_rollout.cuh", "tree_env.cuh", "tree_engine.cuh", "tree_model.h",
                                                     "mjcf_flatten.cpp", "mjcf_flatten.h")]
    if _stale(out, deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", out, src, os.path.join(csrc, "mjcf_flatten.cpp")])
    return MlpHarness(out, oracle.model3d_path())


def random_params(rng, shape, log_std):
    """a flat vector of `shape` in rllab's layout with Glorot-scaled W, non-zero biases and the given log_std"""
    widths = (45,) + tuple(shape) + (10,)
    parts = []
    for fi, fo in zip(widths[:-1], widths[1:]):
        parts += [rng.uniform(-1, 1, (fi, fo)) * np.sqrt(6.0 / (fi + fo)), rng.normal(size=fo) * 0.3]
    parts.append(np.full(10, log_std))
    return np.concatenate([x.reshape(-1) for x in parts])


def mean_np(flat, shape, obs):
    """GaussianMLPPolicy's mean: W [in][out], y = x W + b, tanh hidden layers, linear head; and log_std"""
    widths = (45,) + tuple(shape) + (10,)
    h, k = obs, 0
    for i, (fi, fo) in enumerate(zip(widths[:-1], widths[1:])):
        W = flat[k:k + fi * fo].reshape(fi, fo); k += fi * fo
        b = flat[k:k + fo]; k += fo
        h = h @ W + b
        if i < len(shape):
            h = np.tanh(h)
    assert k + 10 == flat.size
    return h, flat[k:]


def random_state(rng):
    q = pose3d(0.9 + 0.1 * rng.random())
    qu = np.array([1.0, 0, 0, 0]) + rng.normal(size=4) * 0.2
    q[3:7] = qu / np.linalg.norm(qu)
    q[7:] += rng.normal(size=14) * 0.2
    return q, rng.normal(size=20)


# ------------------------------------------------------------------ the prologue
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_prologue_vs_numpy(mlp_harness, shape):
    """mean, raw action and env action against numpy within 1e-12, in both action modes, with and without the
    normalizing map; log_std is chosen so that the clip is hit on both sides"""
    rng = np.random.default_rng(sum(shape) + len(shape))
    worst = 0.0
    clipped = 0
    for mode in (0, 1):
        lo, hi = mlp_harness.box(mode)
        for normalize in (0, 1):
            for _ in range(4):
                q, v = random_state(rng)
                scale = 1.0 if normalize else 0.5 * (hi - lo).max()
                flat, eps = random_params(rng, shape, np.log(scale)), rng.normal(size=10) * 1.5
                obs, mean, raw, act = mlp_harness.prologue(mode, normalize, shape, q, v, flat, eps)
                want, log_std = mean_np(flat, shape, obs)        # on the harness's own observation
                want_raw = want + np.exp(log_std) * eps
                x = lo + (want_raw + 1.0) * 0.5 * (hi - lo) if normalize else want_raw
                want_act = np.clip(x, lo, hi)
                worst = max(worst, np.abs(mean - want).max(), np.abs(raw - want_raw).max(), np.abs(act - want_act).max())
                clipped += int(np.sum((act == lo) | (act == hi)))
    assert worst < 1e-12, worst
    assert 0 < clipped < 2 * 2 * 4 * 10, clipped


def test_width_does_not_change_other_units(mlp_harness):
    """a unit is one serial dot product: widening the last hidden layer with zero-weight units leaves the mean bit-equal"""
    rng = np.random.default_rng(3)
    q, v = random_state(rng)
    flat = random_params(rng, (64, 40), -1.0)
    # (64, 40) -> (64, 56): 16 extra units of layer 2 with zero in- and out-weights
    W1b1 = flat[:45 * 64 + 64]
    k = W1b1.size
    W2 = flat[k:k + 64 * 40].reshape(64, 40); b2 = flat[k + 64 * 40:k + 64 * 40 + 40]; k += 64 * 40 + 40
    W3 = flat[k:k + 400].reshape(40, 10); rest = flat[k + 400:]
    wide = np.concatenate([W1b1, np.hstack([W2, np.zeros((64, 16))]).reshape(-1), np.append(b2, np.zeros(16)),
                           np.vstack([W3, np.zeros((16, 10))]).reshape(-1), rest])
    eps = rng.normal(size=10)
    a = mlp_harness.prologue(1, 1, (64, 40), q, v, flat, eps)
    b = mlp_harness.prologue(1, 1, (64, 56), q, v, wide, eps)
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_staging_fits_fast_pass_scratch(mlp_harness):
    """obs 45 + two hidden buffers of 256 + mean 10 + raw 10 reals inside the fast pass's 32 x 21 Jacobian storage"""
    assert mlp_harness.L.rmh_stage_reals() == 45 + 2 * 256 + 10 + 10 == 577
    assert mlp_harness.L.rmh_fast_j_reals() == 32 * 21 == 672


# ------------------------------------------------------------------ GaussianMLPPolicy
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_policy_layout(mlp_harness, shape):
    """n_params per shape (Python, the kernel header's count, the flat vector), unpack order against flat, mean against
    numpy"""
    from cassierl_b200 import rollout as R
    pol = R.GaussianMLPPolicy(45, 10, seed=4, device="cpu", dtype=torch.float64, hidden_sizes=shape)
    n = R.n_params(45, 10, shape)
    assert pol.hidden_sizes == tuple(shape)
    assert pol.flat.numel() == n == mlp_harness.params(shape)
    parts = pol.unpack()
    assert len(parts) == 2 * (len(shape) + 1) + 1
    widths = (45,) + tuple(shape) + (10,)
    for i, (fi, fo) in enumerate(zip(widths[:-1], widths[1:])):
        assert parts[2 * i].shape == (fi, fo) and parts[2 * i + 1].shape == (fo,)
    assert parts[-1].shape == (10,) and torch.equal(pol.log_std, parts[-1])
    assert torch.equal(torch.cat([p.reshape(-1) for p in parts]), pol.flat)
    assert torch.equal(pol.log_std, torch.full((10,), math.log(2.0), dtype=torch.float64))
    obs = torch.randn(7, 45, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    want, _ = mean_np(pol.flat.numpy(), shape, obs.numpy())
    assert np.abs(pol.mean(obs).numpy() - want).max() < 1e-12


def test_default_shape_draws_are_unchanged():
    """(32, 32) draws what the fixed-shape initialiser drew, bit for bit, in both dtypes: a restatement of it"""
    from cassierl_b200 import rollout as R

    def fixed_shape_flat(obs_dim, act_dim, init_std, seed):
        g = torch.Generator().manual_seed(seed)
        parts = []
        for fi, fo in ((obs_dim, 32), (32, 32), (32, act_dim)):
            lim = math.sqrt(6.0 / (fi + fo))
            parts += [(torch.rand(fi, fo, generator=g, dtype=torch.float64) * 2 - 1) * lim, torch.zeros(fo, dtype=torch.float64)]
        parts.append(torch.full((act_dim,), math.log(init_std), dtype=torch.float64))
        return torch.cat([p.reshape(-1) for p in parts])

    for od, ad, std, seed in ((45, 10, 2.0, 1), (45, 10, 0.5, 3), (36, 6, 2.0, 8)):
        want = fixed_shape_flat(od, ad, std, seed)
        for dt in (torch.float64, torch.float32):
            pol = R.GaussianMLPPolicy(od, ad, std, seed, "cpu", dt)
            assert pol.hidden_sizes == (32, 32) and torch.equal(pol.flat, want.to(dt))
            assert len(pol.unpack()) == 7
        assert R.n_params(od, ad) == od * 32 + 32 + 32 * 32 + 32 + 32 * ad + 2 * ad
    assert R.n_params(45, 10) == 2868
    with pytest.raises(TypeError):
        R.GaussianMLPPolicy(45, 10, 2.0, 1, "cpu", torch.float64, (64, 64))   # hidden_sizes is keyword-only
