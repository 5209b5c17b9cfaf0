"""DDPG's sampler on the 3-D rollout, on the CPU: the deterministic kind of the policy prologue
(cassierl_b200/csrc/tree_rollout.cuh, kPolicyOu3d) compiled as a one-lane tile in the fast pass's scratch
(tests/host_harness/rollout3d_ou_harness.cpp), fp64, against a numpy restatement of rllab's DeterministicMLPPolicy,
OUStrategy and NormalizedEnv's action map, with eps and the prior OU state injected; and on CPU tensors
DeterministicMLPPolicy's layout and initialiser, the index logic of transitions() and ReplayPool."""
import ctypes as ct
import math
import os
import subprocess

import numpy as np
import pytest
import torch

from conftest import ROOT
from test_rollout3d_mlp_host import SHAPES, _stale, random_state


class OuHarness:
    def __init__(self, path, xml):
        self.L = ct.CDLL(path)
        self.L.roh_error.restype = ct.c_char_p
        self.L.roh_prologue.argtypes = [ct.c_int, ct.c_int, ct.c_int, ct.c_void_p] + [ct.c_void_p] * 4 + [ct.c_double] * 3 + \
            [ct.c_void_p, ct.c_int] + [ct.c_void_p] * 5
        assert self.L.roh_load(xml.encode()) == 0, self.L.roh_error()

    @staticmethod
    def p(a):
        assert a.dtype == np.float64 and a.flags.c_contiguous
        return a.ctypes.data

    @staticmethod
    def sizes(shape):
        return len(shape), (ct.c_int * len(shape))(*shape)

    def params(self, shape):
        return self.L.roh_params(*self.sizes(shape))

    def prologue(self, mode, normalize, shape, q, v, params, eps, mu, theta, sigma, x_prev, path_start, x_next=None):
        """obs, mean, raw, env action, advanced OU state; x_next given: the state is written there (may be x_prev)"""
        obs, mean, raw, act = np.zeros(45), np.zeros(10), np.zeros(10), np.zeros(10)
        xn = np.zeros(10) if x_next is None else x_next
        c = lambda x: np.ascontiguousarray(x, np.float64)
        q, v, params, eps = c(q), c(v), c(params), c(eps)
        n, sz = self.sizes(shape)
        self.L.roh_prologue(int(mode), int(normalize), n, ct.cast(sz, ct.c_void_p), self.p(q), self.p(v), self.p(params),
                            self.p(eps), float(mu), float(theta), float(sigma), self.p(x_prev), int(path_start), self.p(obs),
                            self.p(mean), self.p(raw), self.p(act), self.p(xn))
        return obs, mean, raw, act, xn

    def box(self, mode):
        lo, hi = np.zeros(10), np.zeros(10)
        dp = ct.POINTER(ct.c_double)
        self.L.roh_box(int(mode), lo.ctypes.data_as(dp), hi.ctypes.data_as(dp))
        return lo, hi


@pytest.fixture(scope="module")
def ou_harness(oracle):
    src = os.path.join(ROOT, "tests", "host_harness", "rollout3d_ou_harness.cpp")
    csrc = os.path.join(ROOT, "cassierl_b200", "csrc")
    out = os.path.join(ROOT, "tests", "_build", "librollout3d_ou_harness.so")
    deps = [src] + [os.path.join(csrc, f) for f in ("tree_rollout.cuh", "tree_env.cuh", "tree_engine.cuh", "tree_model.h",
                                                     "mjcf_flatten.cpp", "mjcf_flatten.h")]
    if _stale(out, deps):
        os.makedirs(os.path.dirname(out), exist_ok=True)
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-o", out, src, os.path.join(csrc, "mjcf_flatten.cpp")])
    return OuHarness(out, oracle.model3d_path())


def random_det_params(rng, shape):
    """a flat vector of `shape` in DeterministicMLPPolicy's layout, scaled so that the tanh head is not saturated"""
    widths = (45,) + tuple(shape) + (10,)
    parts = []
    for fi, fo in zip(widths[:-1], widths[1:]):
        parts += [rng.uniform(-1, 1, (fi, fo)) * np.sqrt(3.0 / fi), rng.normal(size=fo) * 0.3]
    return np.concatenate([x.reshape(-1) for x in parts])


def det_mean_np(flat, shape, obs):
    """DeterministicMLPPolicy's action: W [in][out], y = x W + b, relu hidden layers, tanh head"""
    widths = (45,) + tuple(shape) + (10,)
    h, k = obs, 0
    for i, (fi, fo) in enumerate(zip(widths[:-1], widths[1:])):
        W = flat[k:k + fi * fo].reshape(fi, fo); k += fi * fo
        b = flat[k:k + fo]; k += fo
        h = h @ W + b
        h = np.maximum(h, 0.0) if i < len(shape) else np.tanh(h)
    assert k == flat.size
    return h


def ou_np(x_prev, path_start, mu, theta, sigma, eps):
    x = np.full(10, mu) if path_start else x_prev
    return x + theta * (mu - x) + sigma * eps


def action_np(mean, x, lo, hi, normalize):
    """(raw, env action): the clipped exploratory action in [-1, 1] (normalize) or the box, then the map and clip"""
    if normalize:
        raw = np.clip(mean + x, -1.0, 1.0)
        return raw, np.clip(lo + (raw + 1.0) * 0.5 * (hi - lo), lo, hi)
    raw = np.clip(mean + x, lo, hi)
    return raw, np.clip(raw, lo, hi)


# ------------------------------------------------------------------ the prologue
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_prologue_vs_numpy(ou_harness, shape):
    """mean, OU step, clipped action and env action against numpy within 1e-12, in both action modes, with and without
    normalize, at path starts and within paths; the OU scale is chosen so that the clip is hit on both sides"""
    rng = np.random.default_rng(100 + sum(shape) + len(shape))
    worst, clipped, n = 0.0, 0, 0
    for mode in (0, 1):
        lo, hi = ou_harness.box(mode)
        for normalize in (0, 1):
            scale = 1.0 if normalize else 0.5 * (hi - lo).max()
            for it in range(4):
                q, v = random_state(rng)
                flat, eps = random_det_params(rng, shape), rng.normal(size=10) * 1.5
                mu, theta, sigma = rng.normal() * 0.3 * scale, 0.15 + 0.1 * it, 0.5 * scale
                x_prev = rng.normal(size=10) * scale
                start = it % 2
                obs, mean, raw, act, xn = ou_harness.prologue(mode, normalize, shape, q, v, flat, eps, mu, theta, sigma,
                                                              x_prev, start)
                want = det_mean_np(flat, shape, obs)               # on the harness's own observation
                want_x = ou_np(x_prev, start, mu, theta, sigma, eps)
                want_raw, want_act = action_np(want, want_x, lo, hi, normalize)
                worst = max(worst, *(np.abs(a - b).max() for a, b in ((mean, want), (xn, want_x), (raw, want_raw),
                                                                       (act, want_act))))
                b_lo, b_hi = (-1.0, 1.0) if normalize else (lo, hi)
                clipped += int(np.sum(raw == b_lo)) + int(np.sum(raw == b_hi))
                n += 10
    assert worst < 1e-12, worst
    assert 0 < clipped < n, clipped


def test_ou_recurrence_in_place(ou_harness):
    """twelve steps advancing the state in place (x_next is x_prev, as in the kernel), a path start at steps 0 and 7:
    the state follows the numpy recurrence and restarts from mu"""
    rng = np.random.default_rng(8)
    shape, mu, theta, sigma = (32, 32), 0.2, 0.15, 0.3
    flat = random_det_params(rng, shape)
    q, v = random_state(rng)
    x = np.full(10, 5.0)                     # the stale state of a previous path: overwritten at the first start
    want = x.copy()
    for k in range(12):
        eps = rng.normal(size=10)
        start = k in (0, 7)
        ou_harness.prologue(1, 1, shape, q, v, flat, eps, mu, theta, sigma, x, start, x_next=x)
        want = ou_np(want, start, mu, theta, sigma, eps)
        assert np.abs(x - want).max() < 1e-12, k
        if start:
            assert np.abs(x - (mu + sigma * eps)).max() < 1e-12     # theta (mu - mu) = 0 at a path start


def test_zero_sigma_is_the_deterministic_action(ou_harness):
    """sigma = 0 and mu = 0 at a path start: the clipped action is the deterministic mean, bit for bit"""
    rng = np.random.default_rng(9)
    for shape in SHAPES:
        flat = random_det_params(rng, shape)
        q, v = random_state(rng)
        _, mean, raw, _, xn = ou_harness.prologue(0, 1, shape, q, v, flat, rng.normal(size=10), 0.0, 0.15, 0.0,
                                                  np.full(10, 3.0), 1)
        assert np.array_equal(raw, mean) and np.array_equal(xn, np.zeros(10)), shape


# ------------------------------------------------------------------ DeterministicMLPPolicy
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_policy_layout_and_initialiser(ou_harness, shape):
    """n_params without log_std (Python, the kernel header's count, the flat vector), unpack order against flat, rllab's
    initialiser bounds, mean against numpy"""
    from cassierl_b200 import rollout as R
    pol = R.DeterministicMLPPolicy(45, 10, seed=4, device="cpu", dtype=torch.float64, hidden_sizes=shape)
    n = R.n_params(45, 10, shape, log_std=False)
    assert n == R.n_params(45, 10, shape) - 10
    assert pol.hidden_sizes == tuple(shape)
    assert pol.flat.numel() == n == ou_harness.params(shape)
    parts = pol.unpack()
    assert len(parts) == 2 * (len(shape) + 1)
    widths = (45,) + tuple(shape) + (10,)
    for i, (fi, fo) in enumerate(zip(widths[:-1], widths[1:])):
        W, b = parts[2 * i], parts[2 * i + 1]
        assert W.shape == (fi, fo) and b.shape == (fo,)
        if i < len(shape):                   # HeUniform, zero bias
            lim = math.sqrt(3.0 / fi)
            assert W.abs().max() <= lim and W.abs().max() > 0.9 * lim and not b.any()
        else:                                # U(+-3e-3) weights and bias
            assert W.abs().max() <= 3e-3 and b.abs().max() <= 3e-3 and b.any()
    assert torch.equal(torch.cat([p.reshape(-1) for p in parts]), pol.flat)
    obs = torch.randn(7, 45, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    assert np.abs(pol.mean(obs).numpy() - det_mean_np(pol.flat.numpy(), shape, obs.numpy())).max() < 1e-12
    again = R.DeterministicMLPPolicy(45, 10, seed=4, device="cpu", dtype=torch.float32, hidden_sizes=shape)
    assert torch.equal(again.flat, pol.flat.float())


def test_ou_strategy_defaults():
    from cassierl_b200 import rollout as R
    es = R.OUStrategy()
    assert (es.mu, es.theta, es.sigma) == (0.0, 0.15, 0.3)


# ------------------------------------------------------------------ transitions() index logic
def _buffers(T=5, n=3, od=4, ad=2):
    obs = torch.arange(T * n * od, dtype=torch.float64).reshape(T, n, od)
    act = -torch.arange(T * n * ad, dtype=torch.float64).reshape(T, n, ad)
    rew = torch.arange(T * n, dtype=torch.float64).reshape(T, n) * 0.5
    done = torch.zeros(T, n, dtype=torch.uint8)
    done[1, 0] = 1; done[3, 0] = 2; done[2, 2] = 2; done[4, 1] = 1
    last = 1000 + torch.arange(n * od, dtype=torch.float64).reshape(n, od)
    return obs, act, rew, done, last


@pytest.mark.parametrize("include", [False, True])
def test_transitions_index_logic(include):
    """(k, env) order, next observation = the same env's next row or the recorded last observation, terminals and the
    dropped rows of paths cut at max_path_length"""
    from cassierl_b200.rollout import transitions_from_buffers
    obs, act, rew, done, last = _buffers()
    T, n = done.shape
    tr = transitions_from_buffers(obs, act, rew, done, last, include)
    rows = [(k, e) for k in range(T) for e in range(n) if include or done[k, e] != 2]
    assert len(rows) == (T * n if include else T * n - 2)
    assert tr["terminals"].dtype == torch.bool
    for i, (k, e) in enumerate(rows):
        assert torch.equal(tr["observations"][i], obs[k, e])
        assert torch.equal(tr["actions"][i], act[k, e])
        assert float(tr["rewards"][i]) == float(rew[k, e])
        assert torch.equal(tr["next_observations"][i], obs[k + 1, e] if k + 1 < T else last[e])
        assert bool(tr["terminals"][i]) == (done[k, e] == 1 or (include and done[k, e] == 2))
    assert int(tr["terminals"].sum()) == (4 if include else 2)


# ------------------------------------------------------------------ ReplayPool
def test_replay_pool_wraps_around():
    """rows land in a ring of max_pool_size: the oldest are overwritten, also by a batch larger than the pool"""
    from cassierl_b200.rollout import ReplayPool
    pool = ReplayPool(7, 2, 1, device="cpu", dtype=torch.float64)

    def batch(start, m):
        i = torch.arange(start, start + m, dtype=torch.float64)
        return dict(observations=i[:, None].repeat(1, 2), actions=-i[:, None], rewards=i, terminals=(i % 3) == 0,
                    next_observations=i[:, None].repeat(1, 2) + 0.5)

    pool.add(batch(0, 4))
    assert pool.size == 4
    pool.add(batch(4, 5))                    # 9 rows into 7: rows 0 and 1 overwritten
    assert pool.size == 7
    assert sorted(pool._data["rewards"].tolist()) == list(range(2, 9))
    assert torch.equal(pool._data["rewards"], torch.tensor([7, 8, 2, 3, 4, 5, 6], dtype=torch.float64))
    pool.add(batch(100, 10))                 # larger than the pool: its last 7 rows, in ring order from the top
    assert pool.size == 7
    assert sorted(pool._data["rewards"].tolist()) == list(range(103, 110))
    d = pool._data
    assert torch.equal(d["observations"][:, 0], d["rewards"]) and torch.equal(d["actions"][:, 0], -d["rewards"])
    assert torch.equal(d["next_observations"][:, 1], d["rewards"] + 0.5)
    assert torch.equal(d["terminals"], (d["rewards"] % 3) == 0)
    pool.add(batch(200, 1))                  # the ring continues where it stopped
    assert sorted(pool._data["rewards"].tolist()) == list(range(104, 110)) + [200]


def test_replay_pool_seeded_sampling():
    """random_batch draws uniformly with replacement over the stored rows only, reproducibly for a seeded generator"""
    from cassierl_b200.rollout import ReplayPool
    pool = ReplayPool(1000, 3, 2, device="cpu", dtype=torch.float32)
    with pytest.raises(ValueError):
        pool.random_batch(4)
    i = torch.arange(300, dtype=torch.float32)
    pool.add(dict(observations=i[:, None].repeat(1, 3), actions=i[:, None].repeat(1, 2), rewards=i,
                  terminals=torch.zeros(300, dtype=torch.bool), next_observations=i[:, None].repeat(1, 3) + 1))
    a = pool.random_batch(256, generator=torch.Generator().manual_seed(5))
    b = pool.random_batch(256, generator=torch.Generator().manual_seed(5))
    for k in a:
        assert torch.equal(a[k], b[k]), k
    assert a["observations"].shape == (256, 3) and a["terminals"].shape == (256,)
    assert torch.equal(a["observations"][:, 0], a["rewards"]) and torch.equal(a["next_observations"][:, 0], a["rewards"] + 1)
    big = pool.random_batch(60000, generator=torch.Generator().manual_seed(6))["rewards"]
    assert big.max() == 299 and big.min() == 0                      # only stored rows, the newest included
    counts = torch.bincount(big.long(), minlength=300).double()
    assert abs(counts.mean() - 200) < 1e-9 and counts.std() < 30    # uniform: binomial std ~14
    assert len(torch.unique(pool.random_batch(256, generator=torch.Generator().manual_seed(7))["rewards"])) < 256
