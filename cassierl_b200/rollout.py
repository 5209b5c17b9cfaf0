"""Rollout collection for the reference's TRPO launcher (rllab/envs/trpo_cassie.py:13-55), batched:
GaussianMLPPolicy(hidden_sizes=(32, 32)) + normalize(Cassie2dEnv) + rollout(max_path_length), fused in
one CUDA kernel per T policy steps (csrc/rollout_kernels.cuh); RolloutCollector3d does the same on the 3-D stand env
(csrc/tree_rollout.cuh, one launch pass per policy step) for any hidden_sizes of 1 to 4 layers up to 256 wide.
Paths come back in rllab's dict layout (SURVEY App. E): observations[T,odim], actions[T,adim] (raw policy outputs), rewards[T],
agent_infos{mean, log_std}, env_infos{}.  The TRPO update itself is rllab's and out of scope.

DDPG's sampler (the reference's ddpg_cassie.py) runs on the 3-D collector too: DeterministicMLPPolicy explored by
OUStrategy (Cassie3dBatchRolloutOU), transitions() for the pool rows and ReplayPool, rllab's SimpleReplayPool on the
device.  The DDPG update (Q function, target networks, scale_reward) is rllab's and out of scope.
"""
import math

import numpy as np
import torch

from . import lib as _lib
from .envs import ACTION_DIM, MODE_BY_NAME, OBS_DIM, Cassie2dBatch, _stream_ptr

DEFAULT_HIDDEN_SIZES = (32, 32)   # trpo_cassie.py:21


def n_params(obs_dim, act_dim, hidden_sizes=DEFAULT_HIDDEN_SIZES, log_std=True):
    """length of GaussianMLPPolicy.flat: (in + 1) out per dense layer, plus log_std; log_std=False: the length of
    DeterministicMLPPolicy.flat"""
    n, fi = 0, obs_dim
    for fo in tuple(hidden_sizes) + (act_dim,):
        n += fi * fo + fo
        fi = fo
    return n + (act_dim if log_std else 0)


def _unpack_dense(f, widths):
    """[W1, b1, ..., W(L+1), b(L+1)] views of the front of `f` for the layer widths (in, h1, ..., out), and the rest"""
    out, k = [], 0
    for fi, fo in zip(widths[:-1], widths[1:]):
        out += [f[k:k + fi * fo].reshape(fi, fo), f[k + fi * fo:k + fi * fo + fo]]
        k += fi * fo + fo
    return out, f[k:]


class GaussianMLPPolicy:
    """Parameter container with rllab's conventions: Lasagne DenseLayer weights W[in, out] (y = x W + b),
    Glorot-uniform W, zero b, tanh hidden layers of `hidden_sizes` units, linear mean head, state-independent log_std
    initialised to log(init_std) (trpo_cassie.py:21-27: hidden_sizes=(32, 32), init_std=2.0; vpg_cassie.py uses
    (128, 128)).  `flat` is the vector rllab's get_param_values() returns: W1 b1 W2 b2 ... W(L+1) b(L+1) log_std.
    The planar collector takes (32, 32) only; RolloutCollector3d takes 1 to 4 hidden layers of 1 to 256 units."""

    def __init__(self, obs_dim, act_dim, init_std=2.0, seed=1, device="cuda", dtype=torch.float32, *,
                 hidden_sizes=DEFAULT_HIDDEN_SIZES):
        self.hidden_sizes = tuple(int(h) for h in hidden_sizes)
        g = torch.Generator().manual_seed(seed)
        widths = (obs_dim,) + self.hidden_sizes + (act_dim,)
        parts = []
        for fi, fo in zip(widths[:-1], widths[1:]):
            lim = math.sqrt(6.0 / (fi + fo))
            parts += [(torch.rand(fi, fo, generator=g, dtype=torch.float64) * 2 - 1) * lim, torch.zeros(fo, dtype=torch.float64)]
        parts.append(torch.full((act_dim,), math.log(init_std), dtype=torch.float64))
        self.obs_dim, self.act_dim = obs_dim, act_dim
        self.flat = torch.cat([p.reshape(-1) for p in parts]).to(dtype=dtype, device=device).contiguous()
        assert self.flat.numel() == n_params(obs_dim, act_dim, self.hidden_sizes)

    def unpack(self, flat=None):
        """[W1, b1, ..., W(L+1), b(L+1), log_std], views of `flat`"""
        f = self.flat if flat is None else flat
        dense, rest = _unpack_dense(f, (self.obs_dim,) + self.hidden_sizes + (self.act_dim,))
        return dense + [rest[:self.act_dim]]

    def mean(self, obs):
        """plain PyTorch reference of the kernel's forward pass (used by the tests)"""
        p = self.unpack()
        h = obs
        for i in range(0, len(p) - 3, 2):
            h = torch.tanh(h @ p[i] + p[i + 1])
        return h @ p[-3] + p[-2]

    @property
    def log_std(self):
        return self.unpack()[-1]


class DeterministicMLPPolicy:
    """rllab's DeterministicMLPPolicy(env_spec, hidden_sizes=(32, 32)) [EXT], DDPG's policy: relu hidden layers, tanh
    output layer, Lasagne's W[in, out] (y = x W + b).  Initialiser: hidden W HeUniform, U(+-sqrt(3 / fan_in)) with
    fan_in = in, hidden b zero; output W and b U(+-3e-3); drawn from one torch generator in the order W1, W2, ..., W(L+1),
    b(L+1).  `flat` is rllab's get_param_values(): W1 b1 ... W(L+1) b(L+1), no log_std.  Only RolloutCollector3d takes
    it (1 to 4 hidden layers of 1 to 256 units), with an OUStrategy."""

    def __init__(self, obs_dim, act_dim, seed=1, device="cuda", dtype=torch.float32, *, hidden_sizes=DEFAULT_HIDDEN_SIZES):
        self.hidden_sizes = tuple(int(h) for h in hidden_sizes)
        g = torch.Generator().manual_seed(seed)
        widths = (obs_dim,) + self.hidden_sizes + (act_dim,)
        u = lambda shape, lim: (torch.rand(shape, generator=g, dtype=torch.float64) * 2 - 1) * lim
        parts = []
        for fi, fo in zip(widths[:-2], widths[1:-1]):
            parts += [u((fi, fo), math.sqrt(3.0 / fi)), torch.zeros(fo, dtype=torch.float64)]
        parts.append(u((widths[-2], act_dim), 3e-3))
        parts.append(u((act_dim,), 3e-3))
        self.obs_dim, self.act_dim = obs_dim, act_dim
        self.flat = torch.cat([p.reshape(-1) for p in parts]).to(dtype=dtype, device=device).contiguous()
        assert self.flat.numel() == n_params(obs_dim, act_dim, self.hidden_sizes, log_std=False)

    def unpack(self, flat=None):
        """[W1, b1, ..., W(L+1), b(L+1)], views of `flat`"""
        f = self.flat if flat is None else flat
        dense, rest = _unpack_dense(f, (self.obs_dim,) + self.hidden_sizes + (self.act_dim,))
        assert rest.numel() == 0
        return dense

    def mean(self, obs):
        """plain PyTorch reference of the kernel's forward pass: the deterministic action before exploration"""
        p = self.unpack()
        h = obs
        for i in range(0, len(p) - 2, 2):
            h = torch.relu(h @ p[i] + p[i + 1])
        return torch.tanh(h @ p[-2] + p[-1])


class OUStrategy:
    """rllab's OUStrategy(env_spec, mu=0, theta=0.15, sigma=0.3) [EXT]: per action slot x = mu at every path start,
    then x += theta (mu - x) + sigma N(0, 1) per policy step; the action is clip(policy(o) + x, low, high).  The state
    lives in the collector's env handle (Cassie3dBatchRolloutOU); this object holds the parameters only."""

    def __init__(self, mu=0.0, theta=0.15, sigma=0.3):
        self.mu, self.theta, self.sigma = float(mu), float(theta), float(sigma)


def transitions_from_buffers(obs, act, rew, done, last_obs, include_horizon_terminal_transitions=False):
    """DDPG's pool rows of [T, N, .] path buffers, in (k, env) order: observations, actions, rewards, terminals,
    next_observations.  next_observations[k] is observations[k + 1] of the same env, `last_obs` ([N, odim], the
    observation after the last step) for k = T - 1; after a path end that is the next path's first observation, which
    rllab's pool also pairs with a terminal row.  terminals = done == 1, plus done == 2 when the flag is set; rows with
    done == 2 (cut at max_path_length) are dropped unless it is (rllab's include_horizon_terminal_transitions)."""
    T, n = done.shape
    nxt = torch.cat([obs[1:], last_obs.unsqueeze(0)]) if T else obs
    d = done.reshape(-1)
    keep = torch.ones_like(d, dtype=torch.bool) if include_horizon_terminal_transitions else d != 2
    term = (d != 0) if include_horizon_terminal_transitions else (d == 1)
    return dict(observations=obs.reshape(T * n, -1)[keep], actions=act.reshape(T * n, -1)[keep], rewards=rew.reshape(-1)[keep],
                terminals=term[keep], next_observations=nxt.reshape(T * n, -1)[keep])


class ReplayPool:
    """rllab's SimpleReplayPool(max_pool_size, observation_dim, action_dim) [EXT] on the device: a ring that overwrites
    its oldest rows, sampled uniformly with replacement.  Unlike rllab's pool it stores next_observations explicitly:
    the samples of N envs interleave, so the next stored row is another env's, not the next state.  It therefore
    draws from every stored row (rllab's excludes the newest, whose successor it has not seen).  DDPG's scale_reward
    belongs to the update and is not applied here."""

    KEYS = ("observations", "actions", "rewards", "terminals", "next_observations")

    def __init__(self, max_pool_size, obs_dim, act_dim, device="cuda", dtype=torch.float32):
        if max_pool_size < 1:
            raise ValueError("max_pool_size must be positive")
        self.max_pool_size, self.device = int(max_pool_size), torch.device(device)
        mk = lambda *s, dt=dtype: torch.zeros((self.max_pool_size,) + s, dtype=dt, device=self.device)
        self._data = dict(observations=mk(obs_dim), actions=mk(act_dim), rewards=mk(), terminals=mk(dt=torch.bool),
                          next_observations=mk(obs_dim))
        self._top, self.size = 0, 0

    def add(self, transitions):
        """append the rows of a transitions() dict; the oldest rows are overwritten once the pool is full"""
        m = int(transitions["rewards"].shape[0])
        skip = max(0, m - self.max_pool_size)            # rows that would be overwritten within this call
        idx = (self._top + skip + torch.arange(m - skip, device=self.device)) % self.max_pool_size
        for k in self.KEYS:
            self._data[k][idx] = transitions[k][skip:].to(self._data[k].device, self._data[k].dtype)
        self._top = (self._top + m) % self.max_pool_size
        self.size = min(self.size + m, self.max_pool_size)

    def random_batch(self, batch_size, generator=None):
        """`batch_size` rows drawn uniformly with replacement from the stored ones (indices from `generator` on its
        device, else the default generator of the pool's device)"""
        if self.size == 0:
            raise ValueError("the pool is empty")
        dev = generator.device if generator is not None else self.device
        idx = torch.randint(0, self.size, (int(batch_size),), generator=generator, device=dev).to(self.device)
        return {k: v[idx] for k, v in self._data.items()}


class _PathSampler:
    """Host side shared by the planar and the 3-D collector: the LinearFeatureBaseline solve on the device-accumulated
    normal equations and the split of the [T, N, .] buffers into rllab paths.  Needs batch, obs_dim, act_dim, _T."""

    def _buffers(self, T):
        if T != self._T:
            b, n = self.batch, self.batch.n
            mk = lambda *s, dt=None: torch.empty(s, dtype=dt or b.dtype, device=b.device)
            self.obs, self.act, self.mean = mk(T, n, self.obs_dim), mk(T, n, self.act_dim), mk(T, n, self.act_dim)
            self.rew, self.done = mk(T, n), mk(T, n, dt=torch.uint8)
            self._T = T

    def _solve_baseline(self, mom, D, reg_coeff):
        m = mom.cpu().numpy()
        FtF = np.zeros((D, D)); iu = np.triu_indices(D)
        FtF[iu] = m[:D * (D + 1) // 2]; FtF = FtF + FtF.T - np.diag(np.diag(FtF))
        Fty = m[D * (D + 1) // 2:]
        self.baseline_moments = (FtF, Fty)
        coeffs = None
        for _ in range(5):                           # rllab retries with a 10x larger regulariser on NaNs
            coeffs = np.linalg.lstsq(FtF + reg_coeff * np.eye(D), Fty, rcond=None)[0]
            if not np.any(np.isnan(coeffs)):
                break
            reg_coeff *= 10
        b = self.batch
        self.baseline_coeffs = torch.tensor(coeffs, dtype=b.dtype, device=b.device)
        return self.baseline_coeffs

    def paths(self, policy, envs=None):
        """Split the last collect() into rllab path dicts (one per finished or truncated episode)."""
        obs, act, mean, rew, done = (x.cpu().numpy() for x in (self.obs, self.act, self.mean, self.rew, self.done))
        det = isinstance(policy, DeterministicMLPPolicy)        # rllab's get_action returns (action, {})
        log_std = None if det else policy.log_std.cpu().numpy()
        out = []
        for e in (range(obs.shape[1]) if envs is None else envs):
            start = 0
            ends = list(np.nonzero(done[:, e])[0]) + ([obs.shape[0] - 1] if done[-1, e] == 0 else [])
            for k in ends:
                sl = slice(start, k + 1)
                out.append(dict(observations=obs[sl, e], actions=act[sl, e], rewards=rew[sl, e],
                                agent_infos={} if det else dict(mean=mean[sl, e], log_std=np.tile(log_std, (k + 1 - start, 1))),
                                env_infos={}, env=e, start=start, terminated=bool(done[k, e] == 1)))
                start = k + 1
        return out


class RolloutCollector(_PathSampler):
    """Owns the env batch and the [T, N, .] path buffers; `collect(T)` launches one kernel."""

    def __init__(self, n_envs, device=0, task="stand", control_mode="OSC", precision=32, max_path_length=1000,
                 n_substeps=10, normalize=True, reference_faithful=True, seed=1, first_global_env=0, trajectory=None):
        self.batch = Cassie2dBatch(n_envs, device, precision)
        self.task = _lib.TASK_STAND if task == "stand" else _lib.TASK_IMITATE
        self.mode = MODE_BY_NAME[control_mode]
        self.obs_dim, self.act_dim = OBS_DIM[self.task], ACTION_DIM[self.mode]
        self.max_path_length, self.n_substeps, self.normalize = max_path_length, n_substeps, normalize
        self.flags = 0 if reference_faithful else (_lib.FRESH_OBS_ON_RESET | _lib.LIVE_QSTATE)
        self.seed, self.env0 = seed, first_global_env
        if self.task == _lib.TASK_IMITATE:
            from .trajectory import Cassie2dTraj
            tr = trajectory if trajectory is not None else Cassie2dTraj()
            qq = np.ascontiguousarray(tr.qpos, np.float64)
            _lib.check(self.batch.L.Cassie2dBatchSetTrajectory(
                self.batch.h, qq.ctypes.data_as(_lib.ct.POINTER(_lib.ct.c_double)), qq.shape[0], float(tr.time[-1])), "SetTrajectory")
        # env.reset() for every env (clocks, episode counters)
        b = self.batch
        with torch.cuda.device(b.device):
            _lib.check(b.L.Cassie2dBatchEnvReset(b.h, self.task, self.flags, None, _stream_ptr()), "EnvReset")
        self._T = 0

    def collect(self, policy, T):
        if not isinstance(policy, GaussianMLPPolicy):
            raise TypeError("the planar rollout takes a GaussianMLPPolicy; DeterministicMLPPolicy runs on RolloutCollector3d")
        self._buffers(T)
        b = self.batch
        p = policy.flat.to(dtype=b.dtype, device=b.device).contiguous()
        # episodes continue across collect() calls: remember where each env's current path stands so that the
        # baseline's time features (al, al^2, al^3) of the first path of this batch start at the right index
        if getattr(self, "_path_start", None) is None:
            self._path_start = torch.empty(b.n, dtype=torch.int32, device=b.device)
        with torch.cuda.device(b.device):
            _lib.check(b.L.Cassie2dBatchGetEpisodeLengths(b.h, self._path_start.data_ptr(), _stream_ptr()), "GetEpisodeLengths")
            _lib.check(b.L.Cassie2dBatchRollout(
                b.h, self.task, self.mode, p.data_ptr(), p.numel(), int(T), self.n_substeps, self.max_path_length, self.flags,
                int(self.normalize), self.seed, self.env0, self.obs.data_ptr(), self.act.data_ptr(), self.mean.data_ptr(),
                self.rew.data_ptr(), self.done.data_ptr(), _stream_ptr()), "Rollout")
        return dict(observations=self.obs, actions=self.act, means=self.mean, rewards=self.rew, dones=self.done)

    def discounted_returns(self, gamma=0.99, tail=None):
        """returns[T, N] of the last collect() (discount 0.99: trpo_cassie.py:38), on device.  Paths still running
        when the buffer ends are truncated there: they are bootstrapped with `tail` (real [N], e.g. the baseline's
        value of the last observation) or with 0 when tail is None -- rllab's sampler truncates a batch the same way."""
        b = self.batch
        ret = torch.empty_like(self.rew)
        with torch.cuda.device(b.device):
            _lib.check(b.L.Cassie2dBatchDiscountedReturns(b.h, self.rew.data_ptr(), self.done.data_ptr(),
                                                          tail.data_ptr() if tail is not None else None, float(gamma),
                                                          int(self._T), ret.data_ptr(), _stream_ptr()), "DiscountedReturns")
        return ret

    def fit_baseline(self, returns, reg_coeff=1e-5):
        """LinearFeatureBaseline.fit (rllab [EXT]): normal equations accumulated on device, the
        D x D solve (D = 2 obs_dim + 4) on the host.  Returns the coefficient tensor (device)."""
        b = self.batch
        D = 2 * self.obs_dim + 4
        T = self._T
        if getattr(self, "_pidx", None) is None or self._pidx.shape[0] != T:
            self._pidx = torch.empty((T, b.n), dtype=torch.int32, device=b.device)
        mom = torch.empty(D * (D + 1) // 2 + D, dtype=torch.float64, device=b.device)
        with torch.cuda.device(b.device):
            _lib.check(b.L.Cassie2dBatchBaselineMoments(b.h, self.task, self.obs.data_ptr(), returns.data_ptr(), self.done.data_ptr(),
                                                        self._path_start.data_ptr(), int(T), self._pidx.data_ptr(), mom.data_ptr(),
                                                        _stream_ptr()), "BaselineMoments")
        return self._solve_baseline(mom, D, reg_coeff)

    def advantages(self, gamma=0.99, gae_lambda=1.0, coeffs=None):
        """GAE advantages and baseline values [T, N] of the last collect() (after fit_baseline)."""
        b = self.batch
        c = self.baseline_coeffs if coeffs is None else coeffs
        adv = torch.empty_like(self.rew); val = torch.empty_like(self.rew)
        with torch.cuda.device(b.device):
            _lib.check(b.L.Cassie2dBatchAdvantages(b.h, self.task, self.obs.data_ptr(), self.rew.data_ptr(), self.done.data_ptr(),
                                                   self._pidx.data_ptr(), c.data_ptr(), float(gamma), float(gae_lambda), int(self._T),
                                                   adv.data_ptr(), val.data_ptr(), _stream_ptr()), "Advantages")
        return adv, val

    def close(self):
        self.batch.close()


class RolloutCollector3d(_PathSampler):
    """The planar collector's interface on the 3-D stand env (include/cassie3d.h, Cassie3dBatchRolloutMlp):
    GaussianMLPPolicy(45, 10, hidden_sizes=...) + normalize(Cassie3dBatchEnv) + rollout(max_path_length), the policy
    taking 1 to 4 hidden layers of 1 to 256 units.  `collect(policy, T)` enqueues
    one launch pass per policy step (the policy forward, the noise and the action map are fused into the env step) and
    returns the same dict as RolloutCollector.collect; dones are path codes: 1 terminated (fell or diverged), 2 cut at
    max_path_length.  Episodes continue across collect() calls.

    DDPG's sampler: `collect(DeterministicMLPPolicy, T, es=OUStrategy(...))` (Cassie3dBatchRolloutOU); actions are then
    the clipped exploratory actions, means the deterministic outputs, and the observation after the last step is kept
    for transitions()."""

    def __init__(self, n_envs, device=0, control_mode="PD", precision=32, max_path_length=1000, n_substeps=10,
                 normalize=True, seed=1, first_global_env=0, lanes=None):
        from .envs3d import MODE3D_BY_NAME, Cassie3dBatch
        if control_mode not in MODE3D_BY_NAME:
            raise ValueError("control_mode must be 'PD' or 'Torque'")
        self.batch = Cassie3dBatch(n_envs, device, precision, lanes=lanes)
        self.control_mode, self.mode = control_mode, MODE3D_BY_NAME[control_mode]
        self.obs_dim, self.act_dim = _lib.OBS_DIM_3D, self.batch.nu
        self.max_path_length, self.n_substeps, self.normalize = int(max_path_length), int(n_substeps), normalize
        self.seed, self.env0 = seed, first_global_env
        b = self.batch
        with torch.cuda.device(b.device):
            self._check(b.L.Cassie3dBatchEnvReset(b.h, None, None, _stream_ptr()), "EnvReset")
        self._T = 0
        self._path_start = torch.empty(b.n, dtype=torch.int32, device=b.device)
        self.last_obs = None     # [n, obs_dim] after a deterministic collect

    @staticmethod
    def _check(rc, what):
        from .envs3d import _check
        _check(rc, what)

    @property
    def action_space(self):
        """(lb, ub) of the action map and clip, as the library takes them from the model"""
        lo, hi = np.zeros(self.act_dim), np.zeros(self.act_dim)
        dp = _lib.ct.POINTER(_lib.ct.c_double)
        self._check(self.batch.L.Cassie3dBatchActionBox(self.batch.h, self.mode, lo.ctypes.data_as(dp), hi.ctypes.data_as(dp)), "ActionBox")
        return lo, hi

    def collect(self, policy, T, es=None):
        """T policy steps of every env.  A GaussianMLPPolicy takes no `es`; a DeterministicMLPPolicy needs an
        OUStrategy."""
        det = isinstance(policy, DeterministicMLPPolicy)
        if not det and not isinstance(policy, GaussianMLPPolicy):
            raise TypeError("collect() takes a GaussianMLPPolicy or a DeterministicMLPPolicy")
        if det and not isinstance(es, OUStrategy):
            raise ValueError("a DeterministicMLPPolicy explores with an OUStrategy: pass es=OUStrategy(...)")
        if not det and es is not None:
            raise ValueError("a GaussianMLPPolicy draws its own noise: es must be None")
        self._buffers(T)
        b = self.batch
        p = policy.flat.to(dtype=b.dtype, device=b.device).contiguous()
        with torch.cuda.device(b.device):
            # where each env's current path stands: the in-path index of this batch's first samples (baseline features)
            self._check(b.L.Cassie3dBatchGetEpisodeLengths(b.h, self._path_start.data_ptr(), _stream_ptr()), "GetEpisodeLengths")
            hs = policy.hidden_sizes
            sizes = (_lib.ct.c_int32 * len(hs))(*hs)
            bufs = (self.obs.data_ptr(), self.act.data_ptr(), self.mean.data_ptr(), self.rew.data_ptr(), self.done.data_ptr(),
                    _stream_ptr())
            if det:
                self._check(b.L.Cassie3dBatchRolloutOU(
                    b.h, self.mode, len(hs), sizes, p.data_ptr(), p.numel(), es.mu, es.theta, es.sigma, int(T), self.n_substeps,
                    self.max_path_length, int(self.normalize), self.seed, self.env0, *bufs), "RolloutOU")
                # the next observation of the last row
                if self.last_obs is None:
                    self.last_obs = torch.empty(b.n, self.obs_dim, dtype=b.dtype, device=b.device)
                self._check(b.L.Cassie3dBatchObserve(b.h, self.last_obs.data_ptr(), _stream_ptr()), "Observe")
            else:
                self._check(b.L.Cassie3dBatchRolloutMlp(
                    b.h, self.mode, len(hs), sizes, p.data_ptr(), p.numel(), int(T), self.n_substeps,
                    self.max_path_length, int(self.normalize), self.seed, self.env0, *bufs), "Rollout")
        self._det = det
        return dict(observations=self.obs, actions=self.act, means=self.mean, rewards=self.rew, dones=self.done)

    def transitions(self, include_horizon_terminal_transitions=False):
        """the last deterministic collect() as DDPG's pool rows (transitions_from_buffers), device tensors"""
        if not getattr(self, "_det", False):
            raise RuntimeError("transitions() follows a collect() with a DeterministicMLPPolicy")
        return transitions_from_buffers(self.obs, self.act, self.rew, self.done, self.last_obs,
                                        include_horizon_terminal_transitions)

    def discounted_returns(self, gamma=0.99, tail=None):
        """returns[T, N] of the last collect(), on device; unfinished paths bootstrapped with `tail` (real [N]) or 0"""
        b = self.batch
        ret = torch.empty_like(self.rew)
        with torch.cuda.device(b.device):
            self._check(b.L.Cassie3dBatchDiscountedReturns(b.h, self.rew.data_ptr(), self.done.data_ptr(),
                                                           tail.data_ptr() if tail is not None else None, float(gamma),
                                                           int(self._T), ret.data_ptr(), _stream_ptr()), "DiscountedReturns")
        return ret

    def fit_baseline(self, returns, reg_coeff=1e-5):
        """LinearFeatureBaseline.fit: normal equations (D = 94) accumulated on device, the solve on the host"""
        b = self.batch
        D = 2 * self.obs_dim + 4
        T = self._T
        if getattr(self, "_pidx", None) is None or self._pidx.shape[0] != T:
            self._pidx = torch.empty((T, b.n), dtype=torch.int32, device=b.device)
        mom = torch.empty(D * (D + 1) // 2 + D, dtype=torch.float64, device=b.device)
        with torch.cuda.device(b.device):
            self._check(b.L.Cassie3dBatchBaselineMoments(b.h, self.obs.data_ptr(), returns.data_ptr(), self.done.data_ptr(),
                                                         self._path_start.data_ptr(), int(T), self._pidx.data_ptr(), mom.data_ptr(),
                                                         _stream_ptr()), "BaselineMoments")
        return self._solve_baseline(mom, D, reg_coeff)

    def advantages(self, gamma=0.99, gae_lambda=1.0, coeffs=None):
        """GAE advantages and baseline values [T, N] of the last collect() (after fit_baseline)."""
        b = self.batch
        c = self.baseline_coeffs if coeffs is None else coeffs
        adv = torch.empty_like(self.rew); val = torch.empty_like(self.rew)
        with torch.cuda.device(b.device):
            self._check(b.L.Cassie3dBatchAdvantages(b.h, self.obs.data_ptr(), self.rew.data_ptr(), self.done.data_ptr(),
                                                    self._pidx.data_ptr(), c.data_ptr(), float(gamma), float(gae_lambda),
                                                    int(self._T), adv.data_ptr(), val.data_ptr(), _stream_ptr()), "Advantages")
        return adv, val

    def close(self):
        self.batch.close()
