"""Rollout collection for the reference's TRPO launcher (rllab/envs/trpo_cassie.py:13-55), batched:
GaussianMLPPolicy(hidden_sizes=(32, 32)) + normalize(Cassie2dEnv) + rollout(max_path_length), fused in
one CUDA kernel per T policy steps (csrc/rollout_kernels.cuh); RolloutCollector3d does the same on the 3-D stand env
(csrc/tree_rollout.cuh, one launch pass per policy step) for any hidden_sizes of 1 to 4 layers up to 256 wide.
Paths come back in rllab's dict layout (SURVEY App. E): observations[T,odim], actions[T,adim] (raw policy outputs), rewards[T],
agent_infos{mean, log_std}, env_infos{}.  The TRPO update itself is rllab's and out of scope.
"""
import math

import numpy as np
import torch

from . import lib as _lib
from .envs import ACTION_DIM, MODE_BY_NAME, OBS_DIM, Cassie2dBatch, _stream_ptr

DEFAULT_HIDDEN_SIZES = (32, 32)   # trpo_cassie.py:21


def n_params(obs_dim, act_dim, hidden_sizes=DEFAULT_HIDDEN_SIZES):
    """length of GaussianMLPPolicy.flat: (in + 1) out per dense layer, plus log_std"""
    n, fi = 0, obs_dim
    for fo in tuple(hidden_sizes) + (act_dim,):
        n += fi * fo + fo
        fi = fo
    return n + act_dim


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
        widths = (self.obs_dim,) + self.hidden_sizes + (self.act_dim,)
        sizes = [s for fi, fo in zip(widths[:-1], widths[1:]) for s in ((fi, fo), (fo,))] + [(self.act_dim,)]
        out, k = [], 0
        for s in sizes:
            n = int(np.prod(s)); out.append(f[k:k + n].reshape(s)); k += n
        return out

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
        log_std = policy.log_std.cpu().numpy()
        out = []
        for e in (range(obs.shape[1]) if envs is None else envs):
            start = 0
            ends = list(np.nonzero(done[:, e])[0]) + ([obs.shape[0] - 1] if done[-1, e] == 0 else [])
            for k in ends:
                sl = slice(start, k + 1)
                out.append(dict(observations=obs[sl, e], actions=act[sl, e], rewards=rew[sl, e],
                                agent_infos=dict(mean=mean[sl, e], log_std=np.tile(log_std, (k + 1 - start, 1))),
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
    max_path_length.  Episodes continue across collect() calls."""

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

    def collect(self, policy, T):
        self._buffers(T)
        b = self.batch
        p = policy.flat.to(dtype=b.dtype, device=b.device).contiguous()
        with torch.cuda.device(b.device):
            # where each env's current path stands: the in-path index of this batch's first samples (baseline features)
            self._check(b.L.Cassie3dBatchGetEpisodeLengths(b.h, self._path_start.data_ptr(), _stream_ptr()), "GetEpisodeLengths")
            hs = policy.hidden_sizes
            self._check(b.L.Cassie3dBatchRolloutMlp(
                b.h, self.mode, len(hs), (_lib.ct.c_int32 * len(hs))(*hs), p.data_ptr(), p.numel(), int(T), self.n_substeps,
                self.max_path_length, int(self.normalize), self.seed, self.env0, self.obs.data_ptr(), self.act.data_ptr(),
                self.mean.data_ptr(), self.rew.data_ptr(), self.done.data_ptr(), _stream_ptr()), "Rollout")
        return dict(observations=self.obs, actions=self.act, means=self.mean, rewards=self.rew, dones=self.done)

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
