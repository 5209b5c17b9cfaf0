"""Batched 3-D Cassie (model/cassie3d_stiff.xml) on the tree engine: BASELINE.json configs[3], and a stand-task env on it
(`Cassie3dBatchEnv`).

The reference has no library or Python env for its 3-D model (SURVEY 8(d) config 4); this class is the batch analogue
of the planar `Cassie2dBatch` for it: torque actions on the ten motors (cassie3d_stiff.xml:180-191), n substeps of
mj_step per call, done when the pelvis drops below `z_done` (rule of rllab/envs/cassie_stand2d.py:131-133), auto-reset
to a standing pose.  PyTorch holds device memory and streams only; the arithmetic is in libcassie2d.so
(csrc/tree_engine.cuh through include/cassie3d.h).
"""
import ctypes as ct

import numpy as np
import torch

from . import lib as _lib

# ctrlrange of the ten motors (cassie3d_stiff.xml:181-190): abduction, yaw, hip, knee, toe per leg
TORQUE_HIGH_3D = np.array([4.5, 4.5, 12.2, 12.2, 0.9] * 2)
# ranges of the ten actuated joints (cassie3d_stiff.xml:21-84), the PD action space [rad]
PD_LOW_3D = np.radians([-15.0, -22.5, -50.0, -164.0, -140.0] * 2)
PD_HIGH_3D = np.radians([22.5, 22.5, 80.0, -37.0, -30.0] * 2)
MODE3D_BY_NAME = {"Torque": _lib.MODE3D_TORQUE, "PD": _lib.MODE3D_PD}


def _check(rc, what):
    if rc != 0:
        raise RuntimeError("libcassie2d %s failed: %s" % (what, _lib.load().Cassie3dGetLastError().decode()))


def _stream_ptr():
    return torch.cuda.current_stream().cuda_stream


class Cassie3dBatch:
    def __init__(self, n_envs, device=0, precision=32, xml_path=None, lanes=None):
        if not torch.cuda.is_available():
            raise RuntimeError("cassierl_b200 needs a CUDA device (there is no CPU fallback)")
        self.L = _lib.load()
        self.n = int(n_envs)
        self.device = torch.device("cuda", int(device))
        self.dtype = torch.float64 if precision == 64 else torch.float32
        torch.cuda.init()
        with torch.cuda.device(self.device):
            self.h = self.L.Cassie3dBatchCreate(xml_path.encode() if xml_path else None, self.n, int(device), int(precision))
        if not self.h:
            raise RuntimeError("Cassie3dBatchCreate failed: " + self.L.Cassie3dGetLastError().decode())
        sz = (ct.c_int32 * 6)()
        _check(self.L.Cassie3dBatchSizes(self.h, sz), "Sizes")
        self.nq, self.nv, self.nu, self.max_rows, self.max_contacts, self.smem_per_env = list(sz)
        if lanes is not None:
            self.set_lanes(lanes)

    def set_lanes(self, lanes):
        _check(self.L.Cassie3dBatchSetLanes(self.h, int(lanes)), "SetLanes")

    def reset_state(self):
        q = np.zeros(self.nq); v = np.zeros(self.nv)
        dp = ct.POINTER(ct.c_double)
        _check(self.L.Cassie3dBatchGetResetState(self.h, q.ctypes.data_as(dp), v.ctypes.data_as(dp)), "GetResetState")
        return q, v

    def set_reset_state(self, qpos, qvel):
        q = np.ascontiguousarray(qpos, np.float64); v = np.ascontiguousarray(qvel, np.float64)
        assert q.shape == (self.nq,) and v.shape == (self.nv,)
        dp = ct.POINTER(ct.c_double)
        _check(self.L.Cassie3dBatchSetResetState(self.h, q.ctypes.data_as(dp), v.ctypes.data_as(dp)), "SetResetState")

    def reset(self, mask=None):
        with torch.cuda.device(self.device):
            m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
            _check(self.L.Cassie3dBatchResetAll(self.h, None if m is None else m.data_ptr(), _stream_ptr()), "ResetAll")

    def set_state(self, qpos, qvel):
        q = torch.as_tensor(qpos, dtype=self.dtype, device=self.device).contiguous()
        v = torch.as_tensor(qvel, dtype=self.dtype, device=self.device).contiguous()
        assert q.shape == (self.n, self.nq) and v.shape == (self.n, self.nv)
        with torch.cuda.device(self.device):
            _check(self.L.Cassie3dBatchSetState(self.h, q.data_ptr(), v.data_ptr(), _stream_ptr()), "SetState")

    def state(self):
        q = torch.empty((self.n, self.nq), dtype=self.dtype, device=self.device)
        v = torch.empty((self.n, self.nv), dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.L.Cassie3dBatchGetState(self.h, q.data_ptr(), v.data_ptr(), _stream_ptr()), "GetState")
        return q, v

    def warm_start(self):
        w = torch.empty((self.n, self.nv), dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.L.Cassie3dBatchGetWarmStart(self.h, w.data_ptr(), _stream_ptr()), "GetWarmStart")
        return w

    def set_warm_start(self, w):
        w = torch.as_tensor(w, dtype=self.dtype, device=self.device).contiguous()
        assert w.shape == (self.n, self.nv)
        with torch.cuda.device(self.device):
            _check(self.L.Cassie3dBatchSetWarmStart(self.h, w.data_ptr(), _stream_ptr()), "SetWarmStart")

    def step(self, action=None, n=10, z_done=0.0, auto_reset=False, done=None):
        """n x mj_step with the torques `action` [N, nu] held; returns the done flags when z_done > 0 (uint8 [N])."""
        a = None
        if action is not None:
            a = torch.as_tensor(action, dtype=self.dtype, device=self.device).contiguous()
            assert a.shape == (self.n, self.nu)
        if done is None and z_done > 0:
            done = torch.empty(self.n, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.L.Cassie3dBatchStep(self.h, None if a is None else a.data_ptr(), int(n), float(z_done), int(auto_reset),
                                            None if done is None else done.data_ptr(), _stream_ptr()), "Step")
        return done

    def step_host(self, action_h, qpos_h, qvel_h, done_h, n=10, z_done=0.0, auto_reset=False):
        """host buffers in and out (pinned tensors), copies inside the call: the end-to-end path"""
        _check(self.L.Cassie3dBatchStepHost(self.h, action_h.data_ptr(), int(n), float(z_done), int(auto_reset),
                                            qpos_h.data_ptr(), qvel_h.data_ptr(), done_h.data_ptr()), "StepHost")

    def stats(self):
        s = torch.empty((self.n, 4), dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.L.Cassie3dBatchGetStats(self.h, s.data_ptr(), _stream_ptr()), "GetStats")
        return s

    def resets(self):
        r = torch.empty(self.n, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _check(self.L.Cassie3dBatchGetResets(self.h, r.data_ptr(), _stream_ptr()), "GetResets")
        return r

    def close(self):
        if self.h:
            self.L.Cassie3dBatchDestroy(self.h)
            self.h = None


class Cassie3dBatchEnv:
    """Stand-task env on the 3-D model (include/cassie3d.h, Cassie3dBatchEnvStep), the counterpart of the planar
    `Cassie2dBatchEnv(task='stand')`: 45-d observation, stand reward, done 1 (fell) / 2 (diverged) / 3 (time limit),
    auto-reset inside the step.  control_mode 'PD' (joint targets, the PD law runs at every simulator step) or 'Torque'.
    Observation, reward and done are device tensors owned by the env and overwritten by the next call."""

    def __init__(self, n_envs, device=0, control_mode="PD", precision=32, auto_reset=True, terminal_obs=False,
                 max_path_length=0, lanes=None):
        if control_mode not in MODE3D_BY_NAME:
            raise ValueError("control_mode must be 'PD' or 'Torque'")
        self.batch = Cassie3dBatch(n_envs, device, precision, lanes=lanes)
        self.n = self.batch.n
        self.control_mode = control_mode
        self.mode = MODE3D_BY_NAME[control_mode]
        self.flags = (_lib.AUTO_RESET_3D if auto_reset else 0) | (_lib.TERMINAL_OBS_3D if terminal_obs else 0)
        self.max_path_length = int(max_path_length)
        self.obs_dim, self.action_dim = _lib.OBS_DIM_3D, self.batch.nu
        b = self.batch
        self._obs = torch.empty((self.n, self.obs_dim), dtype=b.dtype, device=b.device)
        self._rew = torch.empty(self.n, dtype=b.dtype, device=b.device)
        self._done = torch.empty(self.n, dtype=torch.uint8, device=b.device)

    @property
    def observation_space(self):
        high = np.full((self.obs_dim,), 1e20)
        return -high, high

    @property
    def action_space(self):
        if self.control_mode == "Torque":
            return -TORQUE_HIGH_3D, TORQUE_HIGH_3D.copy()
        return PD_LOW_3D.copy(), PD_HIGH_3D.copy()

    def set_pd_gains(self, kp, kd):
        """per-motor gains [nu] of the PD action space (default kp = 10, kd = 5)"""
        p = np.ascontiguousarray(np.broadcast_to(np.asarray(kp, np.float64), (self.action_dim,)))
        d = np.ascontiguousarray(np.broadcast_to(np.asarray(kd, np.float64), (self.action_dim,)))
        dp = ct.POINTER(ct.c_double)
        _check(self.batch.L.Cassie3dBatchSetPdGains(self.batch.h, p.ctypes.data_as(dp), d.ctypes.data_as(dp)), "SetPdGains")

    def reset(self, mask=None):
        """every env (or the masked ones) back to the reset state; returns the observation of every env"""
        b = self.batch
        with torch.cuda.device(b.device):
            m = None if mask is None else mask.to(device=b.device, dtype=torch.uint8).contiguous()
            _check(b.L.Cassie3dBatchEnvReset(b.h, None if m is None else m.data_ptr(), self._obs.data_ptr(), _stream_ptr()), "EnvReset")
        return self._obs

    def observe(self):
        """the observation of the current state, without stepping (e.g. after batch.set_state)"""
        b = self.batch
        with torch.cuda.device(b.device):
            _check(b.L.Cassie3dBatchObserve(b.h, self._obs.data_ptr(), _stream_ptr()), "Observe")
        return self._obs

    def step(self, action, n=10):
        """n simulator steps -> obs, reward, done.  With auto_reset a done env has been reset when the call returns
        and its obs is the reset state's (terminal_obs=True keeps the terminal one)."""
        b = self.batch
        a = torch.as_tensor(action, dtype=b.dtype, device=b.device).contiguous()
        assert a.shape == (self.n, self.action_dim)
        with torch.cuda.device(b.device):
            _check(b.L.Cassie3dBatchEnvStep(b.h, self.mode, a.data_ptr(), int(n), self.max_path_length, self.flags,
                                            self._obs.data_ptr(), self._rew.data_ptr(), self._done.data_ptr(),
                                            _stream_ptr()), "EnvStep")
        return self._obs, self._rew, self._done

    def step_host(self, action_host, obs_host, reward_host, done_host, n=10):
        """end-to-end variant: pinned host tensors in and out, copies, launches and synchronisation inside the call"""
        b = self.batch
        _check(b.L.Cassie3dBatchEnvStepHost(b.h, self.mode, action_host.data_ptr(), int(n), self.max_path_length, self.flags,
                                            obs_host.data_ptr(), reward_host.data_ptr(), done_host.data_ptr()), "EnvStepHost")

    def episode_lengths(self):
        b = self.batch
        ln = torch.empty(self.n, dtype=torch.int32, device=b.device)
        with torch.cuda.device(b.device):
            _check(b.L.Cassie3dBatchGetEpisodeLengths(b.h, ln.data_ptr(), _stream_ptr()), "GetEpisodeLengths")
        return ln

    def terminate(self):
        self.batch.close()
