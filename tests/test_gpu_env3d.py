"""GPU checks of the 3-D stand env (include/cassie3d.h: Cassie3dBatchEnvStep, Observe, EnvReset; cassierl_b200.envs3d
.Cassie3dBatchEnv) against the fp64 oracle with the env's semantics restated in Python (tests/test_env3d_host.py).

Where the oracle "follows" the device, every EnvStep of the oracle starts from the device's state and warm start before
that call: free-running multi-contact standing amplifies last-bit differences between the engine and the oracle (see
test_env3d_host.test_pd_trajectory_vs_oracle), so long free-running comparisons are made in the air only."""
import numpy as np
import pytest

from conftest import TORQUE_HIGH_3D, lying3d, pose3d
from test_env3d_host import PD_HIGH, PD_LOW, motor_index, obs_np, oracle_sites, pd_step, random_poses, reward_np

pytestmark = pytest.mark.gpu


def _starts(n, seed=0, z=0.945):
    """standing poses with perturbed joints, headings and small velocities"""
    rng = np.random.default_rng(seed)
    q = np.tile(pose3d(z), (n, 1))
    q[:, 7:] += rng.normal(size=(n, 14)) * 0.03
    yaw = rng.uniform(-np.pi, np.pi, n)
    q[:, 3] = np.cos(yaw / 2); q[:, 6] = np.sin(yaw / 2)
    q[:, 0:2] = rng.normal(size=(n, 2)) * 3.0
    return q, rng.normal(size=(n, 20)) * 0.05


def _err(q, v, qo, vo):
    return max(np.abs(q - qo).max(), np.abs(v - vo).max() / max(1.0, np.abs(vo).max()))


def oracle_env_step(oracle, m, q, v, w, act, mode, length, max_path_length=0, flags=0, reset=None, n_sub=10):
    """one EnvStep of one env on the oracle with the env's semantics (include/cassie3d.h)"""
    qi, vi = motor_index(m)
    d = oracle.Data(m); d.set_state(q, v); d.set_warmstart(w)
    for _ in range(n_sub):
        if mode == 1:
            pd_step(d, act, qi, vi)
        else:
            d.step(act)
    q1, v1 = d.state(); w1 = d.warmstart()
    bad = not (np.all(np.abs(q1) < 1e10) and np.all(np.abs(v1) < 1e10))
    length += 1
    done = 2 if bad else (1 if q1[2] < 0.5 else (3 if max_path_length > 0 and length >= max_path_length else 0))
    term = obs_np(q1, v1, oracle_sites(oracle, m, q1))
    rew = 0.0 if bad else reward_np(term, act)
    obs = term
    if bad or (done and flags & 1):
        q1, v1, w1 = reset[0].copy(), reset[1].copy(), np.zeros(20)
        length = 0
        if bad or not flags & 8:
            obs = obs_np(q1, v1, oracle_sites(oracle, m, q1))
    return done, rew, obs, length, q1, v1, w1


def _state(b):
    q, v = (x.cpu().numpy() for x in b.state())
    return q, v, b.warm_start().cpu().numpy()


@pytest.mark.parametrize("lanes", [8, 16, 32])
def test_env3d_pd_trajectory_vs_oracle(oracle, omodel3d, lanes):
    """fp64, 16 envs x 200 simulator steps in the PD action space, random targets over the joint ranges held 10 steps.
    Envs 0-7 tumble in the air and run free against a free-running oracle PD loop: final state 1e-8 (typically 1e-11; the
    worst env, 7e-9 on a B200 and 2e-9 on the CPU harness, drives joints through their limits, and a limit row switching on
    is a hard event that amplifies rounding differences).  Envs 8-15 stand on the floor; the oracle follows them: every
    EnvStep 1e-9 (measured 8e-12)."""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    n, steps = 16, 20
    rng = np.random.default_rng(1)
    q0, v0 = _starts(n, seed=0)
    air = np.arange(8)
    q0[air, 2] = 3.0
    qu = rng.normal(size=(8, 4)); q0[air, 3:7] = qu / np.linalg.norm(qu, axis=1, keepdims=True)
    v0[air] = rng.normal(size=(8, 20)) * 0.5
    T = rng.uniform(PD_LOW, PD_HIGH, (steps, n, 10))
    env = Cassie3dBatchEnv(n, precision=64, lanes=lanes, auto_reset=False)
    env.batch.set_state(q0, v0)
    datas = [oracle.Data(omodel3d) for _ in air]
    for e in air:
        datas[e].set_state(q0[e], v0[e])
    qi, vi = motor_index(omodel3d)
    ground, rows = 0.0, np.zeros(n, np.int64)
    for k in range(steps):
        q, v, w = _state(env.batch)
        env.step(torch.tensor(T[k]), n=10)
        q1, v1, _ = _state(env.batch)
        rows = np.maximum(rows, env.batch.stats().cpu().numpy()[:, 0])
        for e in range(8, n):
            _, _, _, _, qo, vo, _ = oracle_env_step(oracle, omodel3d, q[e], v[e], w[e], T[k, e], 1, 0)
            ground = max(ground, _err(q1[e], v1[e], qo, vo))
        for e in air:
            for _ in range(10):
                pd_step(datas[e], T[k, e], qi, vi)
    free = max(_err(q1[e], v1[e], *datas[e].state()) for e in air)
    env.terminate()
    assert free < 1e-8 and ground < 1e-9, (free, ground)
    assert rows[8:].min() >= 9 and rows[:8].max() == 6  # floor contacts for the standing envs, connect rows only in the air


def test_env3d_observe_vs_numpy(oracle, omodel3d):
    """Observe after SetState at 64 random states (tumbled pelvis orientations) against numpy + the oracle's sites:
    fp64 1e-12; fp32 1e-5 relative to max(1, |value|)"""
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    n = 64
    q = random_poses(n, 7)
    v = np.random.default_rng(8).normal(size=(n, 20))
    ref = np.stack([obs_np(q[e], v[e], oracle_sites(oracle, omodel3d, q[e])) for e in range(n)])
    for prec, tol in ((64, 1e-12), (32, 1e-5)):
        env = Cassie3dBatchEnv(n, precision=prec)
        env.batch.set_state(q, v)
        o = env.observe().cpu().numpy().astype(np.float64)
        env.terminate()
        err = np.max(np.abs(o - ref) / np.maximum(1.0, np.abs(ref)))
        assert err < tol, (prec, err)


def test_env3d_step_sequence_vs_oracle(oracle, omodel3d):
    """fp64, 24 envs x 100 EnvSteps, PD, auto-reset, max_path_length 30; a third of the envs start tumbling.  Against
    the oracle following the device with the same semantics: done bit-exact, reward and observation 1e-9, episode
    lengths bit-exact; both falls (1) and time limits (3) occur"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    n, steps, mpl = 24, 100, 30
    q0, v0 = _starts(n, seed=3)
    tilt = np.arange(0, n, 3)                          # rolled 1.2 rad, spinning, pelvis below the fall height
    q0[tilt, 2] = 0.45; q0[tilt, 3:7] = [np.cos(0.6), np.sin(0.6), 0.0, 0.0]
    v0[tilt, 3:6] += np.random.default_rng(4).normal(size=(8, 3)) * 2.0
    rng = np.random.default_rng(5)
    T = rng.uniform(PD_LOW, PD_HIGH, (steps, n, 10))
    env = Cassie3dBatchEnv(n, precision=64, max_path_length=mpl)
    reset = env.batch.reset_state()
    env.batch.set_state(q0, v0)
    lengths = np.zeros(n, np.int64)
    seen, worst = set(), 0.0
    for k in range(steps):
        q, v, w = _state(env.batch)
        obs, rew, done = (x.cpu().numpy() for x in env.step(torch.tensor(T[k]), n=10))
        ln = env.episode_lengths().cpu().numpy()
        for e in range(n):
            do, ro, oo, lengths[e], _, _, _ = oracle_env_step(oracle, omodel3d, q[e], v[e], w[e], T[k, e], 1, lengths[e], mpl, 1, reset)
            assert done[e] == do, (k, e, done[e], do)
            worst = max(worst, abs(rew[e] - ro), np.abs(obs[e] - oo).max())
            seen.add(do)
        assert (ln == lengths).all(), k
    env.terminate()
    assert worst < 1e-9, worst
    assert {1, 3} <= seen, seen


def test_env3d_terminal_obs():
    """a done env's observation: the reset state's by default, the terminal one with CASSIE3D_TERMINAL_OBS"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    n = 8
    out = {}
    for term in (False, True):
        env = Cassie3dBatchEnv(n, precision=64, terminal_obs=term, control_mode="Torque")
        first = env.reset().clone()
        q, v = (x.cpu().numpy() for x in env.batch.state())
        q[:4, 2] = 0.3                                 # half the batch below the fall height
        env.batch.set_state(q, v)
        obs, _, done = env.step(torch.zeros((n, 10), dtype=torch.float64), n=1)
        out[term] = (obs.cpu().numpy(), done.cpu().numpy(), first.cpu().numpy())
        assert (env.episode_lengths().cpu().numpy() == [0] * 4 + [1] * 4).all()
        env.terminate()
    (o0, d0, f0), (o1, d1, _) = out[False], out[True]
    assert (d0[:4] == 1).all() and (d0[4:] == 0).all() and (d1 == d0).all()
    assert np.abs(o0[:4] - f0[:4]).max() < 1e-12 and np.abs(o1[:4, 0] - 0.3).max() < 0.01
    assert np.array_equal(o0[4:], o1[4:])


def test_env3d_divergence():
    """a NaN injected with SetState: done 2, reward 0, finite observation, the env reset, its warm start zero -- without
    auto-reset too; the other envs are untouched by it"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    n = 32
    env = Cassie3dBatchEnv(n, precision=32, auto_reset=False)
    rq, rv = env.batch.reset_state()
    env.reset()
    q, v = env.batch.state()
    q[5, 9] = float("nan"); v[17, 2] = float("inf")
    env.batch.set_state(q, v)
    a = torch.tensor(np.tile(rq[[7, 8, 9, 10, 12, 14, 15, 16, 17, 19]], (n, 1)), dtype=torch.float32)
    for _ in range(3):
        obs, rew, done = (x.cpu().numpy() for x in env.step(a, n=10))
        if _ == 0:
            assert done[5] == 2 and done[17] == 2 and (np.delete(done, [5, 17]) == 0).all()
            assert rew[5] == 0 and rew[17] == 0 and np.isfinite(obs).all() and np.isfinite(rew).all()
            q2, v2 = (x.cpu().numpy() for x in env.batch.state())
            w2 = env.batch.warm_start().cpu().numpy()
            assert np.abs(q2[[5, 17]] - rq).max() < 1e-6 and np.abs(v2[[5, 17]] - rv).max() < 1e-6
            assert not w2[[5, 17]].any()
            assert (env.episode_lengths().cpu().numpy() == np.where(np.isin(np.arange(n), [5, 17]), 0, 1)).all()
    assert (done == 0).all() and np.isfinite(obs).all()
    env.terminate()


@pytest.mark.parametrize("lanes", [8, 32])
def test_env3d_two_pass_vs_oracle(oracle, omodel3d, lanes):
    """robots pressed into the floor (33-36 rows: more than the fast capacity) between standing ones, fp64, PD, three
    EnvSteps of 10 simulator steps: the handed-on envs are finished by the full-capacity pass, which also runs their
    epilogue once: state 1e-8 against the free-running oracle, observation, reward and done per step"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    n, steps = 13, 3
    q0, v0 = _starts(n, seed=21)
    for e, q in ((2, lying3d(0.10, "x", 1.5708)), (3, lying3d(0.14, "y", -1.5708, straight=True)),
                 (7, lying3d(0.12, "x", 1.5708, straight=True)), (12, lying3d(0.06, "y", 1.5708))):
        q0[e] = q; v0[e] = 0
    T = np.random.default_rng(22).uniform(PD_LOW, PD_HIGH, (steps, n, 10))
    env = Cassie3dBatchEnv(n, precision=64, lanes=lanes, auto_reset=False)
    env.batch.set_state(q0, v0)
    qo, vo, wo = q0.copy(), v0.copy(), np.zeros((n, 20))
    lengths = np.zeros(n, np.int64)
    worst = 0.0
    for k in range(steps):
        obs, rew, done = (x.cpu().numpy() for x in env.step(torch.tensor(T[k]), n=10))
        for e in range(n):
            do, ro, oo, lengths[e], qo[e], vo[e], wo[e] = oracle_env_step(oracle, omodel3d, qo[e], vo[e], wo[e], T[k, e], 1, lengths[e])
            assert done[e] == do
            worst = max(worst, abs(rew[e] - ro), np.abs(obs[e] - oo).max())
    q, v, _ = _state(env.batch)
    st = env.batch.stats().cpu().numpy()
    assert (env.episode_lengths().cpu().numpy() == steps).all()
    env.terminate()
    assert st[:, 3].sum() == 0
    assert done[[2, 3, 7, 12]].all()                   # the lying robots report a fall (no auto-reset here)
    assert worst < 1e-8 and max(_err(q[e], v[e], qo[e], vo[e]) for e in range(n)) < 1e-8, worst


def test_env3d_torque_physics_unchanged():
    """EnvStep in torque mode moves the state like Cassie3dBatchStep on a twin handle with the same inputs (fp64, ragged
    batch, 5 x 10 simulator steps): the same engine code, but a separate kernel, which ptxas may contract into FMAs
    differently -- so agreement to 1e-12, not bit for bit (in fp32 such last-bit differences grow to 1e-3 within 50
    steps of contact-rich motion)"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatch, Cassie3dBatchEnv
    n = 1000 + 3
    q0, v0 = _starts(n, seed=31)
    A = torch.tensor(np.random.default_rng(32).uniform(-1, 1, (5, n, 10)) * TORQUE_HIGH_3D, dtype=torch.float64)
    env = Cassie3dBatchEnv(n, precision=64, control_mode="Torque", auto_reset=False)
    b = Cassie3dBatch(n, precision=64)
    env.batch.set_state(q0, v0); b.set_state(q0, v0)
    for k in range(5):
        env.step(A[k].cuda(), n=10)
        b.step(A[k].cuda(), n=10)
    q1, v1 = env.batch.state(); q2, v2 = b.state()
    assert torch.equal(env.batch.stats(), b.stats())
    err = max((q1 - q2).abs().max().item(), ((v1 - v2).abs().max(dim=1).values / v2.abs().max(dim=1).values.clamp(min=1)).max().item())
    assert err < 1e-12, err
    env.terminate(); b.close()


def test_env3d_step_host_and_pd_gains():
    """EnvStepHost equals EnvStep; the PD gains are per handle and take effect"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    n = 64
    a = torch.tensor(np.random.default_rng(41).uniform(PD_LOW, PD_HIGH, (n, 10)), dtype=torch.float32)
    e1, e2, e3 = (Cassie3dBatchEnv(n, max_path_length=5) for _ in range(3))
    o1, r1, d1 = e1.step(a.cuda(), n=10)
    oh = torch.empty((n, 45)).pin_memory(); rh = torch.empty(n).pin_memory(); dh = torch.empty(n, dtype=torch.uint8).pin_memory()
    e2.step_host(a.pin_memory(), oh, rh, dh, n=10)
    assert torch.equal(o1.cpu(), oh) and torch.equal(r1.cpu(), rh) and torch.equal(d1.cpu(), dh)
    e3.set_pd_gains(np.full(10, 40.0), np.full(10, 2.0))
    o3, _, _ = e3.step(a.cuda(), n=10)
    assert not torch.equal(o1, o3)
    lo, hi = e1.action_space
    assert np.allclose(lo, PD_LOW) and np.allclose(hi, PD_HIGH)
    for e in (e1, e2, e3):
        e.terminate()
