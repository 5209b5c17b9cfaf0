"""Rollout collection on the 3-D stand env (Cassie3dBatchRollout, k_tree_rollout_step, RolloutCollector3d) on the GPU:
the fused policy forward against the PyTorch reference, the noise against a numpy Philox4x32-10 + Box-Muller, sharding
invariance, the transitions against Cassie3dBatchEnv.step replaying the recorded actions, the launch knobs (one worker
process per setting, tests/rollout3d_variants_worker.py), the path bookkeeping, the sampler side (returns,
LinearFeatureBaseline moments, GAE) against numpy, and argument validation."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, lying3d, pose3d
from test_gpu_rollout import philox4x32_10

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

KNOBS = ("CASSIE3D_TWO_PASS", "CASSIE3D_STEP_BARRIER", "CASSIE3D_TILES", "CASSIE3D_SORT", "CASSIE3D_LANES")


def normal10(seed, env, step):
    """the ten standard normals of (seed, env, step): blocks 0 and 1 as the planar rollout, then the first pair of block 2"""
    out = []
    for b in range(3):
        c = philox4x32_10([env, step, b, 0], seed & 0xFFFFFFFF, seed >> 32)
        for p in range(2 if b < 2 else 1):
            u1 = (np.float32(c[2 * p] >> 8) + np.float32(1)) * np.float32(1 / 16777216.0)
            u2 = np.float32(c[2 * p + 1] >> 8) * np.float32(1 / 16777216.0)
            rad = np.sqrt(np.float32(-2) * np.log(u1))
            out += [rad * np.cos(np.float32(2 * np.pi) * u2), rad * np.sin(np.float32(2 * np.pi) * u2)]
    return np.array(out, np.float64)


def path_codes(env_done):
    """Cassie3dBatchEnvStep's done codes -> the rollout's: fell / diverged -> 1, time limit -> 2"""
    return torch.where(env_done == 3, 2, torch.where(env_done != 0, 1, 0)).to(torch.uint8)


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    from cassierl_b200 import rollout
    return rollout


# ------------------------------------------------------------------ 1. forward, noise, action map
@pytest.mark.parametrize("lanes", [8, 16, 32])
@pytest.mark.parametrize("mode", ["PD", "Torque"])
def test_policy_forward_noise_and_action_map(R, mode, lanes):
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    n, T = 101, 6
    col = R.RolloutCollector3d(n, control_mode=mode, precision=32, seed=12345, first_global_env=1000, lanes=lanes)
    pol = R.GaussianMLPPolicy(col.obs_dim, col.act_dim, seed=3)
    out = col.collect(pol, T)
    obs, act, mean = out["observations"], out["actions"], out["means"]
    assert obs.shape == (T, n, 45) and act.shape == (T, n, 10)
    assert torch.isfinite(obs).all() and torch.isfinite(act).all()
    ref = pol.mean(obs.reshape(-1, col.obs_dim)).reshape(T, n, col.act_dim)
    assert float((mean - ref).abs().max() / ref.abs().max().clamp(min=1)) < 1e-5
    eps = ((act - mean) / pol.log_std.exp()).cpu().numpy().astype(np.float64)
    for (k, e) in ((0, 0), (0, 17), (3, 100), (5, 40), (2, 63)):
        want = normal10(12345, 1000 + e, k)
        assert np.allclose(eps[k, e], want, atol=2e-5 * max(1.0, np.abs(want).max())), (k, e)
    assert abs(eps.mean()) < 0.1 and abs(eps.std() - 1.0) < 0.1
    # the box the library maps into is the env's action space
    env = Cassie3dBatchEnv(1, control_mode=mode)
    for got, want in zip(col.action_space, env.action_space):
        assert np.abs(got - want).max() < 1e-12
    env.terminate(); col.close()


# ------------------------------------------------------------------ 2. sharding invariance
@pytest.mark.parametrize("mode", ["PD", "Torque"])
def test_sharding_invariance(R, mode):
    """32 envs at global ids 1037.. reproduce that slice of a 101-env run bit for bit (the offset is not at a CTA
    boundary): what the multi-GPU gather relies on"""
    T = 6
    pol = R.GaussianMLPPolicy(45, 10, seed=3)
    col = R.RolloutCollector3d(101, control_mode=mode, precision=32, seed=12345, first_global_env=1000)
    out = {k: v.clone() for k, v in col.collect(pol, T).items()}
    col2 = R.RolloutCollector3d(32, control_mode=mode, precision=32, seed=12345, first_global_env=1037)
    out2 = col2.collect(pol, T)
    for k in ("observations", "actions", "means", "rewards", "dones"):
        assert torch.equal(out2[k], out[k][:, 37:69]), k
    col.close(); col2.close()


# ------------------------------------------------------------------ 3. transitions equal EnvStep
@pytest.mark.parametrize("mode", ["PD", "Torque"])
def test_transitions_match_env_step(R, mode):
    """Replaying the recorded actions (mapped and clipped) through Cassie3dBatchEnv(auto_reset, max_path_length=12) from
    the same start state reproduces the rollout's observations, rewards and done codes (fp64).  A third of the envs start
    tipped over low (falls), three lie on the floor (steps beyond the fast capacity, finished by the continuation pass)."""
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    n, T, mpl = 24, 30, 12
    rng = np.random.default_rng(4)
    q0 = np.tile(pose3d(0.945), (n, 1)); q0[:, 7:] += rng.normal(size=(n, 14)) * 0.03
    v0 = rng.normal(size=(n, 20)) * 0.05
    for e in range(0, n, 3):
        q0[e, 2] = 0.62; q0[e, 3:7] = [np.cos(0.6), 0.0, np.sin(0.6), 0.0]
    for e in (1, 11, n - 1):
        q0[e] = lying3d(0.10); v0[e] = 0
    col = R.RolloutCollector3d(n, control_mode=mode, precision=64, max_path_length=mpl, seed=7, first_global_env=3)
    col.batch.set_state(q0, v0)
    pol = R.GaussianMLPPolicy(col.obs_dim, col.act_dim, seed=5, dtype=torch.float64)
    first = {k: v.clone() for k, v in col.collect(pol, 1).items()}
    assert int((col.batch.stats()[:, 0] > 32).sum()) >= 1     # the continuation pass finished this step
    rest = col.collect(pol, T - 1)
    out = {k: torch.cat([first[k], rest[k]]) for k in first}
    env = Cassie3dBatchEnv(n, control_mode=mode, precision=64, auto_reset=True, max_path_length=mpl)
    env.batch.set_state(q0, v0)
    o = env.observe().clone()
    lo, hi = (torch.tensor(x, dtype=torch.float64, device=o.device) for x in col.action_space)
    err_o = err_r = 0.0
    for k in range(T):
        err_o = max(err_o, float((out["observations"][k] - o).abs().max()))
        a = (lo + (out["actions"][k] + 1.0) * 0.5 * (hi - lo)).clamp(lo, hi)
        o, r, d = env.step(a, n=10)
        o = o.clone()
        err_r = max(err_r, float((out["rewards"][k] - r).abs().max()))
        assert torch.equal(out["dones"][k], path_codes(d)), k
    print("max |obs diff| %.3e  max |reward diff| %.3e" % (err_o, err_r))
    assert err_o < 1e-9 and err_r < 1e-9, (err_o, err_r)
    codes = set(np.unique(out["dones"].cpu().numpy()).tolist())
    assert {1, 2} <= codes, codes
    col.close(); env.terminate()


# ------------------------------------------------------------------ 4. launch knobs
SETTINGS = {"default": {}, "tiles7": {"CASSIE3D_TILES": "7"}, "no_barrier": {"CASSIE3D_STEP_BARRIER": "0"},
            "one_pass": {"CASSIE3D_TWO_PASS": "0"}}


@pytest.fixture(scope="module")
def variant_runs(tmp_path_factory):
    d = tmp_path_factory.mktemp("rollout3d_variants")
    worker = os.path.join(ROOT, "tests", "rollout3d_variants_worker.py")
    procs = {}
    try:
        for name, knobs in SETTINGS.items():
            env = {k: v for k, v in os.environ.items() if k not in KNOBS}
            env.update(knobs)
            if sys.flags.no_user_site:
                env["PYTHONNOUSERSITE"] = "1"
            log = open(d / (name + ".log"), "w")
            procs[name] = (subprocess.Popen([sys.executable, worker, str(d / (name + ".npz"))], cwd=ROOT, env=env,
                                            stdout=log, stderr=subprocess.STDOUT), log)
        runs = {}
        for name, (p, log) in procs.items():
            rc = p.wait(timeout=900)
            log.close()
            text = (d / (name + ".log")).read_text()
            assert rc == 0, "worker %s failed:\n%s" % (name, text[-3000:])
            with np.load(d / (name + ".npz")) as z:
                runs[name] = dict(z)
        return runs
    finally:
        for p, log in procs.values():
            if p.poll() is None:
                p.kill()
                p.wait()
            log.close()


@pytest.mark.parametrize("setting", ["tiles7", "no_barrier"])
def test_launch_knob_is_bit_identical(variant_runs, setting):
    base, run = variant_runs["default"], variant_runs[setting]
    assert sorted(base) == sorted(run)
    bad = [k for k in base if not np.array_equal(base[k], run[k], equal_nan=True)]
    assert not bad, bad


def test_single_pass_agrees(variant_runs):
    """CASSIE3D_TWO_PASS=0: identical done codes in both precisions, fp64 within 1e-9"""
    base, run = variant_runs["default"], variant_runs["one_pass"]
    assert base["p64_l32_dones"].any()
    worst = 0.0
    for k in base:
        if k.endswith(("_dones", "_resets")):
            assert np.array_equal(base[k], run[k]), k
        elif k.startswith("p64_"):
            worst = max(worst, float(np.abs(base[k] - run[k]).max()))
    assert worst < 1e-9, worst


# ------------------------------------------------------------------ 5. path bookkeeping
def test_paths_bookkeeping(R):
    n, T, seed = 8, 10, 1
    col = R.RolloutCollector3d(n, control_mode="Torque", precision=32, max_path_length=4, seed=seed)
    pol = R.GaussianMLPPolicy(col.obs_dim, col.act_dim, seed=2)
    out = col.collect(pol, T)
    d = out["dones"].cpu().numpy()
    paths = col.paths(pol)
    assert sum(len(p["rewards"]) for p in paths) == n * T
    for p in paths:
        ln = len(p["rewards"])
        assert ln <= 4
        assert p["observations"].shape == (ln, 45) and p["actions"].shape == (ln, 10)
        assert p["agent_infos"]["mean"].shape == (ln, 10) and p["agent_infos"]["log_std"].shape == (ln, 10)
    cut = [e for e in range(n) if (d[:, e] == 1).sum() == 0]
    assert cut
    for e in cut:
        assert list(np.nonzero(d[:, e])[0]) == [3, 7]
    # episodes and the noise counter continue across collect() calls
    out = col.collect(pol, 2)
    d2 = out["dones"].cpu().numpy()
    for e in cut:
        if (d2[:, e] == 1).sum() == 0:
            assert list(np.nonzero(d2[:, e])[0]) == [1]
    eps = ((out["actions"][0] - out["means"][0]) / pol.log_std.exp()).cpu().numpy().astype(np.float64)
    assert np.allclose(eps[5], normal10(seed, 5, T), atol=2e-5 * 4)
    col.close()


# ------------------------------------------------------------------ 6. sampler side
def test_returns_baseline_and_gae(R):
    """discounted returns (numpy scan and rllab's per-path discount_cumsum), the LinearFeatureBaseline normal equations
    (D = 94), values and GAE advantages per path against numpy, fp64.  The first collect() leaves paths running, so the
    time features of the second batch's first paths start at the envs' episode lengths."""
    n, T, mpl, gamma, lam = 128, 40, 15, 0.99, 0.97
    col = R.RolloutCollector3d(n, control_mode="PD", precision=64, max_path_length=mpl, seed=11)
    pol = R.GaussianMLPPolicy(col.obs_dim, col.act_dim, seed=4, dtype=torch.float64)
    col.collect(pol, 7)
    col.collect(pol, T)
    start0 = col._path_start.cpu().numpy()
    assert start0.max() > 0
    ret = col.discounted_returns(gamma)
    retn = ret.cpu().numpy(); rew = col.rew.cpu().numpy(); done = col.done.cpu().numpy()
    want = np.zeros_like(rew); acc = np.zeros(n)
    for k in range(T - 1, -1, -1):
        acc = rew[k] + np.where(done[k] != 0, 0.0, gamma * acc)
        want[k] = acc
    assert np.allclose(retn, want, rtol=1e-12, atol=1e-12)
    paths = col.paths(pol)
    for p in paths[:20]:
        r = p["rewards"]
        dc = np.array([np.sum(r[i:] * gamma ** np.arange(len(r) - i)) for i in range(len(r))])
        assert np.allclose(retn[p["start"]:p["start"] + len(r), p["env"]], dc, rtol=1e-10, atol=1e-10)
    coeffs = col.fit_baseline(ret).cpu().numpy()
    adv, val = (x.cpu().numpy() for x in col.advantages(gamma, lam))
    feats, rets = [], []
    for p in paths:
        o = np.clip(p["observations"], -10, 10); ln = len(p["rewards"])
        al = ((start0[p["env"]] if p["start"] == 0 else 0) + np.arange(ln)).reshape(-1, 1) / 100.0
        feats.append(np.concatenate([o, o ** 2, al, al ** 2, al ** 3, np.ones((ln, 1))], axis=1))
        rets.append(retn[p["start"]:p["start"] + ln, p["env"]])
    F = np.concatenate(feats); y = np.concatenate(rets)
    assert F.shape == (n * T, 94)
    FtF, Fty = col.baseline_moments
    assert np.allclose(FtF, F.T @ F, rtol=1e-10, atol=1e-10) and np.allclose(Fty, F.T @ y, rtol=1e-10, atol=1e-10)
    for f, p in zip(feats, paths):
        e, a, ln = p["env"], p["start"], len(p["rewards"])
        v = f @ coeffs
        vb = np.append(v, 0.0)
        deltas = p["rewards"] + gamma * vb[1:] - vb[:-1]
        want_adv = np.array([np.sum(deltas[i:] * (gamma * lam) ** np.arange(ln - i)) for i in range(ln)])
        assert np.allclose(val[a:a + ln, e], v, rtol=1e-8, atol=1e-8)
        assert np.allclose(adv[a:a + ln, e], want_adv, rtol=1e-7, atol=1e-7)
    col.close()


# ------------------------------------------------------------------ 7. argument validation
def test_rollout_rejects_bad_arguments(R):
    from cassierl_b200 import lib
    col = R.RolloutCollector3d(4, precision=32)
    pol = R.GaussianMLPPolicy(45, 10)
    col.collect(pol, 2)
    b = col.batch
    L = b.L
    p = pol.flat
    bufs = [col.obs.data_ptr(), col.act.data_ptr(), col.mean.data_ptr(), col.rew.data_ptr(), col.done.data_ptr()]

    def call(mode=lib.MODE3D_PD, params=p.data_ptr(), n_params=p.numel(), n_sub=10, mpl=100, bufs=bufs):
        return L.Cassie3dBatchRollout(b.h, mode, params, n_params, 2, n_sub, mpl, 1, 1, 0, *bufs, None)

    def err():
        return L.Cassie3dGetLastError().decode()

    assert call() == 0
    torch.cuda.synchronize()
    assert call(params=None) == -1 and "null" in err()
    assert call(bufs=bufs[:3] + [None] + bufs[4:]) == -1 and "null" in err()
    assert call(mode=7) == -1 and "mode" in err()
    assert call(n_sub=0) == -1 and "n_substeps" in err()
    assert call(mpl=0) == -1 and "max_path_length" in err()
    assert call(mpl=-3) == -1 and "max_path_length" in err()
    assert call(n_params=2867) == -1 and "2868" in err() and "2867" in err()
    assert L.Cassie3dBatchRollout(None, 1, p.data_ptr(), 2868, 2, 10, 100, 1, 1, 0, *bufs, None) == -1 and "null" in err()
    col.close()
