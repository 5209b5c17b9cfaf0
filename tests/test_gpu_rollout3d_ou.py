"""DDPG's sampler on the 3-D fused rollout (Cassie3dBatchRolloutOU, RolloutCollector3d with DeterministicMLPPolicy and
OUStrategy) on the GPU: the means against the PyTorch reference at every shape, lane width and action mode; the OU
recurrence and its reset at path starts against numpy; evaluation rollouts and the clip; the transitions against
Cassie3dBatchEnv.step; sharding invariance over a ragged batch; the launch knobs (one worker process per setting,
tests/rollout3d_ou_variants_worker.py); transitions() and ReplayPool on the device; argument validation and the
collectors' refusals."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT, lying3d, pose3d
from test_gpu_rollout3d import KNOBS, normal10, path_codes

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

SHAPES = [(32, 32), (64, 64), (128, 128), (256, 256), (100, 50, 25), (256,), (8, 8, 8, 8)]


@pytest.fixture(scope="module")
def R():
    if not torch.cuda.is_available():
        pytest.fail("-m gpu tests need a CUDA device")
    from cassierl_b200 import rollout
    return rollout


def start_state(n, seed):
    """standing envs with perturbed joints, every fourth tipped low (it falls within the run)"""
    rng = np.random.default_rng(seed)
    q = np.tile(pose3d(0.945), (n, 1)); q[:, 7:] += rng.normal(size=(n, 14)) * 0.05
    v = rng.normal(size=(n, 20)) * 0.05
    for e in range(0, n, 4):
        q[e, 2] = 0.62; q[e, 3:7] = [np.cos(0.6), 0.0, np.sin(0.6), 0.0]
    return q, v


def scaled_policy(R, col, shape, seed, scale=30.0):
    """a DeterministicMLPPolicy whose output layer is scaled up from rllab's U(+-3e-3), so that the tanh head matters"""
    pol = R.DeterministicMLPPolicy(col.obs_dim, col.act_dim, seed=seed, dtype=col.batch.dtype, hidden_sizes=shape)
    p = pol.unpack()
    p[-2].mul_(scale); p[-1].mul_(scale)
    return pol


# ------------------------------------------------------------------ 1. forward at every shape
@pytest.mark.parametrize("lanes", [8, 16, 32])
@pytest.mark.parametrize("mode", ["PD", "Torque"])
def test_means_every_shape(R, mode, lanes):
    """for each shape: the means within 1e-5 relative (fp32) and 1e-12 (fp64) of DeterministicMLPPolicy.mean on the
    recorded observations"""
    n, T = 37, 3
    for prec, tol in ((32, 1e-5), (64, 1e-12)):
        for shape in SHAPES:
            col = R.RolloutCollector3d(n, control_mode=mode, precision=prec, seed=777, first_global_env=200, lanes=lanes)
            pol = scaled_policy(R, col, shape, 3)
            out = col.collect(pol, T, R.OUStrategy())
            obs, act, mean = out["observations"], out["actions"], out["means"]
            assert torch.isfinite(obs).all() and torch.isfinite(act).all(), shape
            ref = pol.mean(obs.reshape(-1, col.obs_dim)).reshape(T, n, col.act_dim)
            rel = float((mean - ref).abs().max() / ref.abs().max().clamp(min=1))
            assert rel < tol, (prec, shape, rel)
            col.close()


def test_means_bit_identical_across_lanes(R):
    """(128, 128): the same observations give bit-identical means, actions and OU steps at 8, 16 and 32 lanes"""
    n = 45
    q0, v0 = start_state(n, 1)
    runs = []
    for lanes in (8, 16, 32):
        col = R.RolloutCollector3d(n, control_mode="PD", precision=32, seed=5, lanes=lanes)
        col.batch.set_state(q0, v0)
        pol = scaled_policy(R, col, (128, 128), 6)
        runs.append({k: v.clone() for k, v in col.collect(pol, 1, R.OUStrategy(mu=0.1)).items()})
        col.close()
    for r in runs[1:]:
        for k in ("observations", "means", "actions"):
            assert torch.equal(r[k], runs[0][k]), k


# ------------------------------------------------------------------ 2. the OU recurrence
def test_ou_recurrence_and_resets(R):
    """sigma small enough that nothing clips, mu != 0: act - mean follows the numpy recurrence driven by normal10 of
    (seed, global env, step), with x = mu at every path start (time limits of 5 and falls), across two collects"""
    n, T1, T2, mpl = 24, 9, 8, 5
    mu, theta, sigma, seed, env0 = 0.2, 0.15, 0.05, 4242, 17
    q0, v0 = start_state(n, 3)
    for e in (1, 11, n - 1):                                           # on the floor: done 1 at the first step
        q0[e] = lying3d(0.10); v0[e] = 0
    col = R.RolloutCollector3d(n, control_mode="PD", precision=64, max_path_length=mpl, seed=seed, first_global_env=env0)
    col.batch.set_state(q0, v0)
    pol = scaled_policy(R, col, (32, 32), 2, scale=0.01)               # means near 0: mean + x never reaches the clip
    es = R.OUStrategy(mu, theta, sigma)
    a = {k: v.clone() for k, v in col.collect(pol, T1, es).items()}
    b = col.collect(pol, T2, es)
    out = {k: torch.cat([a[k], b[k]]) for k in a}
    x = (out["actions"] - out["means"]).cpu().numpy()
    done = out["dones"].cpu().numpy()
    assert float(out["actions"].abs().max()) < 0.9                     # no clip: act - mean is the OU state
    assert (done == 1).any() and (done == 2).any()
    want = np.zeros(10)
    starts = 0
    for e in range(n):
        for k in range(T1 + T2):
            start = k == 0 or done[k - 1, e] != 0
            starts += start
            prev = np.full(10, mu) if start else want
            want = prev + theta * (mu - prev) + sigma * normal10(seed, env0 + e, k)
            # the kernel's normals are fp32 with fast intrinsics: a few 1e-6 relative, summed over the state's memory
            assert np.abs(x[k, e] - want).max() < 1e-3 * sigma, (e, k)
            if start:
                assert np.abs(x[k, e] - (mu + sigma * normal10(seed, env0 + e, k))).max() < 1e-3 * sigma
    assert starts > 2 * n
    col.close()


# ------------------------------------------------------------------ 3. evaluation rollouts and the clip
def test_zero_noise_is_the_deterministic_action_and_clip(R):
    """sigma = 0, mu = 0: actions equal the means bit for bit; sigma = 3: every action in [-1, 1], some clipped"""
    for prec in (32, 64):
        col = R.RolloutCollector3d(64, control_mode="PD", precision=prec, max_path_length=6, seed=1)
        pol = scaled_policy(R, col, (64, 64), 4)
        out = col.collect(pol, 10, R.OUStrategy(mu=0.0, theta=0.15, sigma=0.0))
        assert torch.equal(out["actions"], out["means"]) and float(out["means"].abs().max()) > 0.01
        col.close()
        col = R.RolloutCollector3d(64, control_mode="Torque", precision=prec, seed=1)
        out = col.collect(pol, 10, R.OUStrategy(sigma=3.0))
        act = out["actions"]
        assert float(act.abs().max()) <= 1.0
        assert int((act == 1.0).sum()) > 0 and int((act == -1.0).sum()) > 0
        assert int((act.abs() < 1.0).sum()) > 0
        col.close()


# ------------------------------------------------------------------ 4. transitions equal EnvStep
@pytest.mark.parametrize("mode", ["PD", "Torque"])
def test_transitions_match_env_step(R, mode):
    """fp64: replaying the recorded (clipped exploratory) actions through Cassie3dBatchEnv(auto_reset,
    max_path_length=12) reproduces observations and rewards within 1e-9 and the done codes exactly, with falls, time
    limits and steps finished by the continuation pass"""
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
    pol = scaled_policy(R, col, (64, 64), 5)
    es = R.OUStrategy(sigma=0.5)
    first = {k: v.clone() for k, v in col.collect(pol, 1, es).items()}
    assert int((col.batch.stats()[:, 0] > 32).sum()) >= 1     # the continuation pass finished this step
    rest = col.collect(pol, T - 1, es)
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
    assert float((col.last_obs - o).abs().max()) < 1e-9               # the observation after the last step
    assert err_o < 1e-9 and err_r < 1e-9, (err_o, err_r)
    codes = set(np.unique(out["dones"].cpu().numpy()).tolist())
    assert {1, 2} <= codes, codes
    col.close(); env.terminate()


# ------------------------------------------------------------------ 5. sharding invariance
@pytest.mark.parametrize("mode", ["PD", "Torque"])
def test_sharding_invariance(R, mode):
    """64 envs at global ids 1037.. reproduce envs 37..100 of a 101-env run bit for bit over two collects: the slice
    starts off a CTA boundary and holds the ragged batch's last env, whose mirrored tiles must not advance its OU
    state"""
    pol_shape, T = (128, 128), 6
    es = R.OUStrategy(mu=0.05, sigma=0.3)
    col = R.RolloutCollector3d(101, control_mode=mode, precision=32, seed=12345, first_global_env=1000)
    col2 = R.RolloutCollector3d(64, control_mode=mode, precision=32, seed=12345, first_global_env=1037)
    pol = scaled_policy(R, col, pol_shape, 3)
    for _ in range(2):
        out = {k: v.clone() for k, v in col.collect(pol, T, es).items()}
        out2 = col2.collect(pol, T, es)
        for k in ("observations", "actions", "means", "rewards", "dones"):
            assert torch.equal(out2[k], out[k][:, 37:]), k
        assert torch.equal(col2.last_obs, col.last_obs[37:])
    col.close(); col2.close()


# ------------------------------------------------------------------ 6. launch knobs
SETTINGS = {"default": {}, "tiles7": {"CASSIE3D_TILES": "7"}, "one_pass": {"CASSIE3D_TWO_PASS": "0"}}


@pytest.fixture(scope="module")
def ou_variant_runs(tmp_path_factory):
    d = tmp_path_factory.mktemp("rollout3d_ou_variants")
    worker = os.path.join(ROOT, "tests", "rollout3d_ou_variants_worker.py")
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


def test_tiles_knob_is_bit_identical(ou_variant_runs):
    base, run = ou_variant_runs["default"], ou_variant_runs["tiles7"]
    assert sorted(base) == sorted(run)
    bad = [k for k in base if not np.array_equal(base[k], run[k], equal_nan=True)]
    assert not bad, bad


def test_single_pass_is_bit_identical(ou_variant_runs):
    """CASSIE3D_TWO_PASS=0: every fp64 array and every integer array bit-identical (fp32 physics differs between the
    fast and the full-capacity compile of the step)"""
    base, run = ou_variant_runs["default"], ou_variant_runs["one_pass"]
    assert base["p64_l32_c0_dones"].any()
    bad = [k for k in base if (k.startswith("p64_") or k.endswith(("_dones", "_resets")))
           and not np.array_equal(base[k], run[k], equal_nan=True)]
    assert not bad, bad


# ------------------------------------------------------------------ 7. transitions() and ReplayPool on the device
@pytest.mark.parametrize("include", [False, True])
def test_transitions_and_pool_on_device(R, include):
    n, T, mpl = 40, 12, 5
    col = R.RolloutCollector3d(n, control_mode="PD", precision=32, max_path_length=mpl, seed=3)
    q0, v0 = start_state(n, 7)
    col.batch.set_state(q0, v0)
    pol = scaled_policy(R, col, (32, 32), 1)
    es = R.OUStrategy()
    pool = R.ReplayPool(3 * n * T // 2, col.obs_dim, col.act_dim, device=pol.flat.device, dtype=col.batch.dtype)
    added = 0
    for c in range(3):
        out = col.collect(pol, T, es)
        tr = col.transitions(include_horizon_terminal_transitions=include)
        assert all(v.device == col.obs.device for v in tr.values())
        done = out["dones"]
        n_cut = int((done == 2).sum())
        assert n_cut > 0
        assert tr["rewards"].shape[0] == n * T - (0 if include else n_cut)
        assert int(tr["terminals"].sum()) == int((done == 1).sum()) + (n_cut if include else 0)
        # row by row: next observation of a row that is not done is the same env's next observation
        keep = (torch.ones_like(done, dtype=torch.bool) if include else done != 2).cpu()
        pos = torch.cumsum(keep.reshape(-1).long(), 0).reshape(T, n) - 1
        o, a, lo = out["observations"].cpu(), out["actions"].cpu(), col.last_obs.cpu()
        tro, tra, trn = tr["observations"].cpu(), tr["actions"].cpu(), tr["next_observations"].cpu()
        for k in range(T):
            for e in range(n):
                if not keep[k, e]:
                    continue
                i = int(pos[k, e])
                assert torch.equal(tro[i], o[k, e]) and torch.equal(tra[i], a[k, e])
                assert torch.equal(trn[i], o[k + 1, e] if k + 1 < T else lo[e]), (k, e)
        last = col.last_obs.clone()
        pool.add(tr)
        added += tr["rewards"].shape[0]
        assert pool.size == min(added, pool.max_pool_size)
        nxt = col.collect(pol, 1, es)                                   # the last observation is the next start
        assert float((nxt["observations"][0] - last).abs().max()) < 1e-5
    assert added > pool.max_pool_size                                   # the ring wrapped
    g = torch.Generator(device=col.obs.device).manual_seed(11)
    batch = pool.random_batch(256, generator=g)
    assert batch["observations"].shape == (256, col.obs_dim) and batch["observations"].device == col.obs.device
    col.close()


# ------------------------------------------------------------------ 8. argument validation and refusals
def test_rollout_ou_rejects_bad_arguments(R):
    from cassierl_b200 import lib
    ct = lib.ct
    col = R.RolloutCollector3d(4, precision=32)
    pol = R.DeterministicMLPPolicy(45, 10, hidden_sizes=(64, 48))
    col.collect(pol, 2, R.OUStrategy())
    b = col.batch
    L = b.L
    p = pol.flat
    bufs = [col.obs.data_ptr(), col.act.data_ptr(), col.mean.data_ptr(), col.rew.data_ptr(), col.done.data_ptr()]
    arr = lambda *s: (ct.c_int32 * max(len(s), 1))(*s)

    def call(sizes=(64, 48), n_hidden=None, sizes_ptr=None, mode=lib.MODE3D_PD, params=p.data_ptr(), n_params=p.numel(),
             mu=0.0, theta=0.15, sigma=0.3, n_sub=10, mpl=100, steps=2, h=b.h, bufs=bufs):
        ptr = arr(*sizes) if sizes_ptr is None else sizes_ptr
        return L.Cassie3dBatchRolloutOU(h, mode, len(sizes) if n_hidden is None else n_hidden, ptr, params, n_params, mu, theta,
                                        sigma, steps, n_sub, mpl, 1, 1, 0, *bufs, None)

    def err():
        return L.Cassie3dGetLastError().decode()

    assert call() == 0
    torch.cuda.synchronize()
    assert call(sizes_ptr=ct.cast(None, ct.POINTER(ct.c_int32))) == -1 and "null" in err()
    assert call(h=None) == -1 and "null" in err()
    assert call(params=None) == -1 and "null" in err()
    for i in range(5):
        assert call(bufs=bufs[:i] + [None] + bufs[i + 1:]) == -1 and "null" in err()
    assert call(mode=5) == -1 and "mode" in err()
    assert call(steps=-1) == -1 and "n_policy_steps" in err()
    assert call(n_sub=0) == -1 and "n_substeps" in err()
    assert call(mpl=0) == -1 and "max_path_length" in err()
    assert call(sizes=(), n_hidden=0) == -1 and "n_hidden" in err()
    assert call(sizes=(8, 8, 8, 8, 8)) == -1 and "n_hidden" in err() and "1 to 4" in err()
    assert call(sizes=(64, 0)) == -1 and "hidden_sizes[1]" in err()
    assert call(sizes=(257, 48)) == -1 and "hidden_sizes[0]" in err() and "256" in err()
    want = R.n_params(45, 10, (64, 48), log_std=False)
    assert call(n_params=want + 1) == -1 and str(want) in err() and str(want + 1) in err()
    gauss = R.GaussianMLPPolicy(45, 10, hidden_sizes=(64, 48)).flat       # a Gaussian vector: log_std included
    assert call(params=gauss.data_ptr(), n_params=gauss.numel()) == -1 and "log_std" in err() and str(want) in err()
    for bad in (dict(mu=float("nan")), dict(theta=float("inf")), dict(sigma=float("-inf")), dict(sigma=float("nan"))):
        assert call(**bad) == -1 and "finite" in err(), bad
    assert call(sigma=-0.1) == -1 and "sigma" in err() and "negative" in err()
    assert call(sigma=0.0, theta=-2.0, mu=-5.0) == 0                  # sigma 0 and any finite mu / theta are valid
    torch.cuda.synchronize()
    col.close()


def test_collector_refusals(R):
    """Gaussian with es, deterministic without es, a deterministic policy on the planar collector"""
    col = R.RolloutCollector3d(4, precision=32)
    with pytest.raises(ValueError, match="es must be None"):
        col.collect(R.GaussianMLPPolicy(45, 10), 1, R.OUStrategy())
    with pytest.raises(ValueError, match="OUStrategy"):
        col.collect(R.DeterministicMLPPolicy(45, 10), 1)
    with pytest.raises(RuntimeError, match="DeterministicMLPPolicy"):
        col.collect(R.GaussianMLPPolicy(45, 10), 1)
        col.transitions()
    out = col.collect(R.DeterministicMLPPolicy(45, 10), 1, R.OUStrategy())
    paths = col.paths(R.DeterministicMLPPolicy(45, 10))
    assert sum(len(p["rewards"]) for p in paths) == 4 and all(p["agent_infos"] == {} for p in paths)
    assert out["actions"].shape == (1, 4, 10)
    col.close()
    planar = R.RolloutCollector(4)
    with pytest.raises(TypeError, match="GaussianMLPPolicy"):
        planar.collect(R.DeterministicMLPPolicy(planar.obs_dim, planar.act_dim), 1)
    planar.close()
