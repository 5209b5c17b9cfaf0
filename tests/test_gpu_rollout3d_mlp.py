"""The 3-D fused rollout with rllab's hidden_sizes (Cassie3dBatchRolloutMlp, RolloutCollector3d with
GaussianMLPPolicy(hidden_sizes=...)) on the GPU: the means against the PyTorch reference and the noise against numpy at
every shape, lane width and action mode; lane-width and sharding invariance; Cassie3dBatchRollout as RolloutMlp at
(32, 32); the transitions against Cassie3dBatchEnv.step; the launch knobs (one worker process per setting,
tests/rollout3d_mlp_variants_worker.py); argument validation, and the planar collector's refusal of other shapes."""
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
sid = lambda s: "x".join(map(str, s))


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


# ------------------------------------------------------------------ 1. forward and noise at every shape
@pytest.mark.parametrize("lanes", [8, 16, 32])
@pytest.mark.parametrize("mode", ["PD", "Torque"])
def test_means_and_noise_every_shape(R, mode, lanes):
    """for each shape: the means within 1e-5 relative of GaussianMLPPolicy.mean on the recorded observations, and the
    noise equal to the shape-independent normal10 of (seed, global env, step)"""
    n, T = 37, 3
    for shape in SHAPES:
        col = R.RolloutCollector3d(n, control_mode=mode, precision=32, seed=777, first_global_env=200, lanes=lanes)
        pol = R.GaussianMLPPolicy(col.obs_dim, col.act_dim, seed=3, hidden_sizes=shape)
        out = col.collect(pol, T)
        obs, act, mean = out["observations"], out["actions"], out["means"]
        assert torch.isfinite(obs).all() and torch.isfinite(act).all(), shape
        ref = pol.mean(obs.reshape(-1, col.obs_dim)).reshape(T, n, col.act_dim)
        rel = float((mean - ref).abs().max() / ref.abs().max().clamp(min=1))
        assert rel < 1e-5, (shape, rel)
        eps = ((act - mean) / pol.log_std.exp()).cpu().numpy().astype(np.float64)
        for (k, e) in ((0, 0), (0, 36), (1, 17), (2, 5)):
            want = normal10(777, 200 + e, k)
            assert np.allclose(eps[k, e], want, atol=2e-5 * max(1.0, np.abs(want).max())), (shape, k, e)
        col.close()


# ------------------------------------------------------------------ 2. lane width
def test_means_bit_identical_across_lanes(R):
    """(128, 128): the same observations give bit-identical means at 8, 16 and 32 lanes (no cross-lane reduction)"""
    n = 45
    q0, v0 = start_state(n, 1)
    runs = []
    for lanes in (8, 16, 32):
        col = R.RolloutCollector3d(n, control_mode="PD", precision=32, seed=5, lanes=lanes)
        col.batch.set_state(q0, v0)
        pol = R.GaussianMLPPolicy(col.obs_dim, col.act_dim, seed=6, hidden_sizes=(128, 128))
        runs.append({k: v.clone() for k, v in col.collect(pol, 1).items()})
        col.close()
    for r in runs[1:]:
        assert torch.equal(r["observations"], runs[0]["observations"])
        assert torch.equal(r["means"], runs[0]["means"])
        assert torch.equal(r["actions"], runs[0]["actions"])


# ------------------------------------------------------------------ 3. the fixed-shape entry point
@pytest.mark.parametrize("precision", [32, 64])
def test_rollout_is_rollout_mlp_at_default_shape(R, precision):
    """Cassie3dBatchRollout and RolloutMlp with (32, 32) give bit-identical path buffers and final states"""
    n, T = 53, 8
    q0, v0 = start_state(n, 2)
    res = []
    for fixed in (False, True):
        col = R.RolloutCollector3d(n, control_mode="PD", precision=precision, max_path_length=5, seed=31, first_global_env=9)
        col.batch.set_state(q0, v0)
        pol = R.GaussianMLPPolicy(col.obs_dim, col.act_dim, seed=2, dtype=col.batch.dtype)
        if fixed:
            col._buffers(T)
            b = col.batch
            with torch.cuda.device(b.device):
                col._check(b.L.Cassie3dBatchRollout(
                    b.h, col.mode, pol.flat.data_ptr(), pol.flat.numel(), T, col.n_substeps, col.max_path_length, 1, col.seed,
                    col.env0, col.obs.data_ptr(), col.act.data_ptr(), col.mean.data_ptr(), col.rew.data_ptr(),
                    col.done.data_ptr(), None), "Rollout")
            out = dict(observations=col.obs, actions=col.act, means=col.mean, rewards=col.rew, dones=col.done)
        else:
            out = col.collect(pol, T)
        q, v = col.batch.state()
        res.append({k: x.clone() for k, x in dict(out, q=q, v=v).items()})
        col.close()
    assert res[0]["dones"].any()
    for k in res[0]:
        assert torch.equal(res[0][k], res[1][k]), k


# ------------------------------------------------------------------ 4. sharding invariance
def test_sharding_invariance_wide(R):
    """(128, 128): 32 envs at global ids 1037.. reproduce that slice of a 101-env run bit for bit"""
    T = 6
    pol = R.GaussianMLPPolicy(45, 10, seed=3, hidden_sizes=(128, 128))
    col = R.RolloutCollector3d(101, control_mode="PD", precision=32, seed=12345, first_global_env=1000)
    out = {k: v.clone() for k, v in col.collect(pol, T).items()}
    col2 = R.RolloutCollector3d(32, control_mode="PD", precision=32, seed=12345, first_global_env=1037)
    out2 = col2.collect(pol, T)
    for k in ("observations", "actions", "means", "rewards", "dones"):
        assert torch.equal(out2[k], out[k][:, 37:69]), k
    col.close(); col2.close()


# ------------------------------------------------------------------ 5. transitions equal EnvStep
def test_wide_transitions_match_env_step(R):
    """fp64, (128, 128): replaying the recorded actions through Cassie3dBatchEnv(auto_reset, max_path_length=12) gives
    bit-identical observations, rewards and done codes, with falls, time limits and steps finished by the continuation
    pass"""
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    n, T, mpl = 24, 30, 12
    rng = np.random.default_rng(4)
    q0 = np.tile(pose3d(0.945), (n, 1)); q0[:, 7:] += rng.normal(size=(n, 14)) * 0.03
    v0 = rng.normal(size=(n, 20)) * 0.05
    for e in range(0, n, 3):
        q0[e, 2] = 0.62; q0[e, 3:7] = [np.cos(0.6), 0.0, np.sin(0.6), 0.0]
    for e in (1, 11, n - 1):
        q0[e] = lying3d(0.10); v0[e] = 0
    col = R.RolloutCollector3d(n, control_mode="PD", precision=64, max_path_length=mpl, seed=7, first_global_env=3)
    col.batch.set_state(q0, v0)
    pol = R.GaussianMLPPolicy(col.obs_dim, col.act_dim, seed=5, dtype=torch.float64, hidden_sizes=(128, 128))
    first = {k: v.clone() for k, v in col.collect(pol, 1).items()}
    assert int((col.batch.stats()[:, 0] > 32).sum()) >= 1     # the continuation pass finished this step
    rest = col.collect(pol, T - 1)
    out = {k: torch.cat([first[k], rest[k]]) for k in first}
    env = Cassie3dBatchEnv(n, control_mode="PD", precision=64, auto_reset=True, max_path_length=mpl)
    env.batch.set_state(q0, v0)
    o = env.observe().clone()
    lo, hi = (torch.tensor(x, dtype=torch.float64, device=o.device) for x in col.action_space)
    for k in range(T):
        assert torch.equal(out["observations"][k], o), k
        a = (lo + (out["actions"][k] + 1.0) * 0.5 * (hi - lo)).clamp(lo, hi)
        o, r, d = env.step(a, n=10)
        o = o.clone()
        assert torch.equal(out["rewards"][k], r), k
        assert torch.equal(out["dones"][k], path_codes(d)), k
    codes = set(np.unique(out["dones"].cpu().numpy()).tolist())
    assert {1, 2} <= codes, codes
    col.close(); env.terminate()


# ------------------------------------------------------------------ 6. launch knobs
SETTINGS = {"default": {}, "tiles7": {"CASSIE3D_TILES": "7"}, "one_pass": {"CASSIE3D_TWO_PASS": "0"}}


@pytest.fixture(scope="module")
def mlp_variant_runs(tmp_path_factory):
    d = tmp_path_factory.mktemp("rollout3d_mlp_variants")
    worker = os.path.join(ROOT, "tests", "rollout3d_mlp_variants_worker.py")
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


def test_tiles_knob_is_bit_identical(mlp_variant_runs):
    base, run = mlp_variant_runs["default"], mlp_variant_runs["tiles7"]
    assert sorted(base) == sorted(run)
    bad = [k for k in base if not np.array_equal(base[k], run[k], equal_nan=True)]
    assert not bad, bad


def test_single_pass_is_bit_identical(mlp_variant_runs):
    """CASSIE3D_TWO_PASS=0: every fp64 array and every integer array bit-identical.  fp32 physics differs between the
    fast and the full-capacity compile of the step (test_gpu_tree_variants.py), so fp32 reals are not compared."""
    base, run = mlp_variant_runs["default"], mlp_variant_runs["one_pass"]
    assert base["p64_l32_dones"].any()
    bad = [k for k in base if (k.startswith("p64_") or k.endswith(("_dones", "_resets")))
           and not np.array_equal(base[k], run[k], equal_nan=True)]
    assert not bad, bad


# ------------------------------------------------------------------ 7. argument validation
def test_rollout_mlp_rejects_bad_arguments(R):
    from cassierl_b200 import lib
    ct = lib.ct
    col = R.RolloutCollector3d(4, precision=32)
    pol = R.GaussianMLPPolicy(45, 10, hidden_sizes=(64, 48))
    col.collect(pol, 2)
    b = col.batch
    L = b.L
    p = pol.flat
    bufs = [col.obs.data_ptr(), col.act.data_ptr(), col.mean.data_ptr(), col.rew.data_ptr(), col.done.data_ptr()]
    arr = lambda *s: (ct.c_int32 * max(len(s), 1))(*s)

    def call(sizes=(64, 48), n_hidden=None, sizes_ptr=None, mode=lib.MODE3D_PD, params=p.data_ptr(), n_params=p.numel(),
             n_sub=10, mpl=100, h=b.h, bufs=bufs):
        ptr = arr(*sizes) if sizes_ptr is None else sizes_ptr
        return L.Cassie3dBatchRolloutMlp(h, mode, len(sizes) if n_hidden is None else n_hidden, ptr, params, n_params, 2,
                                         n_sub, mpl, 1, 1, 0, *bufs, None)

    def err():
        return L.Cassie3dGetLastError().decode()

    assert call() == 0
    torch.cuda.synchronize()
    assert call(sizes_ptr=ct.cast(None, ct.POINTER(ct.c_int32))) == -1 and "null" in err()
    assert call(h=None) == -1 and "null" in err()
    assert call(params=None) == -1 and "null" in err()
    assert call(bufs=bufs[:2] + [None] + bufs[3:]) == -1 and "null" in err()
    assert call(mode=5) == -1 and "mode" in err()
    assert call(n_sub=0) == -1 and "n_substeps" in err()
    assert call(mpl=0) == -1 and "max_path_length" in err()
    assert call(sizes=(), n_hidden=0) == -1 and "n_hidden" in err()
    assert call(sizes=(8, 8, 8, 8, 8)) == -1 and "n_hidden" in err() and "1 to 4" in err()
    assert call(sizes=(64, 0)) == -1 and "hidden_sizes[1]" in err()
    assert call(sizes=(257, 48)) == -1 and "hidden_sizes[0]" in err() and "256" in err()
    assert call(sizes=(64, -3)) == -1 and "hidden_sizes[1]" in err()
    assert call(n_params=p.numel() + 1) == -1 and str(p.numel()) in err() and str(p.numel() + 1) in err()
    assert call(sizes=(48, 64)) == -1 and str(R.n_params(45, 10, (48, 64))) in err()
    # the fixed-shape entry point refuses a wider policy's vector with the (32, 32) count in the message
    assert L.Cassie3dBatchRollout(b.h, 1, p.data_ptr(), p.numel(), 2, 10, 100, 1, 1, 0, *bufs, None) == -1
    assert "2868" in err() and str(p.numel()) in err()
    col.close()


def test_planar_collector_refuses_wide_policy(R):
    """the planar rollout stays (32, 32): its parameter-count check refuses a (128, 128) policy"""
    col = R.RolloutCollector(4)
    pol = R.GaussianMLPPolicy(col.obs_dim, col.act_dim, hidden_sizes=(128, 128))
    with pytest.raises(RuntimeError, match="expected %d" % R.n_params(col.obs_dim, col.act_dim)):
        col.collect(pol, 1)
    col.close()
