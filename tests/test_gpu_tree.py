"""GPU parity of the 3-D tree engine (BASELINE.json configs[3]: cassie3d_stiff.xml) through the C-ABI of
include/cassie3d.h, against the fp64 oracle on the same initial states and torque sequences.  Every lane width of the
step kernel (8, 16, 32 lanes per env) is checked.  Error metric as in tests/test_tree_host.py."""
import numpy as np
import pytest

from conftest import TORQUE_HIGH_3D, lying3d, pose3d

pytestmark = pytest.mark.gpu


def _starts(n, seed=0):
    """standing poses just above the floor with perturbed joints, headings and small velocities"""
    rng = np.random.default_rng(seed)
    q = np.tile(pose3d(0.945), (n, 1))
    q[:, 7:] += rng.normal(size=(n, 14)) * 0.03
    yaw = rng.uniform(-np.pi, np.pi, n)
    roll = rng.normal(size=n) * 0.05
    for e in range(n):
        a = np.array([np.cos(yaw[e] / 2), 0, 0, np.sin(yaw[e] / 2)]); b = np.array([np.cos(roll[e] / 2), np.sin(roll[e] / 2), 0, 0])
        q[e, 3:7] = [a[0] * b[0], a[0] * b[1], a[3] * b[1], a[3] * b[0]]   # quaternion product yaw * roll
        q[e, 3:7] /= np.linalg.norm(q[e, 3:7])
    q[:, 0:2] = rng.normal(size=(n, 2)) * 3.0
    v = rng.normal(size=(n, 20)) * 0.05
    return q, v


def _err(q, v, qo, vo):
    return np.maximum(np.abs(q - qo).max(axis=1), np.abs(v - vo).max(axis=1) / np.maximum(1.0, np.abs(vo).max(axis=1)))


@pytest.mark.parametrize("lanes", [8, 16, 32])
def test_tree_fp64_rollout_vs_oracle(oracle, omodel3d, lanes):
    """16 envs x 200 free-running steps, random torques held 10 steps (configs[3] actions): 1e-9 in the fp64 build"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatch
    n, steps, hold = 16, 200, 10
    q0, v0 = _starts(n)
    rng = np.random.default_rng(1)
    A = rng.uniform(-1, 1, (n, steps // hold, 10)) * TORQUE_HIGH_3D
    b = Cassie3dBatch(n, precision=64, lanes=lanes)
    assert (b.nq, b.nv, b.nu) == (21, 20, 10)
    b.set_state(q0, v0)
    for k in range(steps // hold):
        b.step(torch.tensor(A[:, k]), n=hold)
    q, v = (x.cpu().numpy() for x in b.state())
    st = b.stats().cpu().numpy()
    b.close()
    _, qo, vo, _ = oracle.rollout_tree(omodel3d, q0, v0, steps, actions=A, hold=hold)
    e = _err(q, v, qo, vo)
    assert e.max() < 1e-9, e
    assert st[:, 0].max() >= 9 and st[:, 3].sum() == 0      # rows of the LAST step: connects + at least one floor contact somewhere


def test_tree_fp64_fall_and_autoreset_bit_exact(oracle, omodel3d):
    """robots pushed over: done flags (pelvis below 0.5 m) and the number of auto-resets are bit-exact against the
    oracle's rollout with the same rule, final states agree to 1e-8 (resets included)"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatch
    n, steps, hold = 24, 1200, 10
    q0, v0 = _starts(n, seed=3)
    v0[:, 3:6] += np.random.default_rng(4).normal(size=(n, 3)) * 1.5      # tumbling
    b = Cassie3dBatch(n, precision=64)
    rq, rv = b.reset_state()
    b.set_state(q0, v0)
    dones = np.zeros(n, np.int64)
    for k in range(steps // hold):
        d = b.step(None, n=hold, z_done=0.5, auto_reset=True)
        dones += (d.cpu().numpy() != 0)
    q, v = (x.cpu().numpy() for x in b.state())
    resets = b.resets().cpu().numpy()
    b.close()
    _, qo, vo, ro = oracle.rollout_tree(omodel3d, q0, v0, steps, actions=None, hold=hold, z_done=0.5, reset_qpos=rq, reset_qvel=rv)
    assert (resets == ro).all() and (dones == ro).all()
    assert ro.sum() >= n // 2            # unactuated robots collapse: most envs fell at least once
    assert _err(q, v, qo, vo).max() < 1e-8


@pytest.mark.parametrize("lanes", [8, 16, 32])
def test_tree_fp32_single_step_vs_oracle(oracle, omodel3d, lanes):
    """fp32 build, teacher-forced: every step starts from the oracle's state and warm start.  1e-5 on the steps whose
    constraint-row count equals the oracle's; event mismatches (a contact within fp32 rounding of touching) are rare"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatch
    n, steps = 32, 120
    q0, v0 = _starts(n, seed=5)
    rng = np.random.default_rng(6)
    A = rng.uniform(-1, 1, (n, steps // 10, 10)) * TORQUE_HIGH_3D
    datas = [oracle.Data(omodel3d) for _ in range(n)]
    for e in range(n):
        datas[e].set_state(q0[e], v0[e])
    b = Cassie3dBatch(n, precision=32, lanes=lanes)
    errs, same = [], []
    for k in range(steps):
        qs = np.stack([d.state()[0] for d in datas]); vs = np.stack([d.state()[1] for d in datas])
        ws = np.stack([d.warmstart() for d in datas])
        b.set_state(qs, vs); b.set_warm_start(ws)
        b.step(torch.tensor(A[:, k // 10]), n=1)
        q, v = (x.cpu().numpy().astype(np.float64) for x in b.state())
        rows = b.stats().cpu().numpy()[:, 0]
        for e in range(n):
            datas[e].step(A[e, k // 10])
        qo = np.stack([d.state()[0] for d in datas]); vo = np.stack([d.state()[1] for d in datas])
        ro = np.array([d.efc()["J"].shape[0] for d in datas])
        errs.append(_err(q, v, qo, vo)); same.append(rows == ro)
    b.close()
    errs, same = np.array(errs), np.array(same)
    ok = errs[same]
    assert np.median(ok) < 2e-6 and np.quantile(ok, 0.99) < 1e-5, (np.median(ok), np.quantile(ok, 0.99))
    assert ok.max() < 1e-4, ok.max()
    assert (~same).mean() < 0.02, (~same).mean()


def test_tree_config4_shard_invariants():
    """one GPU's shard of configs[3] (65536 envs over 8 GPUs = 8192 per GPU), fp32, random torques, auto-reset on fall:
    states stay finite, quaternions unit, resets happen, no contact is dropped for capacity in the common case"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatch, TORQUE_HIGH_3D as HI
    n = 8192
    b = Cassie3dBatch(n, precision=32)
    g = torch.Generator(device="cuda").manual_seed(0)
    hi = torch.tensor(HI, dtype=torch.float32, device="cuda")
    fell = torch.zeros(n, dtype=torch.int64, device="cuda")
    for k in range(130):        # 1300 simulator steps: under random torques nearly every robot has fallen once by then
        a = (torch.rand((n, 10), generator=g, device="cuda") * 2 - 1) * hi
        d = b.step(a, n=10, z_done=0.5, auto_reset=True)
        fell += (d != 0)
    q, v = b.state()
    st = b.stats()
    assert torch.isfinite(q).all() and torch.isfinite(v).all()
    assert (q[:, 3:7].norm(dim=1) - 1).abs().max() < 1e-5
    assert (q[:, 2] > 0.3).all()                       # nobody is left lying on the floor
    assert fell.sum() > n // 4 and (b.resets() == fell.to(torch.int32)).all()
    assert (d != 2).all()                              # no env went non-finite
    assert (st[:, 3] > 0).float().mean().item() < 0.05  # envs that ever dropped a contact for capacity are rare
    b.close()


def test_tree_step_host_matches_device():
    import torch
    from cassierl_b200.envs3d import Cassie3dBatch, TORQUE_HIGH_3D as HI
    n = 64
    a = (torch.rand((n, 10)) * 2 - 1) * torch.tensor(HI, dtype=torch.float32)
    b1, b2 = Cassie3dBatch(n), Cassie3dBatch(n)
    b1.step(a.cuda(), n=10)
    q1, v1 = b1.state()
    ah = a.pin_memory(); qh = torch.empty((n, 21)).pin_memory(); vh = torch.empty((n, 20)).pin_memory()
    dh = torch.empty(n, dtype=torch.uint8).pin_memory()
    b2.step_host(ah, qh, vh, dh, n=10)
    assert torch.equal(q1.cpu(), qh) and torch.equal(v1.cpu(), vh)
    b1.close(); b2.close()


def test_tree_nan_guard_and_masked_reset():
    """a non-finite env is reported done = 2 and restarts from the reset state in the same launch (it never poisons its
    neighbours); ResetAll with a mask touches the flagged envs only"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatch
    n = 96
    b = Cassie3dBatch(n, precision=32)
    rq, rv = b.reset_state()
    q, v = b.state()
    q[5, 9] = float("nan"); v[40, 3] = float("inf")
    b.set_state(q, v)
    d = b.step(None, n=10, z_done=0.5, auto_reset=True).cpu().numpy()
    assert d[5] == 2 and d[40] == 2 and (np.delete(d, [5, 40]) == 0).all()
    q2, v2 = b.state()
    assert torch.isfinite(q2).all() and torch.isfinite(v2).all()
    assert np.abs(q2[5].cpu().numpy() - rq).max() < 1e-6 and np.abs(v2[40].cpu().numpy() - rv).max() < 1e-6
    assert (b.resets().cpu().numpy()[[5, 40]] == 1).all() and b.resets().sum().item() == 2
    # neighbours of the bad envs moved like everybody else (all envs started from the same pose)
    assert (q2[6] - q2[7]).abs().max().item() < 1e-6
    # masked reset
    b.step(None, n=50)
    before = b.state()[0].clone()
    mask = torch.zeros(n, dtype=torch.uint8); mask[::3] = 1
    b.reset(mask)
    after = b.state()[0]
    assert torch.equal(after[1::3], before[1::3]) and torch.equal(after[2::3], before[2::3])
    assert np.abs(after[::3].cpu().numpy() - rq.astype(np.float32)).max() < 1e-6
    b.close()


def test_tree_big_ragged_batch_subset_vs_oracle(oracle, omodel3d):
    """configs[3]-sized shard with a ragged tail (8192 + 3 envs: the last CTA has idle tiles), every env in its own state:
    one fp32 step, 22 envs scattered over the grid (first / last CTA, CTA boundaries) checked against the oracle"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatch
    n = 8192 + 3
    q0, v0 = _starts(n, seed=11)
    rng = np.random.default_rng(12)
    A = rng.uniform(-1, 1, (n, 10)) * TORQUE_HIGH_3D
    b = Cassie3dBatch(n, precision=32)
    b.set_state(q0, v0)
    b.step(torch.tensor(A), n=1)
    q, v = (x.cpu().numpy().astype(np.float64) for x in b.state())
    rows = b.stats().cpu().numpy()[:, 0]
    b.close()
    idx = np.unique(np.concatenate([[0, 1, 6, 7, 8, 13, 14, 15], rng.integers(16, n - 16, 8), [n - 8, n - 7, n - 4, n - 3, n - 2, n - 1]]))
    assert np.isfinite(q).all() and np.isfinite(v).all()
    errs = []
    for e in idx:
        d = oracle.Data(omodel3d)
        d.set_state(q0[e], v0[e])
        d.step(A[e])
        qo, vo = d.state()
        assert rows[e] == d.efc()["J"].shape[0], e            # same constraint rows (these starts are not within rounding of touching)
        errs.append(max(np.abs(q[e] - qo).max(), np.abs(v[e] - vo).max() / max(1.0, np.abs(vo).max())))
    errs = np.array(errs)
    # an indexing mistake would be O(1); the fp32 level of a cold first step on penetrating toes is a few 1e-5 at worst
    # (the same envs give the same errors on the CPU harness), 1e-6 typically
    assert np.median(errs) < 1e-5 and errs.max() < 1e-4, errs


@pytest.mark.parametrize("lanes", [8, 32])
def test_tree_two_pass_overflow_vs_oracle(oracle, omodel3d, lanes):
    """envs that need more than the fast capacity (32 rows / 9 contacts) mid-launch are finished by the full-capacity pass:
    robots pressed into the floor (33 and 36 rows at the first step) between standing ones, fp64, 30 free-running steps in
    three launches against the oracle (which has room for everything): 1e-8, nothing dropped"""
    import torch
    from cassierl_b200.envs3d import Cassie3dBatch
    n, steps, hold = 13, 30, 10
    q0, v0 = _starts(n, seed=21)
    for e, q in ((2, lying3d(0.10, "x", 1.5708)), (3, lying3d(0.14, "y", -1.5708, straight=True)), (7, lying3d(0.12, "x", 1.5708, straight=True)),
                 (12, lying3d(0.06, "y", 1.5708))):
        q0[e] = q; v0[e] = 0
    rng = np.random.default_rng(22)
    A = rng.uniform(-1, 1, (n, steps // hold, 10)) * TORQUE_HIGH_3D
    b = Cassie3dBatch(n, precision=64, lanes=lanes)
    b.set_state(q0, v0)
    rows_first = None
    for k in range(steps // hold):
        b.step(torch.tensor(A[:, k]), n=hold)
    q, v = (x.cpu().numpy() for x in b.state())
    st = b.stats().cpu().numpy()
    b.close()
    d = oracle.Data(omodel3d); d.set_state(q0[3], v0[3]); d.forward()
    assert d.efc()["J"].shape[0] > 32                      # the scenario does exceed the fast capacity
    _, qo, vo, _ = oracle.rollout_tree(omodel3d, q0, v0, steps, actions=A, hold=hold)
    assert st[:, 3].sum() == 0
    assert _err(q, v, qo, vo).max() < 1e-8, _err(q, v, qo, vo)
