"""Worker of tests/test_gpu_rollout3d.py: collects one seeded 3-D rollout for precision 32 and 64 at lanes 8, 16 and 32
and saves every path buffer and the final state to an .npz file.

The launch knobs of the tree kernels (CASSIE3D_TWO_PASS, CASSIE3D_STEP_BARRIER, CASSIE3D_TILES) are read once per
process, so the test starts this worker once per setting and compares the files.

    python tests/rollout3d_variants_worker.py OUT.npz
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.dirname(HERE), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from conftest import lying3d, pose3d  # noqa: E402

N, T = 101, 6                                    # prime: the last CTA has idle tiles at every tile count
LYING = (0, 23, 24, 55, 56, N - 1)               # more rows than the fast capacity: finished by the continuation pass
LOW = (5, 33, 77)                                # rolled below the fall height: terminated and reset inside the run


def scenario(seed=0):
    rng = np.random.default_rng(seed)
    q = np.tile(pose3d(0.945), (N, 1))
    q[:, 7:] += rng.normal(size=(N, 14)) * 0.03
    v = rng.normal(size=(N, 20)) * 0.05
    for e in LOW:
        q[e, 2] = 0.6; q[e, 3:7] = [np.cos(0.6), np.sin(0.6), 0.0, 0.0]
    for i, e in enumerate(LYING):
        q[e] = lying3d(0.10 + 0.02 * (i % 2), "xy"[i % 2], 1.5708); v[e] = 0
    return q, v


def run(prec, lanes, out):
    import torch
    from cassierl_b200.rollout import GaussianMLPPolicy, RolloutCollector3d
    q0, v0 = scenario()
    col = RolloutCollector3d(N, control_mode="PD", precision=prec, max_path_length=4, seed=99, first_global_env=5, lanes=lanes)
    col.batch.set_state(q0, v0)
    pol = GaussianMLPPolicy(col.obs_dim, col.act_dim, seed=8, dtype=col.batch.dtype)
    res = col.collect(pol, T)
    q, v = col.batch.state()
    torch.cuda.synchronize()
    pre = "p%d_l%d_" % (prec, lanes)
    for k, x in dict(res, q=q, v=v, resets=col.batch.resets()).items():
        out[pre + k] = x.cpu().numpy().copy()
    col.close()


if __name__ == "__main__":
    out = {}
    for prec in (32, 64):
        for lanes in (8, 16, 32):
            run(prec, lanes, out)
    np.savez(sys.argv[1], **out)
