"""Worker of tests/test_gpu_rollout3d_ou.py: the seeded scenario of rollout3d_variants_worker.py collected with a
DeterministicMLPPolicy(hidden_sizes=(100, 50, 25)) and an OUStrategy, two collects in a row (the OU state carries over),
for precision 32 and 64 at lanes 8, 16 and 32; saves every path buffer, the last observation and the final state to an
.npz file.  The launch knobs are read once per process, so the test starts one worker per setting.

    python tests/rollout3d_ou_variants_worker.py OUT.npz
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
for _p in (os.path.dirname(HERE), HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from rollout3d_variants_worker import N, T, scenario  # noqa: E402

HIDDEN = (100, 50, 25)


def run(prec, lanes, out):
    import torch
    from cassierl_b200.rollout import DeterministicMLPPolicy, OUStrategy, RolloutCollector3d
    q0, v0 = scenario()
    col = RolloutCollector3d(N, control_mode="PD", precision=prec, max_path_length=4, seed=99, first_global_env=5, lanes=lanes)
    col.batch.set_state(q0, v0)
    pol = DeterministicMLPPolicy(col.obs_dim, col.act_dim, seed=8, dtype=col.batch.dtype, hidden_sizes=HIDDEN)
    es = OUStrategy(mu=0.1, theta=0.15, sigma=0.3)
    pre = "p%d_l%d_" % (prec, lanes)
    for c in range(2):
        res = col.collect(pol, T, es)
        for k, x in dict(res, last_obs=col.last_obs).items():
            out[pre + "c%d_" % c + k] = x.cpu().numpy().copy()
    q, v = col.batch.state()
    torch.cuda.synchronize()
    for k, x in dict(q=q, v=v, resets=col.batch.resets()).items():
        out[pre + k] = x.cpu().numpy().copy()
    col.close()


if __name__ == "__main__":
    out = {}
    for prec in (32, 64):
        for lanes in (8, 16, 32):
            run(prec, lanes, out)
    np.savez(sys.argv[1], **out)
