"""BASELINE.json configs[4] (TRPO rollout collection): fused policy MLP + noise + env step kernel, then the
sampler-side pre-processing (returns, LinearFeatureBaseline fit, GAE advantages) on device.  Not the headline
bench (bench.py); prints one JSON line for profiles/.

  python tools/bench_rollout.py [--envs N] [--T T] [--mode PD|OSC|TORQUE]
  python tools/bench_rollout.py --model 3d [--envs N] [--T T] [--mode PD|TORQUE] [--hidden 128,128]   # the 3-D stand env
  python tools/bench_rollout.py --model 3d --policy ou      # DDPG's sampler: DeterministicMLPPolicy + OUStrategy
  python -m torch.distributed.run --nproc-per-node G ... tools/bench_rollout.py     # N envs PER GPU, one rank per GPU

--model 3d (RolloutCollector3d, default 8192 envs per GPU, T = 20, PD; --hidden the policy's hidden_sizes, default
32,32) also sweeps hidden_sizes (32, 32) (64, 64) (128, 128) (256, 256): at each shape it times, in the same process and
alternated twice, the fused collect, the loop a user would otherwise write on Cassie3dBatchEnv (PyTorch policy forward,
randn, affine map, clamp, EnvStep) and EnvStep alone on pre-generated actions (an upper bound for the fused collect).  It
reports the rollout and env kernels' launch resources read from a torch.profiler trace, with the card's name and power
limit.  The sweep spans the reference launchers' (32, 32) and (128, 128) up to the widest shape the kernel takes, whose
fp32 weights (318 KB) no longer fit in L1.

--policy ou (3-D only) adds DDPG's fused collect (DeterministicMLPPolicy + OUStrategy, Cassie3dBatchRolloutOU) to that
alternation, at the reference launchers' (32, 32) and (128, 128) only, and times the sampler side of DDPG instead of
returns + baseline + GAE: transitions() + ReplayPool.add + random_batch(256).

Multi-GPU (SURVEY 8e): envs are sharded by global env id (Philox streams and phases do not depend on G), there is no
collective inside a rollout; after it, NCCL all-reduces the rollout statistics (cassierl_b200.parallel.RolloutStats) and
all-gathers the sample paths for a single learner (parallel.gather_paths) on a side stream, overlapped with the next
rollout.  Times are CUDA-event times, max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from cassierl_b200 import parallel  # noqa: E402
from cassierl_b200.rollout import (DeterministicMLPPolicy, GaussianMLPPolicy, OUStrategy, ReplayPool, RolloutCollector,  # noqa: E402
                                   RolloutCollector3d)

p = argparse.ArgumentParser()
p.add_argument("--model", default="2d", choices=["2d", "3d"], help="planar (cassie2d) or 3-D (cassie3d stand env)")
p.add_argument("--envs", type=int, default=None, help="envs per GPU (default 16384 planar, 8192 3-D)")
p.add_argument("--T", type=int, default=20, help="policy steps per collect() (10 sim steps each)")
p.add_argument("--reps", type=int, default=5)
p.add_argument("--mode", default="PD", choices=["PD", "OSC", "TORQUE"])
p.add_argument("--task", default="stand", choices=["stand", "imitate"])
p.add_argument("--hidden", default="32,32", help="the policy's hidden_sizes, comma-separated (the planar rollout: 32,32)")
p.add_argument("--policy", default="gaussian", choices=["gaussian", "ou"],
               help="gaussian: GaussianMLPPolicy (TRPO / VPG); ou: DeterministicMLPPolicy + OUStrategy (DDPG), 3-D only")
a = p.parse_args()
hidden = tuple(int(h) for h in a.hidden.split(","))
if a.model == "2d" and hidden != (32, 32):
    p.error("the planar rollout takes hidden_sizes (32, 32) only")
if a.envs is None:
    a.envs = 8192 if a.model == "3d" else 16384
if a.model == "3d" and a.mode == "OSC":
    p.error("the 3-D env offers PD and TORQUE")
if a.model == "2d" and a.policy == "ou":
    p.error("the planar rollout takes a GaussianMLPPolicy only")
ou = a.policy == "ou"

world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
n_total = a.envs * world

if a.model == "3d":
    col = RolloutCollector3d(a.envs, device=local, control_mode={"PD": "PD", "TORQUE": "Torque"}[a.mode], max_path_length=1000,
                             first_global_env=rank * a.envs)
else:
    col = RolloutCollector(a.envs, device=local, task=a.task, control_mode=a.mode, max_path_length=1000, first_global_env=rank * a.envs)
pol = (DeterministicMLPPolicy if ou else GaussianMLPPolicy)(col.obs_dim, col.act_dim, device=dev, hidden_sizes=hidden)
es = OUStrategy() if ou else None
if world > 1:
    dist.broadcast(pol.flat, src=0)            # the learner's parameters (8.5 kB), once per iteration
pool = ReplayPool(1000000, col.obs_dim, col.act_dim, device=dev) if ou else None   # rllab DDPG's default pool size


def sampler_side():
    """what the sampler does with a collect: DDPG's pool rows, or TRPO's returns, baseline and advantages"""
    if ou:
        pool.add(col.transitions())
        pool.random_batch(256)
    else:
        r = col.discounted_returns()
        col.fit_baseline(r); col.advantages()


col.collect(pol, a.T, es)                  # warm-up (also sizes the buffers)
sampler_side()
torch.cuda.synchronize()


def maxr(x):
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ms = []
    for _ in range(reps):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return maxr(sorted(ms)[len(ms) // 2])


def card():
    """name, power limit and max SM clock of this rank's GPU (nvidia-smi query; read in the measuring process)"""
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return {"name": torch.cuda.get_device_name(dev), "nvidia_smi": q or "unavailable"}


def kernel_resources(fns, names):
    """launch resources of the kernels whose name contains one of `names`, from a torch.profiler trace of fns (the
    trace goes to a temporary directory)"""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for fn in fns:
            fn()
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as td:
        path = os.path.join(td, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f)["traceEvents"]
    out = {}
    for ev in events:
        if ev.get("cat") != "kernel":
            continue
        for nm in names:
            if nm + "<" in ev["name"] or ev["name"].startswith(nm):
                ar = ev.get("args", {})
                key = ev["name"].split("(")[0].replace("void ", "").replace("cassie::tree::", "")
                out.setdefault(key, {k: ar.get(k) for k in ("registers per thread", "shared memory", "block", "grid",
                                                             "blocks per SM", "warps per SM", "est. achieved occupancy %")})
    return out


SWEEP_3D = ((32, 32), (128, 128)) if ou else ((32, 32), (64, 64), (128, 128), (256, 256))


def compare_3d():
    """at each shape of SWEEP_3D: (a) the fused collect, (b) the unfused loop on Cassie3dBatchEnv, (c) EnvStep alone on
    pre-generated actions, with --policy ou (d) the fused OU collect; same envs and T, alternated twice, CUDA-event times
    (median of --reps each)"""
    from cassierl_b200.envs3d import Cassie3dBatchEnv
    env = Cassie3dBatchEnv(a.envs, device=local, control_mode=col.control_mode, auto_reset=True, max_path_length=1000)
    env.reset()
    n, T = a.envs, a.T
    lo, hi = (torch.tensor(x, dtype=env.batch.dtype, device=dev) for x in col.action_space)
    mk = lambda *sh, dt=env.batch.dtype: torch.empty(sh, dtype=dt, device=dev)
    bo, ba, bm, br, bd = mk(T, n, 45), mk(T, n, 10), mk(T, n, 10), mk(T, n), mk(T, n, dt=torch.uint8)
    state = {"obs": env.observe().clone()}
    pre = (lo + (torch.rand(T, n, 10, device=dev, dtype=env.batch.dtype)) * (hi - lo)).contiguous()

    def env_only():
        for k in range(T):
            env.step(pre[k])

    sweep, res = {}, None
    for shape in SWEEP_3D:
        sp = GaussianMLPPolicy(col.obs_dim, col.act_dim, device=dev, hidden_sizes=shape)
        layers = sp.unpack()
        std = layers[-1].exp()

        def unfused():
            o = state["obs"]
            for k in range(T):
                h = o
                for i in range(0, len(layers) - 3, 2):
                    h = torch.tanh(h @ layers[i] + layers[i + 1])
                mean = h @ layers[-3] + layers[-2]
                act = mean + std * torch.randn_like(mean)
                x = (lo + (act + 1.0) * 0.5 * (hi - lo)).clamp(lo, hi)
                bo[k].copy_(o); ba[k].copy_(act); bm[k].copy_(mean)
                o, r, d = env.step(x)
                br[k].copy_(r); bd[k].copy_(d)
            state["obs"] = o

        dp = DeterministicMLPPolicy(col.obs_dim, col.act_dim, device=dev, hidden_sizes=shape) if ou else None
        col.collect(sp, T); unfused(); env_only()      # warm-up of every shape
        if ou:
            col.collect(dp, T, es)
        torch.cuda.synchronize()
        runs = {"fused_collect": [], "unfused_loop": [], "env_step_only": []}
        if ou:
            runs["fused_ou_collect"] = []
        for _ in range(2):
            runs["fused_collect"].append(timed(lambda: col.collect(sp, T), a.reps))
            runs["unfused_loop"].append(timed(unfused, a.reps))
            runs["env_step_only"].append(timed(env_only, a.reps))
            if ou:
                runs["fused_ou_collect"].append(timed(lambda: col.collect(dp, T, es), a.reps))
        if res is None:
            res = kernel_resources([lambda: col.collect(sp, 2), lambda: env.step(pre[0])], ["k_tree_rollout_step", "k_tree_env_step"])
        best = {k: min(v) for k, v in runs.items()}
        sweep["x".join(map(str, shape))] = {
            "ms_per_collect": runs, "env_steps_per_s": {k: [n * T * 10 / (x * 1e-3) for x in v] for k, v in runs.items()},
            "fused_vs_env_step_only": best["fused_collect"] / best["env_step_only"] - 1.0,
            "fused_vs_unfused": best["fused_collect"] / best["unfused_loop"] - 1.0}
        if ou:
            sweep["x".join(map(str, shape))]["ou_vs_gaussian_collect"] = best["fused_ou_collect"] / best["fused_collect"] - 1.0
    env.terminate()
    return {"hidden_sizes_sweep": sweep, "kernels": res, "card": card()}


ms_collect = timed(lambda: col.collect(pol, a.T, es), a.reps)
cmp3d = compare_3d() if a.model == "3d" else None
col.collect(pol, a.T, es)                  # the buffers of the headline policy for the sampler side
torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(a.reps):
    sampler_side()
torch.cuda.synchronize()
ms_post = maxr((time.perf_counter() - t0) / a.reps * 1e3)

# ---- what a single learner needs from all ranks: statistics (all-reduce) and the sample paths (all-gather)
stats = parallel.RolloutStats(device=dev)
stats.update(col.rew, col.done, col.obs)
red = stats.reduce()
gather = {"world": world, "collective": "none (1 GPU)"}
if world > 1:
    fields = [col.obs, col.act, col.mean, col.rew, col.done]
    local_bytes = sum(x.numel() * x.element_size() for x in fields)

    def do_gather():
        return [parallel.gather_paths(x, n_total) for x in fields]

    g = do_gather()
    assert g[0].shape == (a.T, n_total, col.obs_dim)
    # rank r's shard sits at its global env ids
    assert torch.equal(g[3][:, rank * a.envs:(rank + 1) * a.envs], col.rew)
    ms_gather = timed(do_gather, a.reps)
    # overlapped: the gather of batch k runs on a side stream while batch k+1 is being collected
    side = torch.cuda.Stream(device=dev)
    snap = [x.clone() for x in fields]

    def overlapped():
        for i, x in enumerate(fields):
            snap[i].copy_(x)
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            out = [parallel.gather_paths(x, n_total) for x in snap]
        col.collect(pol, a.T)
        torch.cuda.current_stream().wait_stream(side)
        return out

    ms_overlap = timed(overlapped, a.reps)
    gather = {"world": world, "collective": "ncclAllGather (torch.distributed all_gather) of obs/act/mean/rew/done + ncclAllReduce of 6 statistics",
              "bytes_per_rank": local_bytes, "bytes_gathered_per_rank": local_bytes * world, "gather_ms": ms_gather,
              "gather_GBps_per_rank_in": local_bytes * (world - 1) / (ms_gather * 1e-3) / 1e9,
              "collect_plus_gather_serial_ms": ms_collect + ms_gather, "collect_with_overlapped_gather_ms": ms_overlap}

d = col.done
if a.model == "3d":
    st = col.batch.stats().double()   # [n, 4]: constraint rows, contacts, PGS sweeps, contacts dropped
    if rank == 0:
        print(json.dumps({
            "workload": "rollout: %s(45->%s->10) + %s action space + cassie3d stand env, %d envs per GPU x %d GPUs x %d policy steps x 10 sim steps"
                        % ("DeterministicMLPPolicy + OUStrategy" if ou else "GaussianMLPPolicy", "->".join(map(str, hidden)),
                           col.control_mode, a.envs, world, a.T),
            "n_gpus": world, "collect_ms": ms_collect, "env_steps_per_s": n_total * a.T * 10 / (ms_collect * 1e-3),
            "policy_steps_per_s": n_total * a.T / (ms_collect * 1e-3),
            "env_steps_per_s_with_overlapped_gather": (n_total * a.T * 10 / (gather["collect_with_overlapped_gather_ms"] * 1e-3)) if world > 1 else None,
            ("transitions_pool_add_random_batch256_ms" if ou else "returns_baseline_advantages_ms"): ms_post,
            "episodes_finished": int((d != 0).sum().item()),
            "rollout_stats_all_ranks": red, "gather": gather, "compare_rank0": cmp3d,
            "last_step_rows_mean": float(st[:, 0].mean().item()), "last_step_rows_max": int(st[:, 0].max().item())}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    sys.exit(0)
st = col.batch.stats().double()   # [n, 4]: rows, PGS sweeps, QP iterations, QP status of the last sim step
qp = {"iters_mean": float(st[:, 2].mean().item()), "iters_max": int(st[:, 2].max().item()),
      "iters_p99": float(torch.quantile(st[:, 2], 0.99).item()), "not_optimal": int((st[:, 3] != 0).sum().item()),
      "warp_max_mean": float(st[:, 2].reshape(-1, 32).max(dim=1).values.mean().item())}
if rank == 0:
    print(json.dumps({
        "workload": "rollout: GaussianMLPPolicy(%d->32->32->%d) + %s action space + cassie2d %s env, %d envs per GPU x %d GPUs x %d policy steps x 10 sim steps"
                    % (col.obs_dim, col.act_dim, a.mode, a.task, a.envs, world, a.T),
        "mlp": os.environ.get("CASSIE_MLP", "scalar"), "engine": os.environ.get("CASSIE_ENGINE", "default"),
        "n_gpus": world, "collect_ms": ms_collect, "env_steps_per_s": n_total * a.T * 10 / (ms_collect * 1e-3),
        "policy_steps_per_s": n_total * a.T / (ms_collect * 1e-3),
        "env_steps_per_s_with_overlapped_gather": (n_total * a.T * 10 / (gather["collect_with_overlapped_gather_ms"] * 1e-3)) if world > 1 else None,
        "returns_baseline_advantages_ms": ms_post, "episodes_finished": int((d != 0).sum().item()),
        "rollout_stats_all_ranks": red, "gather": gather,
        "last_step_rows_mean": float(st[:, 0].mean().item()), "last_step_qp": qp}), flush=True)
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
