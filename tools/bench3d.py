#!/usr/bin/env python
"""BASELINE.json configs[3]: cassie3d_stiff.xml, 65536 envs sharded over 8 GPUs (8192 per GPU), uniform-random torques
on the ten motors held 10 simulator steps, done when the pelvis drops below 0.5 m, auto-reset.  Prints ONE JSON line in
bench.py's format (value, e2e, roofline, cpu_baseline, clocks).  Not the headline bench (that is bench.py, configs[2]).

  python tools/bench3d.py [--envs 8192] [--steps 20] [--warmup 3] [--lanes 32]       (under torchrun for N > 1 GPUs)

--workload env_torque: the same torques through Cassie3dBatchEnvStep (observation, reward, done, time limit 1000 policy
steps: what the stand env's epilogue costs); env_pd: uniform-random PD targets within the joint ranges, auto-reset,
max_path_length 1000.  Device-timed and end-to-end (EnvStepHost: obs / reward / done to the host) env-steps/s.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402  (ClockSampler, peaks)

p = argparse.ArgumentParser()
p.add_argument("--envs", type=int, default=8192, help="envs per GPU (65536 / 8)")
p.add_argument("--steps", type=int, default=20)
p.add_argument("--warmup", type=int, default=3)
p.add_argument("--substeps", type=int, default=10)
p.add_argument("--lanes", type=int, default=0)
p.add_argument("--precision", type=int, default=32)
p.add_argument("--preadvance", type=int, default=2000, help="simulator steps before timing: robots fall after ~1000 steps of random torques and reset, by 2000 the batch is a mix of phases")
p.add_argument("--no-cpu-baseline", action="store_true")
p.add_argument("--cpu-seconds", type=float, default=10.0)
p.add_argument("--workload", choices=["torque", "env_torque", "env_pd"], default="torque")
a = p.parse_args()

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402
from cassierl_b200 import lib  # noqa: E402
from cassierl_b200.envs3d import PD_HIGH_3D, PD_LOW_3D, TORQUE_HIGH_3D, Cassie3dBatch, Cassie3dBatchEnv  # noqa: E402

world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local)
dev = torch.device("cuda", local)
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
L = lib.load()
n, sub = a.envs, a.substeps
dt_t = torch.float64 if a.precision == 64 else torch.float32
rs = 8 if a.precision == 64 else 4
ENV = a.workload != "torque"
MPL = 1000


def make():
    if ENV:
        return Cassie3dBatchEnv(n, device=local, control_mode="PD" if a.workload == "env_pd" else "Torque", precision=a.precision,
                                max_path_length=MPL, lanes=a.lanes or None)
    return Cassie3dBatch(n, device=local, precision=a.precision, lanes=a.lanes or None)


e3 = make()
b = e3.batch if ENV else e3
n_pre = (a.preadvance + sub - 1) // sub
total = n_pre + a.warmup + a.steps
gen = torch.Generator(device=dev).manual_seed(1 + rank)
hi = torch.tensor(TORQUE_HIGH_3D, dtype=dt_t, device=dev)
acts = (torch.rand((total, n, 10), generator=gen, device=dev, dtype=dt_t) * 2 - 1) * hi     # resident in HBM before timing
if a.workload == "env_pd":    # uniform within the joint ranges
    lo = torch.tensor(PD_LOW_3D, dtype=dt_t, device=dev); span = torch.tensor(PD_HIGH_3D, dtype=dt_t, device=dev) - lo
    acts = lo + torch.rand((total, n, 10), generator=gen, device=dev, dtype=dt_t) * span
done = torch.empty(n, dtype=torch.uint8, device=dev)


def step(h, act):
    if ENV:
        h.step(act, n=sub)
    else:
        h.step(act, n=sub, z_done=0.5, auto_reset=True, done=done)
flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)


def barrier():
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()


for k in range(n_pre + a.warmup):
    step(e3, acts[k])
barrier()
sampler = bench.ClockSampler(local, "GPU-" + str(torch.cuda.get_device_properties(dev).uuid))
if rank == 0:
    sampler.start()
ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
l0 = L.CassieKernelLaunchCount()
resets0 = b.resets().sum().item()
barrier()
for k in range(a.steps):
    flush.zero_()
    ev[k][0].record()
    step(e3, acts[n_pre + a.warmup + k])
    ev[k][1].record()
barrier()
launches = L.CassieKernelLaunchCount() - l0
ms = sum(x.elapsed_time(y) for x, y in ev)
clocks = sampler.stop() if rank == 0 else None
t = torch.tensor([ms], dtype=torch.float64, device=dev)
if world > 1:
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
ms_max = float(t.item())
value = world * n * sub * a.steps / (ms_max * 1e-3)
st = b.stats().double()
q, v = b.state()
stats = torch.stack([st[:, 0].mean(), st[:, 1].mean(), st[:, 2].mean(), st[:, 3].sum(), torch.tensor(float(b.resets().sum().item() - resets0), device=dev, dtype=torch.float64),
                     (~torch.isfinite(q).all(dim=1)).double().sum()])
if world > 1:
    red = stats.clone(); dist.all_reduce(red); stats[3:] = red[3:]

# end to end: pinned host actions in, qpos / qvel / done out (env workloads: obs / reward / done), copies inside the
# timed region
b2 = make()
for k in range(n_pre):
    step(b2, acts[k])
acts_h = acts[n_pre:].cpu().pin_memory()
qh = torch.empty((n, 21), dtype=dt_t).pin_memory(); vh = torch.empty((n, 20), dtype=dt_t).pin_memory()
dh = torch.empty(n, dtype=torch.uint8).pin_memory()
oh = torch.empty((n, 45), dtype=dt_t).pin_memory(); rh = torch.empty(n, dtype=dt_t).pin_memory()


def step_host(act_h):
    if ENV:
        b2.step_host(act_h, oh, rh, dh, n=sub)
    else:
        b2.step_host(act_h, qh, vh, dh, n=sub, z_done=0.5, auto_reset=True)


for k in range(a.warmup):
    step_host(acts_h[k])
barrier()
t0 = time.perf_counter()
for k in range(a.steps):
    step_host(acts_h[a.warmup + k])
torch.cuda.synchronize()
el = torch.tensor([time.perf_counter() - t0], dtype=torch.float64, device=dev)
if world > 1:
    dist.all_reduce(el, op=dist.ReduceOp.MAX)
e2e = world * n * sub * a.steps / float(el.item())

if rank == 0:
    # algorithmic FLOPs of one step: the engine on an operation-counting scalar (tests/host_harness th_count_ops) along this
    # workload's stream is ~1.9e5 at 18 rows / 50 sweeps; measured per run below when the harness is available
    flops = None
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from conftest import TreeHarness, pose3d
        th = TreeHarness(os.path.join(ROOT, "tests", "_build", "libtree_harness.so"), os.path.join(ROOT, "cassierl_b200", "model", "cassie3d_stiff.xml"))
        qq, vv, ww = pose3d(0.94), np.zeros(20), np.zeros(20)
        cnt = []
        for k in range(150):
            if k >= 50:
                cnt.append(int(th.count_ops(qq, vv, ww, np.zeros(10))[:3].sum()))
            th.step(qq, vv, ww, np.zeros(10))
        flops = float(np.mean(cnt))
    except Exception:
        flops = 1.9e5
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    fp32_peak = L.CassieMeasureFp32Peak(local)
    ms_launch = ms_max / a.steps
    achieved = flops * n * sub / (ms_launch * 1e-3) / 1e12
    bytes_launch = n * ((21 + 20 + 20) * 2 * rs + 10 * rs + 1 + 16)
    line = {"metric": "env-steps/sec cassie3d_stiff, random torques, auto-reset on fall", "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms_launch, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if a.precision == 32 else "f64", "data": "synthetic",
            "config": {"workload": "cassie3d_stiff.xml, uniform-random torques held %d sim steps, done at pelvis z < 0.5 m, auto-reset (BASELINE configs[3])" % sub,
                       "envs_per_gpu": n, "envs_total": n * world, "sim_steps_per_launch": sub, "lanes_per_env": a.lanes or int(os.environ.get("CASSIE3D_LANES", "32")),
                       "preadvance_sim_steps": n_pre * sub, "l2": "flushed between timed steps (256 MiB memset)",
                       "parallelism": "env-sharded dp%d, no data-path collective" % world},
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s", "frac": achieved / fp32_peak if fp32_peak else None,
                         "traffic": None, "flops_per_env_step": flops,
                         "flops_source": "tree engine instantiated on an operation-counting scalar (th_count_ops), standing robot, 12-18 rows, PGS at its sweep count",
                         "peak_source": "measured live: register-only FFMA kernel (CassieMeasureFp32Peak)",
                         "hbm": {"achieved_gbs": bytes_launch / (ms_launch * 1e-3) / 1e9, "peak_gbs": peaks.get("hbm_gbs", 6650.0), "algorithmic_bytes_per_launch": bytes_launch}},
            "e2e": {"value": e2e, "unit": "env-steps/s", "h2d_bytes_per_step": n * 10 * rs, "d2h_bytes_per_step": n * (41 * rs + 1)},
            "gpu_launches": int(launches), "clocks": clocks,
            "stats": {"rows_mean": float(stats[0]), "contacts_mean": float(stats[1]), "pgs_sweeps_mean": float(stats[2]), "contacts_dropped": int(stats[3]),
                      "auto_resets_in_timed_region": int(stats[4]), "non_finite_envs": int(stats[5]), "smem_bytes_per_env": b.smem_per_env}}
    if ENV:
        line["metric"] = "env-steps/sec cassie3d_stiff stand env (%s), EnvStep with observation, reward, auto-reset" % a.workload
        line["config"]["workload"] = ("%s actions held %d sim steps through Cassie3dBatchEnvStep: 45-d observation, stand reward, done at "
                                      "pelvis z < 0.5 m or after %d policy steps, auto-reset" %
                                      ("uniform-random torques" if a.workload == "env_torque" else "uniform-random PD targets within the joint ranges", sub, MPL))
        line["config"]["bench_workload"] = a.workload
        line["e2e"]["d2h_bytes_per_step"] = n * (46 * rs + 1)
    if not a.no_cpu_baseline and world == 1:
        from oracle import oracle as O
        O.build()
        m = O.Model(O.model3d_path())
        cores = os.cpu_count() or 1
        ne = cores * 4
        rng = np.random.default_rng(1)
        q0 = np.tile(b.reset_state()[0], (ne, 1)); v0 = np.zeros((ne, 20))
        rq, rv = b.reset_state()
        t0 = time.perf_counter(); O.rollout_tree(m, q0, v0, 50, actions=rng.uniform(-1, 1, (ne, 5, 10)) * TORQUE_HIGH_3D, hold=10, n_threads=cores)
        rate = ne * 50 / (time.perf_counter() - t0)
        ns = int(max(100, min(20000, rate * a.cpu_seconds / ne))) // 10 * 10
        A = rng.uniform(-1, 1, (ne, ns // 10, 10)) * TORQUE_HIGH_3D
        t0 = time.perf_counter()
        tot, _, _, rr = O.rollout_tree(m, q0, v0, ns, actions=A, hold=10, z_done=0.5, reset_qpos=rq, reset_qvel=rv, n_threads=cores)
        dtc = time.perf_counter() - t0
        line["cpu_baseline"] = {"value": tot / dtc, "unit": "env-steps/s", "cores": cores, "kind": "port",
                                "sample": "%d envs x %d sim steps of the same workload (resets %d), fp64 oracle (oracle/, gcc -O3 -fopenmp), %.1f s" % (ne, ns, int(rr.sum()), dtc)}
    print(json.dumps(line), flush=True)
if world > 1:
    dist.barrier()
    dist.destroy_process_group()
