#!/usr/bin/env python
"""Headline benchmark: env-steps/s of the batched cassie2d_stiff step path (BASELINE.json).

  python bench.py --gpus N --steps K --warmup W            # this framework (CUDA, libcassie2d.so)
  python bench.py --impl reference --gpus N ...            # the CPU restatement on the host cores
  python bench.py ... --dump-outputs DIR                   # + the last timed step's results as DIR/<name>.npy

A "step" is one launch of the fused step kernel: `--substeps` (default 10, the Python envs' n,
cassie2d.py:97) simulator steps of dt = 0.5 ms for every env of the batch, with the controller of
the workload in the loop.  env-step = one simulator step of one env = one legacy Step* call
(SURVEY 8d).  Weak scaling: every rank owns `--envs` envs (default 16384, BASELINE configs[2]);
envs are independent, so there is no collective on the data path -- NCCL only reduces the rollout
statistics after the timed region.

Timing: per-step CUDA events on the launching stream, L2 flushed between timed steps, barrier +
synchronize on both sides, MAX over ranks.  The JSON line carries `roofline` (FP32 pipe, measured
peak), `cpu_baseline` (oracle port on the host cores, bounded sample), `e2e` (host buffers through
the C-ABI *Host entry points, copies inside the timed region), `clocks`, `gpu_launches`.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

# Algorithmic FLOPs of ONE simulator step of ONE env (add+sub+mul+div+sqrt, FMA = 2), counted by
# instantiating the engine on an operation-counting scalar (tools/count_flops.py; DESIGN.md 5).
# Mean over the first 100 steps of the squatting stream at four phases (9.5-11 constraint rows, PGS at
# its 50-sweep cap); the fast path's inert padding rows are NOT counted.  torque_random / pd_env use
# the torque / PD step figures of the same stream (their own streams visit more contact states).
FLOPS_PER_STEP = {"squat_osc": 43.3e3, "squat_jacobian": 30.5e3, "torque_random": 24.1e3, "pd_env": 22.5e3}
# Algorithmic HBM bytes of one launch per env: qpos, qvel, warm start read + written (13 reals each),
# lagged op-space state 12 r/w, clock 8 r/w, stats 16 w, + per-workload action/phase/obs traffic.
STATE_BYTES_PER_ENV_F32 = 2 * (39 * 4 + 12 * 4 + 8) + 16

WORKLOADS = {
    "squat_jacobian": "cassie2d_stiff.xml, squatting.py loop with standing_controller_jacobian (StepJacobian) in the kernel",
    "squat_osc": "cassie2d_stiff.xml, squatting loop with standing_controller_osc + OSC_RBDL QP (StepOsc) in the kernel",
    "torque_random": "cassie2d_stiff.xml, uniform-random torques held 10 steps (StepTorque)",
    "pd_env": "cassie2d_stiff.xml, cassie_stand2d env step (StepPd x10 + obs/reward/done + auto-reset)",
}
DEFAULT_WORKLOAD = "squat_osc"   # BASELINE.json configs[2]: 16384 envs, OSC_RBDL squatting controller in the loop
METRIC = "env-steps/sec cassie2d_stiff @16k envs"   # the SAME string on both arms (the driver divides one by the other)
MODE_OF = {"squat_jacobian": 2, "squat_osc": 3, "torque_random": 0, "pd_env": 1}


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=50)
    p.add_argument("--warmup", type=int, default=5)
    p.add_argument("--impl", default="native", choices=["native", "reference"])
    p.add_argument("--envs", type=int, default=16384, help="envs per GPU")
    p.add_argument("--substeps", type=int, default=10)
    p.add_argument("--workload", default=DEFAULT_WORKLOAD, choices=sorted(WORKLOADS))
    p.add_argument("--precision", type=int, default=32, choices=[32, 64])
    p.add_argument("--no-cpu-baseline", action="store_true")
    p.add_argument("--cpu-seconds", type=float, default=10.0)
    p.add_argument("--preadvance", type=int, default=1000,
                   help="simulator steps every env is advanced OUTSIDE the timed region (steady state, not the start-up transient)")
    p.add_argument("--ref-envs", type=int, default=1024, help="--impl reference: envs of the bounded CPU sample")
    p.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                   help="weak: --envs per GPU (the driver's contract); strong: --envs in TOTAL, split evenly over the ranks")
    p.add_argument("--dump-outputs", metavar="DIR",
                   help="after the timed steps, write what the last timed step returned to its caller as DIR/<name>.npy "
                        "(rank r of several writes DIR/<name>_rank<r>.npy), for output-for-output comparison of two builds")
    return p.parse_args()


def kernel_source_hash():
    """sha256 over the CUDA sources of the step path: profiles/traffic.json entries carry the hash of the
    sources their ncu capture ran, and bench.py prints `roofline.traffic` only while it still matches."""
    import hashlib
    h = hashlib.sha256()
    d = os.path.join(ROOT, "cassierl_b200", "csrc")
    for f in sorted(os.listdir(d)):
        # the sources the planar step / squat kernels are compiled from (not the 3-D tree engine, the rollout kernels,
        # the host-side flattener or the C-ABI glue: edits there cannot change the captured kernel)
        if f.endswith((".cuh", ".cu", ".h")) and not f.startswith(("tree_", "cassie3d", "rollout_", "mjcf_flatten", "cassie2d_api")):
            h.update(f.encode()); h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:16]


# ----------------------------------------------------------------------------- CPU arm (oracle)
def oracle_rate(workload, n_envs, n_steps, threads, seed=1):
    """env-steps/s of the fp64 CPU restatement (oracle/, OpenMP over envs) on this box."""
    from oracle import oracle as O
    O.build()
    m = oracle_rate.model = getattr(oracle_rate, "model", None) or O.Model()
    phase = 2 * np.pi * np.arange(n_envs) / max(n_envs, 1)
    t0 = time.perf_counter()
    if workload == "squat_jacobian":
        n, _ = O.rollout(m, n_envs, n_steps, 2, phase=phase, n_threads=threads)
    elif workload == "squat_osc":
        n, _ = O.rollout(m, n_envs, n_steps, 3, phase=phase, n_threads=threads)
    else:
        rng = np.random.default_rng(seed)
        hi = np.array([12.0, 12.0, 0.9, 12.0, 12.0, 0.9])
        nact = (n_steps + 9) // 10
        if workload == "torque_random":
            a = rng.uniform(-1, 1, (n_envs, nact, 6)) * hi
            n, _ = O.rollout(m, n_envs, n_steps, 0, actions=a, hold=10, n_threads=threads)
        else:
            lo = np.radians([-50.0, -164.0, -140.0, -50.0, -164.0, -140.0]); hh = np.radians([80.0, -37.0, -30.0, 80.0, -37.0, -30.0])
            a = rng.uniform(lo, hh, (n_envs, nact, 6))
            n, _ = O.rollout(m, n_envs, n_steps, 1, actions=a, hold=10, n_threads=threads)
    dt = time.perf_counter() - t0
    return n / dt, dt


def cpu_baseline(workload, seconds, preadvance=1000):
    """The oracle port timed on this box's host cores: a bounded sample of the same workload, persistent envs
    pre-advanced like the native arm's (steady state), ~`seconds` of CPU work."""
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    rate, _ = oracle_rate(workload, cores, 50, cores)            # calibration
    n_envs = cores * 4
    mode = MODE_OF[workload]
    pool = O.Pool(oracle_rate.model, n_envs)
    phase = 2 * np.pi * np.arange(n_envs) / n_envs
    rng = np.random.default_rng(1)
    hi = np.array([12.0, 12.0, 0.9, 12.0, 12.0, 0.9])
    lo_pd = np.radians([-50.0, -164.0, -140.0, -50.0, -164.0, -140.0]); hi_pd = np.radians([80.0, -37.0, -30.0, 80.0, -37.0, -30.0])

    def run(n_steps):
        if mode >= 2:
            return pool.run(n_steps, mode, phase=phase, n_threads=cores)[0]
        nact = (n_steps + 9) // 10
        a = rng.uniform(-1, 1, (n_envs, nact, 6)) * hi if mode == 0 else rng.uniform(lo_pd, hi_pd, (n_envs, nact, 6))
        return pool.run(n_steps, mode, actions=a, hold=10, n_threads=cores)[0]

    run(preadvance)
    n_steps = int(max(50, min(20000, rate * seconds / n_envs)))
    t0 = time.perf_counter()
    n = run(n_steps)
    dt = time.perf_counter() - t0
    pool.close()
    return {"value": n / dt, "unit": "env-steps/s", "cores": cores, "kind": "port",
            "sample": "%d persistent envs x %d sim steps of the same workload after %d pre-advance steps, fp64 oracle (oracle/, gcc -O3 -fopenmp), %.1f s"
                      % (n_envs, n_steps, preadvance, dt)}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path cannot be built here (MuJoCo
    1.50 / RBDL / qpOASES absent), so this times the oracle port on all host cores.  The envs are PERSISTENT
    (oracle.Pool): facades, QP hot start and squat clocks live across the bench steps, exactly like the native
    arm's device state, and they are pre-advanced by the same --preadvance simulator steps before timing."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    O.build()
    cores = os.cpu_count() or 1
    n_envs, sub, wl = args.ref_envs, args.substeps, args.workload     # bounded sample of the 16384-env workload
    mode = MODE_OF[wl]
    pool = O.Pool(O.Model(), n_envs)
    phase = 2 * np.pi * np.arange(n_envs) / max(n_envs, 1)
    rng = np.random.default_rng(1)
    hi = np.array([12.0, 12.0, 0.9, 12.0, 12.0, 0.9])
    lo_pd = np.radians([-50.0, -164.0, -140.0, -50.0, -164.0, -140.0]); hi_pd = np.radians([80.0, -37.0, -30.0, 80.0, -37.0, -30.0])

    def one(n_steps):
        if mode >= 2:
            return pool.run(n_steps, mode, phase=phase, n_threads=cores)[0]
        nact = (n_steps + 9) // 10
        a = rng.uniform(-1, 1, (n_envs, nact, 6)) * hi if mode == 0 else rng.uniform(lo_pd, hi_pd, (n_envs, nact, 6))
        return pool.run(n_steps, mode, actions=a, hold=10, n_threads=cores)[0]

    if args.preadvance > 0:
        one(args.preadvance)
    for _ in range(args.warmup):
        one(sub)
    t0 = time.perf_counter()
    total = 0
    for _ in range(args.steps):
        total += one(sub)
    el = time.perf_counter() - t0
    pool.close()
    v = total / el
    sample = "%d persistent envs x %d sim steps per step, %d steps, pre-advanced %d sim steps; fp64 oracle port, OpenMP over envs" % (
        n_envs, sub, args.steps, args.preadvance)
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": "env-steps/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * el / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOADS[wl], "workload_key": wl, "envs_per_step_sample": n_envs, "substeps": sub,
                       "preadvance_sim_steps": args.preadvance,
                       "note": "CPU restatement (oracle port) of MuJoCo+RBDL path; the reference itself is unbuildable here"},
            "cpu_baseline": {"value": v, "unit": "env-steps/s", "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": v, "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- clocks sampler
class ClockSampler:
    """SM clock and throttle reasons DURING the timed region: NVML polled every 5 ms from a thread (a launch list of
    30 x 1.8 ms is over before `nvidia-smi -lms 100` prints its first line); nvidia-smi is the fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    MASKS = (("sw_power_cap", 0x4), ("hw_slowdown", 0x8), ("sw_thermal_slowdown", 0x20), ("hw_thermal_slowdown", 0x40))

    def __init__(self, index, uuid=None):
        self.index, self.uuid, self.rows, self.proc = index, uuid, [], None
        self.nvml, self.handle, self.thread, self.stop_flag = None, None, None, threading.Event()
        self.sm, self.mask, self.sm_max = [], 0, None

    def _nvml_open(self):
        import pynvml
        pynvml.nvmlInit()
        h = None
        if self.uuid:
            for u in (self.uuid, self.uuid.encode()):
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(u)
                    break
                except Exception:
                    h = None
        if h is None:
            h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        self.nvml, self.handle = pynvml, h
        self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))

    def _poll(self):
        n, h = self.nvml, self.handle
        reasons = getattr(n, "nvmlDeviceGetCurrentClocksEventReasons", None) or n.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self.stop_flag.is_set():
            try:
                self.sm.append(float(n.nvmlDeviceGetClockInfo(h, n.NVML_CLOCK_SM)))
                self.mask |= int(reasons(h))
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        try:
            self._nvml_open()
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nvml:
            self.stop_flag.set()
            self.thread.join(timeout=1)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.sm_max,
                    "reasons": sorted(name for name, bit in self.MASKS if self.mask & bit), "samples": len(self.sm),
                    "source": "nvml, 5 ms poll"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if val.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi -lms 100"}


# ----------------------------------------------------------------------------- output dump
DUMP_BYTES = 60 * 10**6   # keeps a dump, .npy headers included, under 64 MB


def dump_outputs(d, arrays, suffix=""):
    """Writes `arrays` (name -> tensor with one row per env) as d/<name><suffix>.npy in float32, or float64 where the
    path computed in fp64.  Above DUMP_BYTES in all, the same seeded sample of envs is taken from every array and
    env_index<suffix>.npy lists the env indices of its rows."""
    host = {k: v.cpu().numpy() for k, v in arrays.items()}
    host = {k: a.astype(np.float64 if a.dtype == np.float64 else np.float32, copy=False) for k, a in host.items()}
    n = len(next(iter(host.values())))
    row_bytes = sum(a.nbytes for a in host.values()) // n
    if n * row_bytes > DUMP_BYTES:
        keep = np.sort(np.random.default_rng(0).choice(n, DUMP_BYTES // (row_bytes + 8), replace=False))
        host = {k: a[keep] for k, a in host.items()}
        host["env_index"] = keep.astype(np.float64)
    os.makedirs(d, exist_ok=True)
    for k, a in host.items():
        np.save(os.path.join(d, k + suffix + ".npy"), a)


# ----------------------------------------------------------------------------- native arm
def run_native(args):
    import torch
    import torch.distributed as dist
    from cassierl_b200 import envs, lib

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the native arm has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L = lib.load()
    n, sub, wl = args.envs, args.substeps, args.workload
    if args.scaling == "strong":
        if n % world:
            raise SystemExit("bench.py: --scaling strong needs --envs divisible by the number of ranks")
        n = n // world
    dt_t = torch.float64 if args.precision == 64 else torch.float32
    rs = 8 if args.precision == 64 else 4
    gid0 = rank * n                                   # global env ids: results independent of the GPU count
    # every block of `n` consecutive global ids spans one full period of the squat target, so each rank
    # carries the same mix of phases (load balance) and rank r's envs do not depend on the GPU count
    phase = (2 * np.pi * ((gid0 + np.arange(n)) % n) / n).astype(np.float64)
    gen = np.random.default_rng(1 + rank)
    hi = np.array([12.0, 12.0, 0.9, 12.0, 12.0, 0.9])
    n_pre = (args.preadvance + sub - 1) // sub if sub > 0 else 0   # launches that advance every env OUTSIDE the timed region
    total_steps = n_pre + args.warmup + args.steps

    def make():
        if wl == "pd_env":
            return envs.Cassie2dBatchEnv(n, device=local, task="stand", control_mode="PD", precision=args.precision)
        return envs.Cassie2dBatch(n, device=local, precision=args.precision)

    # ---- inputs resident in HBM before the timed region
    obj = make()
    b = obj.batch if wl == "pd_env" else obj
    phase_d = torch.tensor(phase, dtype=dt_t, device=dev)
    if wl == "torque_random":
        acts = torch.tensor(gen.uniform(-1, 1, (total_steps, n, 6)) * hi, dtype=dt_t, device=dev)
    elif wl == "pd_env":
        lo, hh = obj.action_space
        acts = torch.tensor(gen.uniform(lo, hh, (total_steps, n, 6)), dtype=dt_t, device=dev)
        obj.reset()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    def one_step(k):
        if wl == "squat_jacobian":
            b.squat(lib.MODE_JACOBIAN, sub, phase=phase_d)
        elif wl == "squat_osc":
            b.squat(lib.MODE_OSC, sub, phase=phase_d)
        elif wl == "torque_random":
            b.step_torque(acts[k], sub)
        else:
            return obj.step(acts[k], n=sub)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def solver_stats_of(batch):
        st = batch.stats().double()
        return {"rows_mean": float(st[:, 0].mean().item()), "rows_max": int(st[:, 0].max().item()),
                "pgs_sweeps_mean": float(st[:, 1].mean().item()), "qp_iters_mean": float(st[:, 2].mean().item()),
                "qp_not_optimal": int((st[:, 3] != 0).sum().item())}

    # steady state, not the start-up transient: every env is advanced >= --preadvance simulator steps first
    for k in range(n_pre):
        one_step(k)
    for k in range(args.warmup):
        one_step(n_pre + k)
    barrier()
    stats_start = solver_stats_of(b)
    try:
        uuid = "GPU-" + str(torch.cuda.get_device_properties(dev).uuid)
    except Exception:
        uuid = None
    sampler = ClockSampler(local, uuid)
    if rank == 0:
        sampler.start()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    launches0 = L.CassieKernelLaunchCount()
    barrier()
    for k in range(args.steps):
        flush.zero_()                                   # L2 flush, outside the timed events
        ev[k][0].record()
        last = one_step(n_pre + args.warmup + k)
        ev[k][1].record()
    barrier()
    launches = L.CassieKernelLaunchCount() - launches0
    ms = sum(a.elapsed_time(c) for a, c in ev)
    clocks = sampler.stop() if rank == 0 else None
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_max = float(t.item())
    # rollout statistics (NCCL reduce, outside the timed region): mean pelvis height, envs below 0.5 m
    s = b.get_general_state()
    if args.dump_outputs:
        out = {"general_state": s, "operational_space_state": b.get_operational_space_state()}
        if wl == "pd_env":
            out.update(zip(("obs", "reward", "done"), last))
        dump_outputs(args.dump_outputs, out, "_rank%d" % rank if world > 1 else "")
    stats = torch.stack([s[:, 1].double().sum(), (s[:, 1] < 0.5).double().sum(), (~torch.isfinite(s).all(dim=1)).double().sum()])
    if world > 1:
        dist.all_reduce(stats)
    # constraint rows / PGS sweeps / QP iterations of the LAST sim step (rank 0's shard): which solver tier the
    # workload sits in at the end of the timed window (<= 8 rows narrow, <= 12 wide register path, more = cold path)
    solver_stats = solver_stats_of(b)
    value = world * n * sub * args.steps / (ms_max * 1e-3)

    # ---- end to end through the host-buffer C-ABI entry points (pinned host memory in and out)
    obj2 = make()
    b2 = obj2.batch if wl == "pd_env" else obj2
    if wl == "pd_env":
        obj2.reset()
    ph_h = torch.tensor(phase, dtype=dt_t).pin_memory()
    st_h = torch.empty((n, 26), dtype=dt_t).pin_memory()
    if wl in ("torque_random", "pd_env"):
        acts_h = acts.cpu().pin_memory()
        obs_h = torch.empty((n, 17), dtype=dt_t).pin_memory(); rew_h = torch.empty(n, dtype=dt_t).pin_memory()
        done_h = torch.empty(n, dtype=torch.uint8).pin_memory()

    def one_e2e(k):
        if wl == "squat_jacobian":
            b2.squat_host(lib.MODE_JACOBIAN, sub, ph_h, st_h); return n * rs, n * 26 * rs
        if wl == "squat_osc":
            b2.squat_host(lib.MODE_OSC, sub, ph_h, st_h); return n * rs, n * 26 * rs
        if wl == "torque_random":
            b2.step_host(lib.MODE_TORQUE, acts_h[k], sub, st_h); return n * 6 * rs, n * 26 * rs
        obj2.step_host(acts_h[k], obs_h, rew_h, done_h, n=sub); return n * 6 * rs, n * (17 * rs + rs + 1)

    for k in range(n_pre):                                    # same steady state as the device-timed leg
        if wl == "squat_jacobian":
            b2.squat(lib.MODE_JACOBIAN, sub, phase=phase_d)
        elif wl == "squat_osc":
            b2.squat(lib.MODE_OSC, sub, phase=phase_d)
        elif wl == "torque_random":
            b2.step_torque(acts[k], sub)
        else:
            obj2.step(acts[k], n=sub)
    for k in range(args.warmup):
        h2d, d2h = one_e2e(n_pre + k)
    barrier()
    t0 = time.perf_counter()
    for k in range(args.steps):
        one_e2e(n_pre + args.warmup + k)
    torch.cuda.synchronize()
    el = time.perf_counter() - t0
    t = torch.tensor([el], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = world * n * sub * args.steps / float(t.item())

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        # DRAM bytes per launch from the last `ncu --set full` capture of this workload -- printed only while the
        # capture's kernel sources are the ones being timed (profiles/traffic.json records their hash), else null
        traffic, traffic_src = None, None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(wl, {})
            if tr.get("kernel_source_sha16") == kernel_source_hash():
                traffic, traffic_src = tr.get("dram_bytes_per_launch"), tr.get("capture")
            elif tr:
                traffic_src = "stale: capture %s ran other kernel sources" % tr.get("capture")
        except Exception:
            pass
        fp32_peak = L.CassieMeasureFp32Peak(local)            # TFLOP/s, measured live on this GPU
        fl = FLOPS_PER_STEP.get(wl) or 0.0
        flops_launch = fl * n * sub
        ms_launch = ms_max / args.steps
        achieved = flops_launch / (ms_launch * 1e-3) / 1e12
        bytes_launch = n * (STATE_BYTES_PER_ENV_F32 * rs // 4 + rs)
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        line = {
            "metric": METRIC, "value": value, "unit": "env-steps/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_launch, "higher_is_better": True, "scaling": args.scaling,
            "vs_baseline": None, "dtype": "f32" if args.precision == 32 else "f64", "data": "synthetic",
            "config": {"workload": WORKLOADS[wl], "workload_key": wl, "envs_per_gpu": n, "sim_steps_per_launch": sub,
                       "policy_steps_per_s": value / sub, "preadvance_sim_steps": n_pre * sub,
                       "l2": "flushed between timed steps (256 MiB memset)",
                       "parallelism": "env-sharded dp%d, no data-path collective" % world},
            "roofline": {"bound": "fp32", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                         "frac": achieved / fp32_peak if fp32_peak > 0 else None, "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": "measured live: register-only FFMA kernel (CassieMeasureFp32Peak); MEASURED_PEAKS.json has no FP32 figure",
                         "flops_per_env_step": fl, "kernel_ms": ms_launch,
                         "hbm": {"achieved_gbs": bytes_launch / (ms_launch * 1e-3) / 1e9, "peak_gbs": hbm_peak,
                                 "peak_source": "MEASURED_PEAKS.json (measured)" if peaks else "fallback",
                                 "algorithmic_bytes_per_launch": bytes_launch}},
            "e2e": {"value": e2e_value, "unit": "env-steps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h},
            "gpu_launches": int(launches), "clocks": clocks,
            "stats": {"mean_pelvis_z": float(stats[0].item()) / (n * world), "envs_below_0.5m": int(stats[1].item()),
                      "non_finite_envs": int(stats[2].item()), "first_timed_step": stats_start, "last_step": solver_stats},
        }
        if not args.no_cpu_baseline and world == 1:
            line["cpu_baseline"] = cpu_baseline(wl, args.cpu_seconds, args.preadvance)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    if a.impl == "reference":
        run_reference(a)
    else:
        run_native(a)
