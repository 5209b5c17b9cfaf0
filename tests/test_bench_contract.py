"""bench.py contract on the CPU: the reference arm runs without a GPU and prints ONE JSON line with the keys the driver
reads (same metric string as the native arm, so that the driver can divide one by the other); the native arm refuses to
run without a CUDA device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import pytest

from conftest import ROOT


def _run(args, **kw):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=600, **kw)


def test_reference_arm_json_line(oracle):
    r = _run(["--impl", "reference", "--steps", "2", "--warmup", "1", "--ref-envs", "8", "--preadvance", "20"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    import bench
    assert d["impl"] == "reference" and d["metric"] == bench.METRIC and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "env-steps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["workload_key"] == bench.DEFAULT_WORKLOAD


def test_reference_arm_other_ranks_exit_quietly(oracle):
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = _run(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"], env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_native_arm_refuses_cpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    r = _run(["--steps", "1", "--warmup", "0"])
    assert r.returncode != 0 and "no CUDA device" in (r.stderr + r.stdout)


@pytest.mark.gpu
@pytest.mark.parametrize("workload", ["squat_osc", "pd_env"])
def test_dump_outputs_repeat_bit_for_bit(workload, tmp_path):
    """--dump-outputs writes the last timed step's results; the same arguments give the same inputs, hence the same files"""
    import numpy as np
    n = 512
    names = ("obs", "reward", "done") if workload == "pd_env" else ()
    dumps = []
    for k in range(2):
        d = tmp_path / str(k)
        r = _run(["--workload", workload, "--envs", str(n), "--steps", "3", "--warmup", "1", "--preadvance", "20",
                  "--no-cpu-baseline", "--dump-outputs", str(d)])
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads([l for l in r.stdout.splitlines() if l.startswith("{")][-1])["steps"] == 3
        dumps.append({f.stem: np.load(f) for f in sorted(d.glob("*.npy"))})
    shapes = {"general_state": (n, 26), "operational_space_state": (n, 18), "obs": (n, 17), "reward": (n,), "done": (n,)}
    assert sorted(dumps[0]) == sorted(("general_state", "operational_space_state") + names)
    for name, a in dumps[0].items():
        assert a.shape == shapes[name] and a.dtype == np.float32 and np.isfinite(a).all()
        assert np.array_equal(a, dumps[1][name]), name


def test_traffic_stamp_matches_sources():
    """profiles/traffic.json carries the hash of the kernel sources its ncu capture ran; bench.py prints the number only
    while they are the sources being timed"""
    import bench
    t = json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
    assert t["squat_osc"]["kernel_source_sha16"] == bench.kernel_source_hash()
    assert 1e6 < t["squat_osc"]["dram_bytes_per_launch"] < 5e7
