"""bench.py contract pieces that do not need a GPU: the reference arm (CPU oracle on config C3) prints one JSON
line with the agreed keys; the CUDA arm refuses to run without a device instead of falling back."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "simulated node-rounds/sec" and d["unit"] == "node-rounds/s"
    assert d["higher_is_better"] is True and d["steps"] == 3 and d["warmup"] == 3 and d["value"] > 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": "node-rounds/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["config"]["n_nodes"] == 1 << 20 and "workload" in d["config"]


def test_reference_arm_dump_outputs_are_bounded_and_repeatable(tmp_path):
    """--dump-outputs at the full C3 size: float64 files within 64 MB, the same bytes from two runs with the same arguments."""
    import numpy as np
    dumps = []
    for run in ("a", "b"):
        out = tmp_path / run
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "3", "--warmup", "3",
                            "--dump-outputs", str(out)], capture_output=True, text=True, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        dumps.append({f: np.load(out / f) for f in sorted(os.listdir(out))})
    a, b = dumps
    assert sorted(a) == sorted(b) and "counters.npy" in a and "nbr.npy" in a
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in a) <= 64 << 20
    assert len(a["sample_nodes.npy"]) == 32768 and a["nbr.npy"].shape == (32768, 32)
    for f in a:
        assert a[f].dtype == np.float64 and np.array_equal(a[f], b[f]), f
    assert a["counters.npy"][0] > 0  # pings of 6 rounds


def test_reference_arm_uses_all_host_threads_under_torchrun():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm must still use every core it may."""
    if len(os.sched_getaffinity(0)) < 2:
        pytest.skip("single-core box")
    env = dict(os.environ, RANK="0", WORLD_SIZE="2", LOCAL_RANK="0", OMP_NUM_THREADS="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "3"],
                       capture_output=True, text=True, timeout=600, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip())
    assert d["cpu_baseline"]["cores"] >= 2 and d["n_gpus"] == 2


def test_reference_arm_other_ranks_stay_silent():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "3"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_cuda_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "3"], capture_output=True, text=True, timeout=300)
    assert r.returncode != 0 and "no CPU fallback" in (r.stderr + r.stdout)
