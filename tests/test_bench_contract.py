"""CPU suite: the reference arm of bench.py (the unmodified reference staged under oracle/_ref — or /root/reference — on the
host cores; the CPU port only where neither exists) runs here and prints ONE JSON line with the contract's keys; the product
arm refuses to run without a CUDA device (no CPU fallback).  On a GPU, the product arm's --dump-outputs is checked."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_json_line():
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1", "--sample", "64"],
                       capture_output=True, text=True, timeout=600)
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "rays/s" and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["metric"].startswith("rays/sec (train fwd+bwd") and d["scaling"] == "weak" and d["data"] == "synthetic"
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["n_gpus"] == 1
    assert d["steps"] == 2 and d["warmup"] == 1                      # --steps / --warmup are honoured, not capped
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.workload_config(4096, 1)             # the SAME config object as the product arm prints
    from oracle import ref_import
    cb = d["cpu_baseline"]
    assert cb["kind"] == ("reference" if ref_import.available() else "port")
    assert cb["cores"] == bench.host_threads() and cb["value"] == d["value"] and "64 of the 4096 rays" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "rays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_uses_all_cores_under_torchrun():
    """torchrun exports OMP_NUM_THREADS=1; the CPU arm must not inherit it (round-1 SCALE ratios were void because it did)."""
    env = dict(os.environ, RANK="0", WORLD_SIZE="2", LOCAL_RANK="0", OMP_NUM_THREADS="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1",
                        "--warmup", "0", "--sample", "32"], capture_output=True, text=True, timeout=600, env=env)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([ln for ln in p.stdout.splitlines() if ln.startswith("{")][0])
    sys.path.insert(0, ROOT)
    import bench
    assert d["cpu_baseline"]["cores"] == bench.host_threads() and d["n_gpus"] == 2


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2", "--steps", "1"],
                       capture_output=True, text=True, timeout=300, env=env)
    assert p.returncode == 0 and not [ln for ln in p.stdout.splitlines() if ln.startswith("{")]


def test_product_arm_has_no_cpu_fallback():
    import torch
    if torch.cuda.is_available():
        return
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1"], capture_output=True, text=True, timeout=300)
    assert p.returncode != 0 and "no CPU fallback" in (p.stderr + p.stdout)


@pytest.mark.gpu
def test_product_arm_dumps_the_last_timed_step(tmp_path):
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "3", "--no-cpu-baseline",
                        "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads([ln for ln in p.stdout.splitlines() if ln.startswith("{")][-1])
    assert d["steps"] == 2
    files = sorted(tmp_path.glob("*.npy"))
    assert sum(f.stat().st_size for f in files) <= 64 << 20
    out = {f.stem: np.load(f) for f in files}
    assert all(v.dtype in (np.float32, np.float64) and np.isfinite(v).all() for v in out.values())
    assert float(out["loss"]) > 0
    params = [k[len("param."):] for k in out if k.startswith("param.")]
    assert len(params) == 48 and sorted(params) == sorted(k[len("grad."):] for k in out if k.startswith("grad."))
    assert len(out) == 1 + 2 * len(params)
    for k in params:
        assert out["param." + k].shape == out["grad." + k].shape and np.abs(out["grad." + k]).max() > 0, k
