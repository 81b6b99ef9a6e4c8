"""bench.py contract (CPU): the reference arm prints exactly one JSON line with the keys the
driver reads; the GPU arm fails loudly without a GPU instead of falling back."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REQUIRED = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
            "vs_baseline", "dtype", "data", "config", "e2e", "impl", "cpu_baseline"}


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600,
                         env={**os.environ, "CUDA_VISIBLE_DEVICES": ""})
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert REQUIRED <= set(d), sorted(REQUIRED - set(d))
    assert d["impl"] == "reference" and d["unit"] == "samples/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "reference" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert d["config"]["workload"].startswith("ResNet-50")


def test_reference_arm_non_zero_ranks_exit_quietly():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=120,
                         env={**os.environ, "RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert out.returncode == 0 and out.stdout.strip() == ""


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bad_arguments_are_refused(extra):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *extra], capture_output=True, text=True,
                         timeout=120)
    assert out.returncode == 2 and out.stdout.strip() == "", out.stderr[-2000:]


@pytest.mark.gpu
def test_gpu_arm_dumps_the_last_timed_step(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "1",
                          "--no-cpu-baseline", "--dump-outputs", str(tmp_path)], capture_output=True, text=True,
                         timeout=900)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1 and json.loads(lines[0])["steps"] == 2
    files = {p.name: p for p in tmp_path.iterdir()}
    assert set(files) == {"loss.npy", "params.npy", "buffers.npy"}
    assert sum(p.stat().st_size for p in files.values()) <= 64 << 20
    for p in files.values():
        a = np.load(p)
        assert a.dtype == np.float32 and a.size > 0 and np.isfinite(a).all(), p.name


def test_gpu_arm_fails_loudly_without_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=300)
    assert out.returncode != 0 and out.stdout.strip() == ""
