"""bench.py's command line: the reference arm (--impl reference), the one leg that runs without a GPU, prints the
benchmark's JSON line on every CPU test run; --dump-outputs writes what the timed path returned (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from conftest import ROOT


def test_reference_arm_prints_the_contract_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "1",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.strip().splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "couplings/s" and d["higher_is_better"] is True
    for key in ("metric", "value", "n_gpus", "steps", "warmup", "ms_per_step", "scaling", "vs_baseline", "dtype",
                "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in d, key
    assert d["steps"] == 1 and d["warmup"] == 1 and d["value"] > 0 and d["gpu_launches"] == 0
    assert "workload" in d["config"]
    cb, e2e = d["cpu_baseline"], d["e2e"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert e2e["value"] == d["value"] and e2e["unit"] == d["unit"]
    assert e2e["h2d_bytes_per_step"] == 0 and e2e["d2h_bytes_per_step"] == 0
    assert abs(d["ms_per_step"] * d["value"] - 1e3) < 1e-6 * 1e3


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", LOCAL_RANK="1", WORLD_SIZE="2")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "1"], capture_output=True, text=True, timeout=600, cwd=ROOT,
                         env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    assert not [ln for ln in out.stdout.splitlines() if ln.startswith("{")]


def test_dump_outputs_is_refused_on_the_reference_arm(tmp_path):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode == 2 and "--dump-outputs" in out.stderr, out.stderr[-2000:]
    assert not list(tmp_path.iterdir())


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_coupled_batch(tmp_path):
    """--dump-outputs DIR: the last timed step's sample_plan pair, float32, within 64 MB; every row is a row of the
    seeded synthetic batch (rank 0: torch.Generator().manual_seed(0), x0 then x1)."""
    env = dict(os.environ, CFM_BENCH_NOCLK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "1",
                          "--no-extra", "--no-ode", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900, cwd=ROOT, env=env)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads([ln for ln in out.stdout.splitlines() if ln.startswith("{")][-1])["steps"] == 2
    files = sorted(p.name for p in tmp_path.iterdir())
    assert files == ["x0_coupled.npy", "x1_coupled.npy"]
    assert sum(p.stat().st_size for p in tmp_path.iterdir()) <= 64 << 20
    g = torch.Generator().manual_seed(0)
    for name in ("x0", "x1"):
        src = torch.randn(8192, 784, generator=g).numpy()
        got = np.load(tmp_path / f"{name}_coupled.npy")
        assert got.dtype == np.float32 and got.shape == src.shape
        rows = {r.tobytes() for r in src}
        assert all(r.tobytes() in rows for r in got), name
