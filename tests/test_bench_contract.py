"""bench.py's driver contract, the parts that run without a GPU: the reference arm prints exactly one JSON line on stdout with the
keys the driver reads; under a multi-rank launch only rank 0 prints; the GPU arm refuses to run without a device (no CPU fallback)."""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(args, env=None, timeout=300):
    e = dict(os.environ, OMP_WAIT_POLICY="PASSIVE")
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True, timeout=timeout, env=e, cwd=ROOT)


def test_reference_arm_prints_one_contract_line():
    r = run_bench(["--impl", "reference", "--steps", "2", "--warmup", "1"])
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "impl",
                "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["steps"] == 2 and d["value"] > 0 and d["higher_is_better"] is True
    assert d["unit"] == "registrations/s" and "workload" in d["config"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["value"] == d["value"] and cb["cores"] >= 1 and cb["sample"]


def test_reference_arm_only_rank0_prints():
    r = run_bench(["--impl", "reference", "--steps", "1", "--warmup", "0", "--gpus", "2"], env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_gpu_arm_refuses_to_run_without_a_device():
    import torch

    if torch.cuda.is_available():
        return
    r = run_bench([])
    assert r.stdout.strip() == "" and "no CPU fallback" in (r.stderr + r.stdout)


def test_dump_outputs_keep_small_arrays_and_sample_large_clouds(tmp_path):
    """--dump-outputs: small arrays are written as they are; aligned clouds above the budget become the same seeded rows of every
    stream, with the row indices beside them, identical from run to run."""
    import bench

    pose = np.arange(32, dtype=np.float64).reshape(2, 4, 4)
    cloud = np.random.default_rng(3).random((2, 50000, 3), dtype=np.float32)
    for d in ("a", "b"):
        bench.write_outputs(str(tmp_path / d), {"pose": pose, "e2e_aligned": cloud}, aligned_budget=120000)
    assert sorted(os.listdir(tmp_path / "a")) == ["e2e_aligned.npy", "e2e_aligned_rows.npy", "pose.npy"]
    assert np.array_equal(np.load(tmp_path / "a" / "pose.npy"), pose)
    got, rows = np.load(tmp_path / "a" / "e2e_aligned.npy"), np.load(tmp_path / "a" / "e2e_aligned_rows.npy")
    assert got.dtype == np.float32 and rows.dtype == np.float64 and got.nbytes <= 120000 and got.shape == (2, len(rows), 3)
    assert len(np.unique(rows)) == len(rows) and np.array_equal(got, cloud[:, rows.astype(np.int64)])
    assert np.array_equal(np.load(tmp_path / "b" / "e2e_aligned.npy"), got)
    bench.write_outputs(str(tmp_path / "c"), {"e2e_aligned": cloud[:, :100]}, aligned_budget=120000)
    assert sorted(os.listdir(tmp_path / "c")) == ["e2e_aligned.npy"] and np.array_equal(np.load(tmp_path / "c" / "e2e_aligned.npy"), cloud[:, :100])
