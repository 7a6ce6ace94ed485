"""bench.py contract on CPU: the reference arm runs without a GPU and prints ONE JSON line with the agreed keys; the
B200 arm refuses to produce a number without a device (no CPU fallback).  On both arms --dump-outputs writes the y
that the timed path computed."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          env=dict(os.environ, **(env or {})), timeout=600)


def test_reference_arm_line():
    r = run("--impl", "reference", "--mini", "--steps", "3", "--warmup", "1")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "SpMV GFLOP/s" and d["unit"] == "GFLOP/s"
    assert d["steps"] == 3 and d["warmup"] == 1 and d["n_gpus"] == 1 and d["higher_is_better"] is True
    assert d["value"] > 0 and d["ms_per_step"] > 0 and d["dtype"] == "f64" and d["data"] == "synthetic"
    assert d["vs_baseline"] is None and d["gpu_launches"] == 0
    assert d["config"]["workload"].startswith("c5:") and d["scaling"] == "strong"
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "rows" in cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "GFLOP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_under_torchrun_env():
    """Ranks other than 0 exit 0 without work; rank 0 ignores the launcher's OMP_NUM_THREADS=1."""
    r = run("--impl", "reference", "--mini", "--steps", "2", "--warmup", "1", "--gpus", "2", env={"RANK": "1", "WORLD_SIZE": "2"})
    assert r.returncode == 0 and r.stdout.strip() == ""
    r = run("--impl", "reference", "--mini", "--steps", "2", "--warmup", "1", "--gpus", "2",
            env={"RANK": "0", "WORLD_SIZE": "2", "OMP_NUM_THREADS": "1"})
    d = json.loads(r.stdout.strip())
    assert d["n_gpus"] == 2 and d["config"]["workload"].startswith("c5:") and d["scaling"] == "strong"


def test_b200_arm_needs_a_gpu():
    import singlespmv_b200 as sp
    if sp.device_count() > 0:
        import pytest
        pytest.skip("a CUDA device is present")
    r = run("--mini", "--steps", "2", "--no-cpu")
    assert r.returncode != 0 and r.stdout.strip() == ""        # no number without the device


def mini_c5_result(oracle):
    """y = A x of the --mini headline matrix (3-D 7-point Laplacian 64^3), x as bench.py makes it."""
    nRow, nCol, row, col, val = oracle.stencil("lap3d7", 64)
    x, _ = oracle.reference_vectors(nCol, 0, 3)
    return oracle.crs_result(nRow, row, col, val, x)


def test_reference_arm_dump_outputs(oracle, tmp_path):
    r = run("--impl", "reference", "--mini", "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["y.npy"]                 # small enough to keep every row
    assert np.array_equal(np.load(tmp_path / "y.npy"), mini_c5_result(oracle))


def test_dump_outputs_samples_large_results(tmp_path):
    import bench
    y = np.random.default_rng(5).standard_normal(bench.DUMP_ROWS + 1000).astype(np.float32)
    bench.dump_outputs(str(tmp_path), y)
    rows = np.load(tmp_path / "y_rows.npy")
    assert rows.dtype == np.float64 and len(rows) == bench.DUMP_ROWS and np.all(np.diff(rows) > 0) and rows[-1] < len(y)
    ys = np.load(tmp_path / "y.npy")
    assert ys.dtype == np.float32 and np.array_equal(ys, y[rows.astype(np.int64)])
    bench.dump_outputs(str(tmp_path), y)                                # fixed sample: the same rows again
    assert np.array_equal(np.load(tmp_path / "y_rows.npy"), rows)
    bench.dump_outputs(str(tmp_path), y[:10])                           # whole result: no stale row list left behind
    assert sorted(os.listdir(tmp_path)) == ["y.npy"] and np.array_equal(np.load(tmp_path / "y.npy"), y[:10])


def test_steps_must_be_positive():
    r = run("--impl", "reference", "--mini", "--steps", "0")
    assert r.returncode != 0 and r.stdout.strip() == ""


@pytest.mark.gpu
def test_b200_arm_dump_outputs(oracle, tmp_path):
    r = run("--mini", "--steps", "4", "--warmup", "3", "--configs", "none", "--no-cpu", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip())
    assert d["steps"] == 4 and d["config"]["format"] == "crs"
    y = np.load(tmp_path / "y.npy")
    y_ref = mini_c5_result(oracle)
    assert y.dtype == np.float64
    np.testing.assert_allclose(y, y_ref, rtol=1e-12, atol=1e-12)
