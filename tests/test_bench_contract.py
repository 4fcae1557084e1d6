"""CPU-side check of bench.py's output contract: the reference arm runs without a GPU, prints exactly one JSON line on
stdout with the keys the driver reads, and the product arm refuses to run without CUDA."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, timeout=300, env=env)


def test_reference_arm_prints_one_json_line():
    out = _run("--impl", "reference", "--ref-points", "60000", "--queries", "20000", "--steps", "2", "--warmup", "1")
    assert out.returncode == 0, out.stderr
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert key in d, key
    assert d["impl"] == "reference" and d["unit"] == "queries/s" and d["value"] > 0 and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["h2d_bytes_per_step"] == 0 and d["e2e"]["d2h_bytes_per_step"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]


def test_product_arm_needs_cuda():
    import torch
    if torch.cuda.is_available():
        return
    out = _run("--ref-points", "1000", "--queries", "1000", "--steps", "1")
    assert out.returncode != 0 and "no CPU fallback" in (out.stderr + out.stdout)
    assert out.stdout.strip() == ""


def test_reference_arm_ignores_omp_num_threads_1():
    """torch.distributed.run exports OMP_NUM_THREADS=1; the reference arm must still use every core it may run on, so that the
    CPU baseline is the same at every --gpus N (round-1 VERDICT: the N >= 2 ratios were void because `cores` fell to 1)."""
    avail = len(os.sched_getaffinity(0))
    out = _run("--impl", "reference", "--gpus", "2", "--ref-points", "60000", "--queries", "20000", "--steps", "1", "--warmup", "1", env={**os.environ, "OMP_NUM_THREADS": "1"})
    assert out.returncode == 0, out.stderr
    d = json.loads([ln for ln in out.stdout.splitlines() if ln.strip()][0])
    assert d["cpu_baseline"]["cores"] == avail and d["n_gpus"] == 2 and d["scaling"] == "strong"


def test_steps_must_be_positive():
    out = _run("--impl", "reference", "--steps", "0")
    assert out.returncode == 2 and "--steps" in out.stderr and out.stdout.strip() == ""


def test_dump_rows_fixed_sample_within_budget():
    import bench
    for n, k in ((10_000_000, 16), (10_000_000, 512), (20_000, 300)):
        rows = bench.dump_rows(n, k)
        assert len(rows) * (12 * k + 8) + 3 * 128 <= 64_000_000 and len(rows) < n
        assert (np.diff(rows) > 0).all() and rows[0] >= 0 and rows[-1] < n
        assert np.array_equal(rows, bench.dump_rows(n, k))
    assert np.array_equal(bench.dump_rows(20_000, 16), np.arange(20_000))


def _check_dump(path, n, nq, k):
    """The dumped rows are the bench workload's kNN rows: same (idx, d2) as the oracle on the same seeded clouds."""
    import argparse

    import bench
    import oracle
    files = {f: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}
    assert list(files) == ["knn_indices.npy", "knn_sqr_distances.npy", "query_rows.npy"]
    assert sum(os.path.getsize(os.path.join(path, f)) for f in files) <= 64_000_000
    rows, idx, d2 = files["query_rows.npy"], files["knn_indices.npy"], files["knn_sqr_distances.npy"]
    assert rows.dtype == idx.dtype == np.float64 and d2.dtype == np.float32 and idx.shape == d2.shape == (len(rows), k)
    ref, qry = bench.make_clouds(argparse.Namespace(cloud="surface", n=n, nq=nq), 0)
    oi, od, _ = oracle.KdTree(ref).knn(qry[rows.astype(np.int64)], k)
    assert np.array_equal(idx, oi) and np.array_equal(d2.view(np.uint32), od.view(np.uint32))


def test_dump_outputs_reference_arm(tmp_path):
    out = _run("--impl", "reference", "--ref-points", "60000", "--queries", "20000", "--steps", "2", "--warmup", "1", "--dump-outputs", str(tmp_path))
    assert out.returncode == 0, out.stderr
    _check_dump(tmp_path, 60000, 20000, 16)


@pytest.mark.gpu
def test_dump_outputs_product_arm(tmp_path):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    out = _run("--ref-points", "200000", "--queries", "400000", "--steps", "2", "--warmup", "1", "--no-cpu", "--no-c4", "--no-parity",
               "--dump-outputs", str(tmp_path))         # 400000 rows exceed the 64 MB budget: the seeded sample is written
    assert out.returncode == 0, out.stderr
    assert json.loads(out.stdout)["steps"] == 2
    _check_dump(tmp_path, 200000, 400000, 16)
