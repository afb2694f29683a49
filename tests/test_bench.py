"""bench.py --dump-outputs: what the timed path computed, whole or as a fixed row sample below 64 MB."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_outputs_whole_matrix(tmp_path):
    phi = np.random.default_rng(1).random((300, 300)).astype(np.float32)
    bench.dump_outputs(str(tmp_path), phi)
    assert os.listdir(tmp_path) == ["phi.npy"]
    got = np.load(tmp_path / "phi.npy")
    assert got.dtype == np.float32 and np.array_equal(got, phi)


@pytest.mark.parametrize("dtype", [np.float32, np.float64])
def test_dump_outputs_row_sample_is_fixed_and_small(tmp_path, dtype):
    n = 4100 if dtype == np.float32 else 2900                      # just above the budget
    phi = np.repeat(np.arange(n, dtype=dtype)[:, None], n, axis=1)   # row i holds i
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), phi)
        assert os.listdir(tmp_path / run) == ["phi_row_sample.npy"]
        assert os.path.getsize(tmp_path / run / "phi_row_sample.npy") < 64_000_000
    a, b = np.load(tmp_path / "a" / "phi_row_sample.npy"), np.load(tmp_path / "b" / "phi_row_sample.npy")
    assert a.dtype == dtype and np.array_equal(a, b)
    rows = a[:, 0].astype(np.int64)
    assert a.shape == (bench.DUMP_BYTES // (n * a.itemsize), n) and len(rows) > n // 2
    assert (np.diff(rows) > 0).all() and (a == a[:, :1]).all()     # distinct whole rows, in order


def run_bench(out_dir, *args):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "genea140", "--steps", "2",
                          "--warmup", "0", "--cpu-seconds", "0", "--e2e-steps", "0", "--dump-outputs", str(out_dir),
                          *args], capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    return json.loads(res.stdout)


def test_reference_arm_dumps_its_matrix(tmp_path, genea140_oracle):
    _, want, _ = genea140_oracle
    line = run_bench(tmp_path, "--impl", "reference", "--ref-mode", "full")
    assert line["parity"]["matches_golden"] is True
    assert np.array_equal(np.load(tmp_path / "phi.npy"), want)


@pytest.mark.gpu
def test_bench_dumps_the_matrix_of_its_timed_steps(tmp_path, genea140_oracle):
    _, want, _ = genea140_oracle
    line = run_bench(tmp_path)
    assert line["steps"] == 2 and line["parity"]["matches_golden"] is True
    got = np.load(tmp_path / "phi.npy")
    assert got.dtype == np.float32 and np.array_equal(got, want)
