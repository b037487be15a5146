"""bench.py --dump-outputs: what the last timed step returned, written as .npy files so that two builds can be compared."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from npairloss_b200 import synth

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_samples_the_rows_of_a_large_gradient(tmp_path):
    """Above the size cap the gradient is written as a seeded sample of its rows, the same rows on every run."""
    code = ("import sys, torch; sys.path.insert(0, sys.argv[2]); import bench; bench.DUMP_BYTES = 3 << 20; "
            "g = torch.arange(4096 * 256, dtype=torch.float32).reshape(4096, 256); "
            "bench.dump_outputs(sys.argv[1], [1, 2, 3, 4, 5], g, 1, 0); bench.dump_outputs(sys.argv[1] + '_small', [1, 2, 3, 4, 5], g[:64], 1, 0)")
    for run in ("a", "b"):
        subprocess.run([sys.executable, "-c", code, str(tmp_path / run), ROOT], check=True, timeout=300)
    a, b = tmp_path / "a", tmp_path / "b"
    assert sorted(os.listdir(a)) == ["dx_sample.npy", "dx_sample_rows.npy", "tops.npy"]
    assert sum(os.path.getsize(a / f) for f in os.listdir(a)) <= 3 << 20
    rows, dx = np.load(a / "dx_sample_rows.npy"), np.load(a / "dx_sample.npy")
    assert rows.dtype == np.float64 and dx.dtype == np.float32 and dx.shape == (rows.size, 256) and rows.size > 1000
    assert np.all(np.diff(rows) > 0) and rows[-1] < 4096
    np.testing.assert_array_equal(dx, np.arange(4096 * 256, dtype=np.float32).reshape(4096, 256)[rows.astype(np.int64)])
    np.testing.assert_array_equal(np.load(b / "dx_sample_rows.npy"), rows)
    np.testing.assert_array_equal(np.load(a / "tops.npy"), np.float32([[1, 2, 3, 4, 5]]))
    small = tmp_path / "a_small"
    assert sorted(os.listdir(small)) == ["dx.npy", "tops.npy"]
    np.testing.assert_array_equal(np.load(small / "dx.npy"), np.arange(64 * 256, dtype=np.float32).reshape(64, 256))


@pytest.mark.gpu
def test_bench_dumps_the_timed_step(tmp_path, oracle):
    """C2 (B = 512, D = 128, RAND mining: every pair, no threshold to land near) through the bench's timed path; the dump
    matches the oracle at the fp32-faithful tolerances of tests/test_golden.py."""
    out = tmp_path / "dump"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--config", "C2", "--steps", "3", "--warmup", "1",
                        "--no-cpu-baseline", "--no-extras", "--dump-outputs", str(out)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stderr[-3000:]
    res = json.loads(r.stdout.strip().splitlines()[-1])
    assert res["steps"] == 3
    assert sorted(os.listdir(out)) == ["dx.npy", "tops.npy"]
    tops, dx = np.load(out / "tops.npy"), np.load(out / "dx.npy")
    assert tops.dtype == np.float32 and tops.shape == (1, 5) and dx.dtype == np.float32 and dx.shape == (512, 128)
    c = synth.CONFIGS["C2"]
    x, lab = synth.config_inputs("C2")
    tops_o, dx_o = oracle.step_world(x, lab, oracle.make_config(512, 128, **c["mining"]), 1.0)
    np.testing.assert_allclose(tops[0, 0], tops_o[0, 0], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(tops[0, 1:4], tops_o[0, 1:4], atol=1.001 / 512)
    np.testing.assert_allclose(tops[0, 4], tops_o[0, 4], rtol=2e-6)
    assert np.linalg.norm(dx - dx_o) <= 1e-5 * np.linalg.norm(dx_o)
