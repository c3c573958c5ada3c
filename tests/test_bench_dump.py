"""bench.py --dump-outputs: the sample it writes is the solution at fixed grid points, in the solution's dtype, and stays
within 64 MB at the benchmark's batch and grid.  (No GPU needed: the writer takes any tensor.)  The writer runs in a
subprocess so that torch's CPU thread pool is not started in this process before test_dist_cpu forks its workers."""
import os
import subprocess
import sys

import numpy as np

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = r'''
import sys
sys.path.insert(0, %(root)r)
import numpy as np, torch
import bench
x = torch.from_numpy(np.random.default_rng(3).standard_normal((bench.B_PER_GPU, bench.GRID[0] * bench.GRID[1]), dtype=np.float32))
for d in sys.argv[1:]:
    bench.dump_outputs(d, x)
'''


def test_dump_is_a_fixed_column_sample_within_64_mb(tmp_path):
    B, M, points = bench.B_PER_GPU, bench.GRID[0] * bench.GRID[1], bench.DUMP_POINTS
    a_dir, b_dir = str(tmp_path / "a"), str(tmp_path / "b")
    r = subprocess.run([sys.executable, "-c", SCRIPT % {"root": ROOT}, a_dir, b_dir], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-3000:]
    assert os.listdir(a_dir) == ["pcg_x_sample.npy"]
    pa = os.path.join(a_dir, "pcg_x_sample.npy")
    a = np.load(pa)
    assert a.dtype == np.float32 and a.shape == (B, points)
    assert os.path.getsize(pa) <= 64 * 2 ** 20
    assert np.array_equal(a, np.load(os.path.join(b_dir, "pcg_x_sample.npy")))
    x = np.random.default_rng(3).standard_normal((B, M), dtype=np.float32)
    cols = np.sort(np.random.default_rng(0).choice(M, points, replace=False))
    assert np.array_equal(a, x[:, cols])
