"""bench.py --dump-outputs on the GPU: the file holds what the timed PCG step returned on the benchmark's seeded input
(rank 0: generator seed 42), at the grid points the writer samples."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_is_the_timed_steps_solution(tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "1", "--warmup", "1", "--quick",
                        "--no-cpu", "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-3000:]
    got = np.load(tmp_path / "pcg_x_sample.npy")
    import torch
    from hipgp_b200.plan import Plan
    dev = torch.device("cuda", 0)
    M = bench.GRID[0] * bench.GRID[1]
    plan = Plan(bench.GRID, torch.float32, dev)
    plan.set_first_row(bench.first_row(torch.float32, dev))
    gen = torch.Generator(device=dev); gen.manual_seed(42)
    b = torch.randn(bench.B_PER_GPU, M, dtype=torch.float32, device=dev, generator=gen)
    x = plan.pcg(b, maxiter=bench.MAXITER, tol=bench.TOL, precond=True)
    cols = np.sort(np.random.default_rng(0).choice(M, bench.DUMP_POINTS, replace=False))
    assert got.shape == (bench.B_PER_GPU, bench.DUMP_POINTS) and got.dtype == np.float32
    assert np.array_equal(got, x[:, torch.from_numpy(cols).to(dev)].cpu().numpy())
