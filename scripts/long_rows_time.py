"""Times 2-D grids whose last axis runs the four-step path (long1d_kernels.cuh between the column passes of the leading axis):
(3000, 3000) and (64, 20000) inducing points, Matern-5/2 kernel, sig2 = 1, lengthscale 2.5 grid steps of the last axis,
jitter 1e-3; B = 16 right-hand sides; fp32 and fp64.

Per shape it reports the median over `--runs` calls after a warm-up:
  * set-up on a fresh plan: plan creation and hipgp_plan_set_first_row (`setup_ms`), and the same followed by the first
    one-row R^T, which builds the wide spectrum (`setup_with_wide_ms`); host clock around work that ends in a device
    synchronise;
  * the K and R^T matvecs (CUDA events), with the per-pass split of `hipgp_plan_profile` (class rows_fwd = forward of the last
    axis, cols_pass = the column pass of the leading axis with the spectrum, rows_inv = inverse of the last axis);
  * the same K written with torch.fft.rfftn / irfftn (cuFFT) at the plan's narrow embedding lengths, on the same GPU in the
    same run;
  * PCG with a fixed 20 iterations (tol -1, so the stopping test never passes);
  * fp32 only: compute_kn at B = 200 (PCG with maxiter 10 at tol 1e-8, then R^T).
Then R^T per inducing point at (2731, 2731), the largest square grid whose wide embedding keeps the row pass, against
(2732, 2732), the smallest that takes the four-step path (fp32 and fp64, B = 16).  The card's name and power limit are read in
the same run.  Prints one JSON line per measurement; `--out` also writes them as one JSON document."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from hipgp_b200 import _lib as L  # noqa: E402
from hipgp_b200 import kernels as hk  # noqa: E402
from hipgp_b200.plan import Plan  # noqa: E402

DEV = "cuda:0"


def median_ms(fn, runs, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(runs):
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    return float(np.median(ts))


def median_host_ms(fn, runs):
    """host clock around fn() + a device synchronise; fn returns what must stay alive until the clock stops"""
    ts = []
    for _ in range(runs):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        keep = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
        del keep
    return float(np.median(ts))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "not available"}


def first_row(dims, dt):
    xg = [torch.linspace(0, (m - 1) / (dims[-1] - 1), m, dtype=dt, device=DEV) for m in dims]
    return xg, hk.first_row(xg, hk.Matern(nu=2.5, dtype=dt), (1.0, 2.5 / (dims[-1] - 1)), jitter=1e-3)


def profile_split(plan, fn, runs):
    """per-class device time of one call (the mean over `runs` calls), in ms"""
    fn(); torch.cuda.synchronize()
    plan.profile(True); plan.profile_read(reset=True)
    for _ in range(runs):
        fn()
    torch.cuda.synchronize()
    out = plan.profile_read(reset=True)
    plan.profile(False)
    return {k: {"ms": ms / runs, "launches": n // runs} for k, (ms, n) in out.items() if n}


def shape_row(dims, dname, dt, B, runs):
    M = int(np.prod(dims))
    _, col = first_row(dims, dt)
    plan = Plan(list(dims), dt, DEV).set_first_row(col)
    Ln, Lw = plan.embedding()
    one = torch.randn(1, M, dtype=dt, device=DEV)
    r = {"dtype": dname, "dims": list(dims), "B": B, "Ln": Ln, "Lw": Lw, "runs": runs}
    r["setup_ms"] = median_host_ms(lambda: Plan(list(dims), dt, DEV).set_first_row(col), max(3, runs // 4))
    r["setup_with_wide_ms"] = median_host_ms(lambda: (lambda p: (p, p.matvec(L.MV_RT, one)))(Plan(list(dims), dt, DEV).set_first_row(col)),
                                             max(3, runs // 4))
    g = torch.Generator(device=DEV); g.manual_seed(B)
    v = torch.randn(B, M, dtype=dt, device=DEV, generator=g)
    r["K_ms"] = median_ms(lambda: plan.matvec(L.MV_K, v), runs)
    r["K_split"] = profile_split(plan, lambda: plan.matvec(L.MV_K, v), runs)
    r["RT_ms"] = median_ms(lambda: plan.matvec(L.MV_RT, v), runs)
    r["RT_split"] = profile_split(plan, lambda: plan.matvec(L.MV_RT, v), runs)
    # the same K with cuFFT: real 2-D FFT of the zero-padded grids at the plan's narrow lengths, times the embedding's spectrum
    h = torch.zeros(Ln, dtype=dt, device=DEV)
    c = col.reshape(dims)
    for s0 in (0, 1):
        for s1 in (0, 1):
            blk = c
            if s0: blk = blk[1:].flip(0)
            if s1: blk = blk[:, 1:].flip(1)
            i0 = slice(0, dims[0]) if not s0 else slice(Ln[0] - dims[0] + 1, Ln[0])
            i1 = slice(0, dims[1]) if not s1 else slice(Ln[1] - dims[1] + 1, Ln[1])
            h[i0, i1] = blk
    spec = torch.fft.rfftn(h).real
    vv = v.reshape((B,) + tuple(dims))
    r["K_cufft_ms"] = median_ms(lambda: torch.fft.irfftn(torch.fft.rfftn(vv, s=Ln, dim=(1, 2)) * spec, s=Ln, dim=(1, 2))[:, :dims[0], :dims[1]], runs)
    assert plan.pcg(v, maxiter=20, tol=-1.0, return_info=True)[1]["iters"] == 20
    r["pcg20_fixed_ms"] = median_ms(lambda: plan.pcg(v, maxiter=20, tol=-1.0), max(3, runs // 4), warm=1)
    del v, spec, h, vv
    torch.cuda.empty_cache()
    if dt == torch.float32:
        g.manual_seed(200)
        knm = torch.randn(200, M, dtype=dt, device=DEV, generator=g)
        r["compute_kn_B200_ms"] = median_ms(lambda: plan.compute_kn(knm, maxiter=10, tol=1e-8), max(3, runs // 4), warm=1)
        del knm
    del plan
    torch.cuda.empty_cache()
    return r


def switch_row(m, dname, dt, B, runs):
    dims = (m, m)
    _, col = first_row(dims, dt)
    plan = Plan(list(dims), dt, DEV).set_first_row(col)
    g = torch.Generator(device=DEV); g.manual_seed(m)
    v = torch.randn(B, m * m, dtype=dt, device=DEV, generator=g)
    plan.matvec(L.MV_RT, v)
    n0 = plan.launch_count(); plan.matvec(L.MV_RT, v)
    r = {"dtype": dname, "dims": list(dims), "B": B, "Lw": plan.embedding()[1], "RT_launches": plan.launch_count() - n0}
    r["RT_ms"] = median_ms(lambda: plan.matvec(L.MV_RT, v), runs)
    r["RT_ns_per_point"] = r["RT_ms"] * 1e6 / (B * m * m)
    del plan, v
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--B", type=int, default=16)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("long_rows_time.py times the GPU; no CUDA device here")
    results = [card()]
    print(json.dumps(results[0]), flush=True)
    for dname, dt in (("fp32", torch.float32), ("fp64", torch.float64)):
        for dims in ((3000, 3000), (64, 20000)):
            results.append(shape_row(dims, dname, dt, a.B, a.runs))
            print(json.dumps(results[-1]), flush=True)
        for m in (2731, 2732):
            results.append(switch_row(m, dname, dt, a.B, a.runs))
            print(json.dumps(results[-1]), flush=True)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
