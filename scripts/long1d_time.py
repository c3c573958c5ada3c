"""Times the four-step path of long 1-D grids (long1d_kernels.cuh) at M = 1e4, 1e5, 1e6 inducing points: Matern-5/2 kernel,
sig2 = 1, lengthscale 2.5 grid steps, jitter 1e-3; B = 1 and 200 right-hand sides; fp32 and fp64.

Per shape it reports the median over `--runs` calls after a warm-up:
  * set-up, on a fresh plan (`setup_fresh_ms`: plan creation and the first hipgp_plan_set_first_row, which also builds the
    four-step tables and the Bluestein chirp spectrum; host clock around work that ends in a device synchronise) and
    repeated on a plan that already has them (`setup_repeat_ms`, CUDA events: Bluestein DCT-I x 3 and the narrow spectra);
    each also followed by the first one-row R^T, which builds the wide spectrum (one more DCT-I and the wide forward);
  * the K and R^T matvecs, with algorithmic bytes w (2 M B + E_h) and w ((M + E) B + E_h) (E_h = M real half-spectrum
    entries, E = 2M - 2) and their share of the 7.7 TB/s HBM3e data-sheet figure;
  * the same K operator written with torch.fft.rfft / irfft (cuFFT) at the plan's length, on the same GPU in the same run;
  * PCG with maxiter 20 at tol 1e-8 as a caller would run it (it may converge earlier: `pcg20_tol_iters` is the number of
    iterations it ran), and a fixed 20 iterations (tol -1, so the stopping test never passes), whose time per iteration
    gives the bandwidth against w (13 M B + 2 E_h) bytes per iteration;
  * at B = 200, the reference harness shape: a fixed 200-iteration PCG followed by R^T.
The working sets at M = 1e4 and at B = 1 fit the 126 MB L2; the B = 200 shapes at M >= 1e5 do not.  The card's name and power
limit are read in the same run.  Prints one JSON line per shape; `--out` also writes them as one JSON document."""
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
HBM = 7.7e12


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


def bw(nbytes, ms):
    return {"GBps": nbytes / ms / 1e6, "share_of_hbm_peak": nbytes / (ms * 1e-3) / HBM}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=20)
    ap.add_argument("--sizes", default="10000,100000,1000000")
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("long1d_time.py times the GPU; no CUDA device here")
    results = [card()]
    print(json.dumps(results[0]), flush=True)
    for dname, dt in (("fp32", torch.float32), ("fp64", torch.float64)):
        w = 4 if dt == torch.float32 else 8
        for M in (int(s) for s in a.sizes.split(",")):
            x = torch.linspace(0, 1, M, dtype=dt, device=DEV)
            col = hk.first_row([x], hk.Matern(nu=2.5, dtype=dt), (1.0, 2.5 / (M - 1)), jitter=1e-3)
            plan = Plan([M], dt, DEV).set_first_row(col)
            Ln, Lw = plan.embedding()[0][0], plan.embedding()[1][0]
            E = 2 * M - 2
            one = torch.randn(1, M, dtype=dt, device=DEV)
            setup_fresh = median_host_ms(lambda: Plan([M], dt, DEV).set_first_row(col), a.runs)
            setup_fresh_wide = median_host_ms(lambda: (lambda p: (p, p.matvec(L.MV_RT, one)))(Plan([M], dt, DEV).set_first_row(col)), a.runs)
            setup = median_ms(lambda: plan.set_first_row(col), a.runs)
            setup_wide = median_ms(lambda: (plan.set_first_row(col), plan.matvec(L.MV_RT, one)), a.runs)
            # the same K with cuFFT: real FFT of the zero-padded rows at the plan's length, times the (unclamped) spectrum
            h = torch.zeros(Ln, dtype=dt, device=DEV); h[:M] = col; h[Ln - M + 1:] = col[1:].flip(0)
            spec = torch.fft.rfft(h).real
            for B in (1, 200):
                g = torch.Generator(device=DEV); g.manual_seed(B)
                v = torch.randn(B, M, dtype=dt, device=DEV, generator=g)
                r = {"dtype": dname, "M": M, "B": B, "Ln": Ln, "Lw": Lw, "runs": a.runs,
                     "setup_fresh_ms": setup_fresh, "setup_fresh_with_wide_ms": setup_fresh_wide,
                     "setup_repeat_ms": setup, "setup_repeat_with_wide_ms": setup_wide}
                t = median_ms(lambda: plan.matvec(L.MV_K, v), a.runs)
                r["K_ms"] = t; r["K_bw"] = bw(w * (2 * M * B + M), t)
                t = median_ms(lambda: plan.matvec(L.MV_RT, v), a.runs)
                r["RT_ms"] = t; r["RT_bw"] = bw(w * ((M + E) * B + M), t)
                t = median_ms(lambda: torch.fft.irfft(torch.fft.rfft(v, n=Ln) * spec, n=Ln)[:, :M], a.runs)
                r["K_cufft_ms"] = t; r["K_cufft_bw"] = bw(w * (2 * M * B + M), t)
                r["pcg20_tol_ms"] = median_ms(lambda: plan.pcg(v, maxiter=20, tol=1e-8), a.runs)
                r["pcg20_tol_iters"] = plan.pcg(v, maxiter=20, tol=1e-8, return_info=True)[1]["iters"]
                assert plan.pcg(v, maxiter=20, tol=-1.0, return_info=True)[1]["iters"] == 20
                t = median_ms(lambda: plan.pcg(v, maxiter=20, tol=-1.0), a.runs)
                r["pcg20_fixed_ms"] = t; r["pcg_iter_bw"] = bw(w * (13 * M * B + 2 * M), t / 20)
                if B == 200:
                    t = median_ms(lambda: plan.matvec(L.MV_RT, plan.pcg(v, maxiter=200, tol=-1.0)), a.runs, warm=1)
                    r["harness_pcg200_rt_ms"] = t
                print(json.dumps(r), flush=True)
                results.append(r)
                del v
                torch.cuda.empty_cache()
            del plan, spec, h
            torch.cuda.empty_cache()
    if a.out:
        with open(a.out, "w") as f:
            json.dump(results, f, indent=1)


if __name__ == "__main__":
    main()
