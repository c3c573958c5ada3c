"""Times hyper-parameter learning with line-integral observations at the BASELINE config 4 shape (128x128x64 grid, SqExp,
analytic line integrals from the origin, batch 200, fp32; the doubly integrated diagonal's table fixed as in
scripts/bench_svi.py so that no host quadrature runs).  Prints JSON lines:

  * hipgp_kxu_param_grad in mode SEMI_ANALYTIC (the backward of K_xu) beside the forward hipgp_kxu at the same shape;
  * one traced MeanFieldToeplitzGP step (learn_kernel=True: elbo_and_grad + (-elbo).backward()) beside the untraced step.

Each figure is CUDA-event time over a window of about one second after a warm-up; K_xu and its upstream gradient (839 MB each)
are larger than L2.  The card's name and power limit are read in the same run."""
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from hipgp_b200 import _lib as L  # noqa: E402
from hipgp_b200 import kernels as hk  # noqa: E402
from hipgp_b200.hipgp import MeanFieldToeplitzGP  # noqa: E402

DEV = "cuda:0"


def timeit(fn, window_s=1.0, warm=3):
    """mean ms per call over a window of about `window_s` seconds"""
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    n = max(3, int(window_s * 1e3 / max(e0.elapsed_time(e1), 1e-3)))
    e0.record()
    for _ in range(n):
        fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n, n


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else "not available"}


def main():
    if not torch.cuda.is_available():
        raise SystemExit("line_learn_time.py times the GPU; no CUDA device here")
    print(json.dumps(card()), flush=True)
    dt = torch.float32
    B = 200
    sig2, ell = 0.1, 0.01
    dims = [128, 128, 64]
    xgrids = [torch.linspace(-.25, .25, 128, dtype=dt), torch.linspace(-.25, .25, 128, dtype=dt), torch.linspace(-.05, .05, 64, dtype=dt)]
    rs = np.random.RandomState(42)
    x = torch.from_numpy(np.stack([rs.uniform(-.25, .25, B), rs.uniform(-.25, .25, B), rs.uniform(-.05, .05, B)], 1)).to(DEV, dt)
    y = torch.from_numpy(rs.uniform(5e-4, 3.2e-2, (B, 1))).to(DEV, dt)
    nb = torch.from_numpy(rs.uniform(0.0025, 0.0075, (B, 1))).to(DEV, dt)

    # (a) the K_xu backward against its forward, both through the C entry points
    lib = L.load()
    M = int(np.prod(dims))
    grids = torch.cat([g.to(DEV) for g in xgrids]).contiguous()
    marr = (C.c_int64 * 3)(*dims)
    ellv = (C.c_double * 1)(ell)
    out = torch.empty(B, M, device=DEV, dtype=dt)
    G = torch.randn(B, M, device=DEV, dtype=dt)
    partial = torch.empty(B, (M + 1023) // 1024, 4, device=DEV, dtype=torch.float64)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)

    def fwd():
        L.check(lib, lib.hipgp_kxu(L.F32, L.K_SQEXP, L.KXU_SEMI_ANALYTIC, sig2, ellv, 1, 1.0, C.c_void_p(x.data_ptr()), B, 3, marr,
                                   C.c_void_p(grids.data_ptr()), None, 0, C.c_void_p(out.data_ptr()), stream))

    def bwd():
        L.check(lib, lib.hipgp_kxu_param_grad(L.F32, L.K_SQEXP, L.KXU_SEMI_ANALYTIC, sig2, ellv, 1, C.c_void_p(x.data_ptr()), B, 3, marr,
                                              C.c_void_p(grids.data_ptr()), None, 0, None, 0, C.c_void_p(G.data_ptr()),
                                              C.c_void_p(partial.data_ptr()), stream))
    t_f, n_f = timeit(fwd)
    t_b, n_b = timeit(bwd)
    print(json.dumps({"grid": dims, "batch": B, "dtype": "fp32", "kernel": "sqexp", "mode": "analytic",
                      "kxu_forward_ms": t_f, "kxu_forward_calls": n_f, "kxu_param_grad_ms": t_b, "kxu_param_grad_calls": n_b}), flush=True)
    del out, G, partial
    torch.cuda.empty_cache()

    # (b) one minibatch step with and without the hyper-parameters on the tape
    tab = np.stack([np.linspace(0, 5, 50), np.zeros(50), np.linspace(1, 0.1, 50)])
    for mode, learn in (("untraced", False), ("traced learn_kernel", True)):
        kern = hk.SqExp(dtype=dt)
        kern._diag_interp = hk.KernelDoublyDiagInterpolator(kern, table=tab)
        mod = MeanFieldToeplitzGP(kern, xgrids, num_obs=5_000_000, sig2_init=sig2, ell_init=ell, dtype=dt, jitter_val=1e-3,
                                  learn_kernel=learn).cuda_params(0)

        def step():
            mod.zero_grad(set_to_none=True)
            elbo = mod.elbo_and_grad(x, y, nb, maxiter_cg=20, integrated_obs=True, semi_integrated_estimator="analytic")
            if elbo.requires_grad:
                (-elbo).backward()
        t, n = timeit(step, warm=2)
        print(json.dumps({"family": "mean-field", "mode": mode, "svi_step_ms": t, "steps": n, "grid": dims, "batch": B,
                          "dtype": "fp32", "integrated_obs": "analytic", "maxiter_cg": 20}), flush=True)
        del mod
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
