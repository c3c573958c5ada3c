"""Times hyper-parameter learning in the block-diagonal family at the BASELINE config 3 shape (300x300 grid -> M' = 598^2,
batch 200, 13x13 chunks -> 2116 blocks of 169, fp32).  Prints JSON lines:

  * hipgp_block_quadform_grad (the backward of knSkn) against the torch composition it replaces,
    block_diag_multiply(S + S^T, kn) * g[:, None], with the largest difference between the two;
  * one traced BlockToeplitzGP step (learn_kernel=True: elbo_and_grad + (-elbo).backward()) beside the untraced block step
    and the traced mean-field step.

Each figure is CUDA-event time over a window of about one second after a warm-up; kn (286 MB) and S (242 MB) are larger than
L2.  The card's name and power limit are read in the same run."""
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
from hipgp_b200 import kernels as hk  # noqa: E402
from hipgp_b200.hipgp import BlockToeplitzGP, MeanFieldToeplitzGP  # noqa: E402
from hipgp_b200.plan import block_diag_multiply, block_quadform_grad  # noqa: E402
from hipgp_b200.util import define_block_chunks  # noqa: E402

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
        raise SystemExit("block_learn_time.py times the GPU; no CUDA device here")
    print(json.dumps(card()), flush=True)
    dt = torch.float32
    B = 200
    idx, _, _ = define_block_chunks([torch.arange(598), torch.arange(598)], [13, 13])
    idxd = idx.to(DEV)
    nblk, bs = idx.shape
    gen = torch.Generator(device=DEV); gen.manual_seed(0)
    kn = torch.randn(B, 598 * 598, device=DEV, dtype=dt, generator=gen)
    S = torch.randn(nblk, bs, bs, device=DEV, dtype=dt, generator=gen)
    g = torch.randn(B, device=DEV, dtype=dt, generator=gen)
    fused = block_quadform_grad(S, kn, g, idxd)
    composed = block_diag_multiply(S + S.transpose(1, 2), kn, idxd) * g[:, None]
    diff = float((fused - composed).abs().max() / composed.abs().max())
    t_new, n_new = timeit(lambda: block_quadform_grad(S, kn, g, idxd))
    t_old, n_old = timeit(lambda: block_diag_multiply(S + S.transpose(1, 2), kn, idxd) * g[:, None])
    t_mul, n_mul = timeit(lambda: block_diag_multiply(S, kn, idxd))
    hbm = 4.0 * (kn.numel() * 2 + S.numel())                     # least traffic: read kn and S once, write dkn once
    print(json.dumps({"block": [13, 13], "num_blocks": nblk, "block_size": bs, "batch": B, "dtype": "fp32",
                      "block_quadform_grad_ms": t_new, "calls": n_new,
                      "torch_composition_ms": t_old, "torch_composition_calls": n_old,
                      "block_diag_multiply_ms": t_mul, "block_diag_multiply_calls": n_mul,
                      "block_quadform_grad_min_bytes_GBps": hbm / t_new / 1e6,
                      "max_abs_diff_over_max_abs": diff}), flush=True)
    del kn, S, g, fused, composed
    torch.cuda.empty_cache()

    xgrids = [torch.linspace(0, 1, 300, dtype=dt), torch.linspace(0, 1, 300, dtype=dt)]
    x = torch.rand(B, 2, device=DEV, dtype=dt, generator=gen); y = torch.randn(B, 1, device=DEV, dtype=dt, generator=gen)
    kern = lambda: hk.Matern(nu=1.5, dtype=dt)
    cases = (("block 13x13", "untraced", BlockToeplitzGP(kern(), xgrids, num_obs=10 ** 6, block_sizes=[13, 13], ell_init=0.02, dtype=dt)),
             ("block 13x13", "traced learn_kernel", BlockToeplitzGP(kern(), xgrids, num_obs=10 ** 6, block_sizes=[13, 13], ell_init=0.02,
                                                                    dtype=dt, learn_kernel=True)),
             ("mean-field", "traced learn_kernel", MeanFieldToeplitzGP(kern(), xgrids, num_obs=10 ** 6, ell_init=0.02, dtype=dt,
                                                                       learn_kernel=True)))
    for family, mode, mod in cases:
        mod = mod.cuda_params(0)

        def step():
            mod.zero_grad(set_to_none=True)
            elbo = mod.elbo_and_grad(x, y, maxiter_cg=20)
            if elbo.requires_grad:
                (-elbo).backward()
        t, n = timeit(step, warm=2)
        print(json.dumps({"family": family, "mode": mode, "svi_step_ms": t, "steps": n, "grid": [300, 300], "batch": B,
                          "dtype": "fp32"}), flush=True)
        del mod
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
