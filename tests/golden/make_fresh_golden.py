"""Writes tests/golden/fresh_oracle_vs_reference.npz: the inputs and the compared outputs of the fresh-input cases of
tests/test_oracle_vs_reference.py (three grids x two dtypes, 3 right-hand sides each, and one mean-field natural-gradient
step), so that the comparison runs on every checkout and not only where the reference tree is present.

    python tests/golden/make_fresh_golden.py      (reference checkout located as in oracle/make_ref.py)

The outputs come from the unmodified reference (ToeplitzTensor, toeplitz_expanded.gram_solve, the mean-field step of
ziggy/hipgp.py:194-276) when oracle/ref_shim.py finds a reference tree.  Without one they come from the CPU oracle; the live
test asserts that the oracle equals the reference bit for bit on these cases (1e-12 relative for the mean-field step),
so both sources give the same file wherever that test passes.  The file's `source` entry records which one wrote it.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import ref_shim  # noqa: E402
from oracle import ziggy_oracle as zo  # noqa: E402

OUT = os.path.join(HERE, "fresh_oracle_vs_reference.npz")
DT = {"f32": torch.float32, "f64": torch.float64}
# (dims, nu, ell): the grid of axis d is linspace(-1 - d, 2 + d / 2, m); sig2 = 1.3, jitter 2e-3
CASES = (((19, 23), 1.5, 0.4), ((7, 5, 9), 2.5, 0.6), ((31,), 0.5, 0.2))
MF_GRIDS = ((-2.0, 1.0, 9), (10.0, 12.5, 12))


def case_tag(dname, dims):
    return "%s_%s" % (dname, "x".join(map(str, dims)))


def grids(dims, dtype):
    return [torch.linspace(-1.0 - d, 2.0 + 0.5 * d, m, dtype=dtype) for d, m in enumerate(dims)]


def main():
    use_ref = ref_shim.reference_root() is not None
    if use_ref:
        ref_shim.import_reference()
        from ziggy.misc.toeplitz_tensor import ToeplitzTensor
        from ziggy.misc import toeplitz_expanded
        from ziggy import kernels as zk, hipgp as zh
    out = {"source": np.array("reference" if use_ref else "oracle")}
    torch.manual_seed(20261018)
    for dname, dtype in DT.items():
        for dims, nu, ell in CASES:
            t = case_tag(dname, dims)
            xg = grids(dims, dtype)
            if use_ref:
                kern = zk.Matern(nu=nu, length_scale=ell, dtype=dtype)
                kfun = lambda x, y: kern.forward(x, y, params=(1.3, ell))
                T = ToeplitzTensor(xgrids=xg, kernel=kfun, batch_shape=None, jitter_val=2e-3)
                E = int(np.prod(T.C.shape))
                mv = (T._matmul_by_K, T._matmul_by_Cinv, T._matmul_by_RT, T._matmul_by_R)
                solve, gram = T._solve, toeplitz_expanded.gram_solve
            else:
                kfun = lambda x, y: zo.matern(x, y, 1.3, ell, nu)
                T = zo.OracleToeplitz(xg, kfun, jitter_val=2e-3)
                E = int(np.prod(T.C.shape))
                mv = (T.matmul_K, T.matmul_Cinv, T.matmul_RT, T.matmul_R)
                solve, gram = T.solve, zo.gram_solve
            M = int(np.prod(dims))
            v = torch.randn(3, M, dtype=dtype); w = torch.randn(3, E, dtype=dtype)
            if use_ref:
                T.set_batch_shape((3,))
            calls = []
            x = solve(v, do_precond=True, maxiter=40, tol=1e-9, callback=lambda n, xx: calls.append(n))
            out.update({t + "_v": v.numpy(), t + "_w": w.numpy(), t + "_column": T.column.numpy(), t + "_D": T.D.numpy(),
                        t + "_Kv": mv[0](v).numpy(), t + "_Cinv_v": mv[1](v).numpy(), t + "_RT_v": mv[2](v).numpy(),
                        t + "_R_w": mv[3](w).numpy(), t + "_solve": x.numpy(), t + "_calls": np.array(calls, dtype=np.int64)})
            if len(dims) > 1:
                out[t + "_gram_rt"] = gram(xg, kfun, v[:1], do_precond=True, tol=1e-9, maxiter=60, mult_RT=True).numpy()
    # one mean-field natural-gradient step (fp64); theta as the model initialises it, with a perturbed theta2
    dtype = torch.float64
    xg = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in MF_GRIDS]
    Mp = int(np.prod([2 * m - 2 for _, _, m in MF_GRIDS]))
    th1 = torch.nn.init.xavier_normal_(torch.zeros(Mp, 1, dtype=dtype))
    th2 = -0.5 / (0.1 + torch.rand(Mp, 1, dtype=dtype))
    lo = torch.tensor([g[0] for g in MF_GRIDS], dtype=dtype); hi = torch.tensor([g[1] for g in MF_GRIDS], dtype=dtype)
    xb = lo + (hi - lo) * torch.rand(6, 2, dtype=dtype); yb = torch.randn(6, 1, dtype=dtype)
    nb = 0.2 + 0.1 * torch.rand(6, 1, dtype=dtype)
    if use_ref:
        kern = zk.Matern(nu=1.5, length_scale=0.6, dtype=dtype)
        mod = zh.MeanFieldToeplitzGP(kern, xg, num_obs=300, sig2_init=0.8, ell_init=0.6, dtype=dtype, jitter_val=1e-3, learn_kernel=False)
        mod.global_theta1.data.copy_(th1); mod.global_theta2.data.copy_(th2)
        elbo = mod.elbo_and_grad(xb, yb, nb, maxiter_cg=15)
        g1, g2 = mod.global_theta1.grad, mod.global_theta2.grad
    else:
        kfun = lambda x, y: zo.matern(x, y, 0.8, 0.6, 1.5)
        Knm = kfun(xb, zo.meshgrid_points(xg)); Knn = torch.full((6,), 0.8, dtype=dtype)
        elbo, g1, g2 = zo.meanfield_elbo_and_grad(xg, kfun, Knm, Knn, yb, nb, th1, th2, 300, maxiter_cg=15, jitter_val=1e-3)
    out.update(mf_theta1=th1.numpy(), mf_theta2=th2.numpy(), mf_x=xb.numpy(), mf_y=yb.numpy(), mf_noise_std=nb.numpy(),
               mf_elbo=np.array(float(elbo)), mf_g1=g1.detach().numpy(), mf_g2=g2.detach().numpy())
    np.savez_compressed(OUT, **out)
    print("wrote", OUT, "from the", str(out["source"]), "size", os.path.getsize(OUT))


if __name__ == "__main__":
    main()
