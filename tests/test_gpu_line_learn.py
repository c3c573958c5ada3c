"""learn_kernel=True / learn_noise=True with line-integral observations (integrated_obs=True, the dust-map configuration): the
hyper-parameter gradients of the two line-integral grams that the reference trains through autograd (kernels.py:85-90,223-237
and 199-218):

  K_xu, analytic SqExp line integral   hipgp_kxu_param_grad, mode SEMI_ANALYTIC  (closed form, reduced on the fly)
  K_nn, doubly integrated diagonal     hipgp_doubly_diag_param_grad              (the interpolation table's derivative)

Checkers: fp64 CPU autograd through the oracle's formulas (kernel level) and through the oracle's mean-field and block ELBOs
with the solve as the reference's InvMatmul node (end to end; DESIGN.md section 1 says why plain autograd through the PCG
iterations is the wrong checker for grids of more than one dimension)."""
from unittest import mock

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DT = {"f32": torch.float32, "f64": torch.float64}
HYPER_TOL = {"f64": 1e-6, "f32": 5e-2}          # the tolerances of test_gpu_learn_kernel.py
ELBO_TOL = {"f64": 1e-8, "f32": 2e-3}
SAMPS = 7                                       # stratified offsets of the mc-biased estimator


def relerr(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    a = a.astype(np.float64); b = b.astype(np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def close(got, want, tol):
    return abs(float(got) - float(want)) <= tol * max(abs(float(want)), 1e-3)


# ---- kernel level -------------------------------------------------------------------------------------------------------
def line_inputs(dtype):
    """a 7 x 6 x 5 grid box and 6 rays from the origin to points inside it, rounded to `dtype`"""
    gen = torch.Generator().manual_seed(12)
    xg = [torch.linspace(0.1, 1.0, 7), torch.linspace(-0.5, 0.5, 6), torch.linspace(0.2, 0.8, 5)]
    xg = [g.to(dtype).double() for g in xg]
    lo = torch.tensor([0.1, -0.5, 0.2], dtype=torch.float64); hi = torch.tensor([1.0, 0.5, 0.8], dtype=torch.float64)
    x = (lo + (hi - lo) * torch.rand(6, 3, dtype=torch.float64, generator=gen)).to(dtype).double()
    G = torch.randn(6, 7 * 6 * 5, dtype=torch.float64, generator=gen).to(dtype).double()
    return xg, x, G


@pytest.mark.parametrize("dname", ["f64", "f32"])
@pytest.mark.parametrize("ell0", [0.3, (0.3, 0.5, 0.9)], ids=["scalar", "per_axis"])
def test_analytic_kxu_gradient_vs_oracle_autograd(dname, ell0):
    """SqExp.k_semi_grid (the grid, as _make_grams calls it) and SqExp.k_semi (an explicit point set) under autograd against fp64
    autograd through oracle.sqexp_k_semi.  The derivative is evaluated and reduced in fp64 whatever the input dtype, so with fp64
    hyper-parameter leaves (no rounding of the returned gradient) fp32 inputs meet the fp64 bound (1e-10) against fp64 autograd
    on the same rounded inputs and the same rounded upstream gradient."""
    from hipgp_b200 import kernels as hk
    from oracle import ziggy_oracle as zo
    dtype = DT[dname]
    xg, x, G = line_inputs(dtype)
    xi = zo.meshgrid_points(xg)
    kern = hk.SqExp(dtype=dtype)
    ell_c = torch.tensor(ell0, dtype=torch.float64)
    s_c = torch.tensor(1.3, dtype=torch.float64, requires_grad=True); e_c = ell_c.clone().requires_grad_(True)
    Kc = zo.sqexp_k_semi(xi, x, s_c, e_c, torch.float64)                          # (M, n)
    (Kc * G.t()).sum().backward()
    for shape in ("grid", "points"):
        s_d = torch.tensor(1.3, dtype=torch.float64, device=DEV, requires_grad=True); e_d = ell_c.to(DEV).requires_grad_(True)
        if shape == "grid":
            K = kern.k_semi_grid([g.to(DEV, dtype) for g in xg], x.to(DEV, dtype), (s_d, e_d))      # (n, M)
            (K * G.to(DEV, dtype)).sum().backward()
        else:
            K = kern.k_semi(xi.to(DEV, dtype), x.to(DEV, dtype), (s_d, e_d)).t()                   # (M, n) -> (n, M)
            (K * G.to(DEV, dtype)).sum().backward()
        assert relerr(K, Kc.t()) < (1e-12 if dname == "f64" else 2e-4), shape      # fp32 forward: fp32 exp / erf
        assert abs(float(s_d.grad) - float(s_c.grad)) <= 1e-10 * abs(float(s_c.grad)), (shape, float(s_d.grad), float(s_c.grad))
        assert relerr(e_d.grad, e_c.grad) < 1e-10, (shape, e_d.grad, e_c.grad)


@pytest.mark.parametrize("dname", ["f64", "f32"])
@pytest.mark.parametrize("kname", ["sqexp", "matern32"])
def test_doubly_diag_gradient_vs_oracle_autograd(dname, kname):
    """k_doubly_diag under autograd against fp64 autograd through oracle.doubly_diag_interp with the kernel's own table; |x| / ell
    runs from 0.05 to 6.5, over every table interval and past dmax = 5 (the last slope's extrapolation).  fp32: the distance and
    the table lookup are evaluated in fp32 as in the forward."""
    from hipgp_b200 import kernels as hk
    from oracle import ziggy_oracle as zo
    dtype = DT[dname]
    kern = hk.SqExp(dtype=dtype) if kname == "sqexp" else hk.Matern(nu=1.5, dtype=dtype)
    di = kern.diag_interp
    table = [t.double() for t in (di.distance_grid, di.slopes, di.knn)]
    gen = torch.Generator().manual_seed(13)
    ell, sig2 = 0.2, 1.3
    r = torch.linspace(0.05, 6.5, 600, dtype=torch.float64) * ell
    d = torch.randn(600, 3, dtype=torch.float64, generator=gen)
    x = (d / d.norm(dim=1, keepdim=True) * r[:, None]).to(dtype).double()
    g = torch.randn(600, dtype=torch.float64, generator=gen).to(dtype).double()
    assert (r / ell > 5.0).sum() > 50
    s_c = torch.tensor(sig2, dtype=torch.float64, requires_grad=True); e_c = torch.tensor(ell, dtype=torch.float64, requires_grad=True)
    out_c = zo.doubly_diag_interp(x, s_c, e_c, *table)
    (out_c * g).sum().backward()
    s_d = torch.tensor(sig2, dtype=dtype, device=DEV, requires_grad=True); e_d = torch.tensor(ell, dtype=dtype, device=DEV, requires_grad=True)
    out = kern.k_doubly_diag(x.to(DEV, dtype), (s_d, e_d))
    (out * g.to(DEV, dtype)).sum().backward()
    tol = 1e-12 if dname == "f64" else 1e-5
    assert relerr(out, out_c) < tol
    assert close(s_d.grad, s_c.grad, tol), (float(s_d.grad), float(s_c.grad))
    assert close(e_d.grad, e_c.grad, tol), (float(e_d.grad), float(e_c.grad))
    # the untraced call returns the same values
    with torch.no_grad():
        assert torch.equal(kern.k_doubly_diag(x.to(DEV, dtype), (s_d, e_d)), out.detach())


# ---- end to end --------------------------------------------------------------------------------------------------------
class _RefInvMatmul(torch.autograd.Function):
    """the reference's InvMatmul (_inv_matmul.py:8-64) on the oracle's Toeplitz operator: PCG in forward; backward = the left
    solves and, for the column, the reference's quadratic form over the FLATTENED M-vectors (oracle.inv_matmul_backward,
    gpt_toeplitz.py:169-209).  For D > 1 that form is not the derivative of the block-Toeplitz solve, so plain autograd
    through the PCG iterations differs from the reference; this node keeps the checker on the reference's own route."""

    @staticmethod
    def forward(ctx, column, rhs, xgrids, maxiter, tol):
        from oracle import ziggy_oracle as zo
        ora = zo.OracleToeplitz(xgrids, lambda a, b: column.detach().reshape(1, -1), jitter_val=None)
        x = ora.solve(rhs.detach(), maxiter=maxiter, tol=tol)
        ctx.ora, ctx.cg = ora, (maxiter, tol)
        ctx.save_for_backward(x)
        return x

    @staticmethod
    def backward(ctx, grad_output):
        from oracle import ziggy_oracle as zo
        (x,) = ctx.saved_tensors
        lhs = ctx.ora.solve(grad_output.contiguous(), maxiter=ctx.cg[0], tol=ctx.cg[1])
        gcol = torch.from_numpy(zo.inv_matmul_backward(lhs.numpy(), x.numpy()))
        return gcol, lhs, None, None, None


def ref_compute_kn(xgrids, kfun, Knm, maxiter_cg=10, tol=1e-8, jitter_val=1e-3):
    """oracle.compute_kn with the solve as the reference's InvMatmul node (hipgp.py:139-146 under learn_kernel=True)"""
    from oracle import ziggy_oracle as zo
    Kmm = zo.OracleToeplitz(xgrids, kfun, batch_shape=None, jitter_val=jitter_val)
    return Kmm.matmul_RT(_RefInvMatmul.apply(Kmm.column, Knm, xgrids, maxiter_cg, tol))


def spd_blocks(gen, nblk, bs):
    A = torch.randn(nblk, bs, bs, dtype=torch.float64, generator=gen)
    return A @ A.transpose(1, 2) / bs + 0.5 * torch.eye(bs, dtype=torch.float64)


ELL = {"sqexp": 0.12, "matern32": 0.12}          # PCG converges within 60 iterations on both sides


def problem(kname, family="meanfield"):
    """a 10 x 8 x 6 grid (M' = 18 x 14 x 10) and 16 rays from the origin to points inside it"""
    gen = torch.Generator().manual_seed(21)
    xg = [torch.linspace(0.1, 1.0, 10, dtype=torch.float64), torch.linspace(-0.4, 0.4, 8, dtype=torch.float64),
          torch.linspace(0.2, 0.7, 6, dtype=torch.float64)]
    lo = torch.tensor([0.1, -0.4, 0.2], dtype=torch.float64); hi = torch.tensor([1.0, 0.4, 0.7], dtype=torch.float64)
    x = lo + (hi - lo) * torch.rand(16, 3, dtype=torch.float64, generator=gen)
    y = torch.randn(16, 1, dtype=torch.float64, generator=gen)
    nb = 0.3 + 0.2 * torch.rand(16, 1, dtype=torch.float64, generator=gen)
    Mp = 18 * 14 * 10
    theta1 = torch.randn(Mp, 1, dtype=torch.float64, generator=gen)
    if family == "meanfield":
        theta2 = -0.5 / (0.1 + torch.rand(Mp, 1, dtype=torch.float64, generator=gen))
    else:
        theta2 = -0.5 * torch.linalg.inv(spd_blocks(gen, 8, 315))
    return dict(xg=xg, x=x, y=y, nb=nb, theta1=theta1, theta2=theta2, chunks=[9, 7, 5], sig2=1.3, ell=ELL[kname], noise2=0.2,
                nobs=1000, jitter=1e-3)


def make_model(p, kname, dtype, learn_kernel, learn_noise, family="meanfield"):
    from hipgp_b200 import kernels as hk
    from hipgp_b200.hipgp import BlockToeplitzGP, MeanFieldToeplitzGP
    kern = hk.SqExp(dtype=dtype) if kname == "sqexp" else hk.Matern(nu=1.5, dtype=dtype)
    kw = dict(num_obs=p["nobs"], sig2_init=p["sig2"], ell_init=p["ell"], noise2_init=p["noise2"], dtype=dtype, jitter_val=p["jitter"],
              learn_kernel=learn_kernel, learn_noise=learn_noise)
    xg = [g.to(dtype) for g in p["xg"]]
    mod = MeanFieldToeplitzGP(kern, xg, **kw) if family == "meanfield" else BlockToeplitzGP(kern, xg, block_sizes=p["chunks"], **kw)
    mod.global_theta1.data.copy_(p["theta1"].to(dtype)); mod.global_theta2.data.copy_(p["theta2"].to(dtype))
    return mod.cuda_params(0)


def oracle_grads(p, kname, estimator, learn_noise, table, alphas=None, family="meanfield", maxiter_cg=60):
    """fp64 CPU autograd of -ELBO through the oracle's ELBO with Knm the line-integral gram (analytic or Monte-Carlo with the
    given offsets), Knn the interpolated doubly integrated diagonal, k_n on the reference's route (`ref_compute_kn`) and sig2,
    ell and the noise variance as leaves; returns the ELBO and the gradients with respect to their logarithms"""
    from oracle import ziggy_oracle as zo
    sig2 = torch.tensor(p["sig2"], dtype=torch.float64, requires_grad=True)
    ell = torch.tensor(p["ell"], dtype=torch.float64, requires_grad=True)
    noise2 = torch.tensor(p["noise2"], dtype=torch.float64, requires_grad=True)
    if kname == "sqexp":
        kfun = lambda a, b: zo.sqexp(a, b, sig2, ell)
    else:
        kfun = lambda a, b: zo.matern(a, b, sig2, ell, 1.5)
    xi = zo.meshgrid_points(p["xg"])
    if estimator == "analytic":
        Knm = zo.sqexp_k_semi(xi, p["x"], sig2, ell, torch.float64).t()
    else:
        Knm = zo.k_semi_mc(kfun, xi, p["x"], alphas).t()
    Knn = zo.doubly_diag_interp(p["x"], sig2, ell, *table)
    nb = torch.sqrt(noise2) * torch.ones_like(p["nb"]) if learn_noise else p["nb"]
    with mock.patch.object(zo, "compute_kn", ref_compute_kn):
        if family == "meanfield":
            elbo = zo.meanfield_elbo_and_grad(p["xg"], kfun, Knm, Knn, p["y"], nb, p["theta1"], p["theta2"], p["nobs"],
                                              maxiter_cg=maxiter_cg, jitter_val=p["jitter"])[0]
        else:
            blk_idx = zo.define_block_chunks([2 * len(g) - 2 for g in p["xg"]], p["chunks"])
            elbo = zo.block_elbo_and_grad(p["xg"], kfun, blk_idx, Knm, Knn, p["y"], nb, p["theta1"], p["theta2"], p["nobs"],
                                          maxiter_cg=maxiter_cg, jitter_val=p["jitter"])[0]
    (-elbo).backward()                          # as the model's training step does (svi_gp.py:317-329)
    out = {"elbo": float(elbo.detach()), "g_log_sig2": float(sig2.grad) * p["sig2"], "g_log_ell": float(ell.grad) * p["ell"]}
    if learn_noise:
        out["g_log_noise2"] = float(noise2.grad) * p["noise2"]
    return out


def table_of(mod):
    di = mod.kernel.diag_interp
    return [t.double().cpu() for t in (di.distance_grid, di.slopes, di.knn)]


@pytest.mark.parametrize("dname", ["f64", "f32"])
@pytest.mark.parametrize("kname,estimator,learn_noise", [("sqexp", "analytic", False), ("sqexp", "analytic", True),
                                                         ("sqexp", "mc-biased", False), ("matern32", "mc-biased", False)])
def test_line_integral_hyperparameter_gradients_vs_oracle_autograd(kname, estimator, learn_noise, dname):
    p = problem(kname)
    dtype = DT[dname]
    mod = make_model(p, kname, dtype, True, learn_noise)
    alphas = None
    if estimator == "mc-biased":
        # the model draws its offsets from the CUDA generator (kernels.mc_alphas); draw the same ones for the oracle
        from hipgp_b200 import kernels as hk
        torch.cuda.manual_seed(77)
        alphas = hk.mc_alphas(SAMPS, dtype, DEV).double().cpu()
    want = oracle_grads(p, kname, estimator, learn_noise, table_of(mod), alphas)
    x, y = p["x"].to(DEV, dtype), p["y"].to(DEV, dtype)
    nb = None if learn_noise else p["nb"].to(DEV, dtype)
    run = dict(maxiter_cg=60, integrated_obs=True, semi_integrated_estimator=estimator, semi_integrated_samps=SAMPS)
    torch.cuda.manual_seed(77)
    elbo = mod.elbo_and_grad(x, y, nb, **run)
    assert elbo.requires_grad
    (-elbo).backward()
    tol = HYPER_TOL[dname]
    assert close(elbo, want["elbo"], ELBO_TOL[dname]), (float(elbo), want["elbo"])
    got = {"g_log_sig2": mod.log_sig2.grad, "g_log_ell": mod.log_ell.grad}
    if learn_noise:
        got["g_log_noise2"] = mod.log_noise2.grad
    for name, g in got.items():
        assert g is not None and close(g, want[name], tol), (name, float(g), want[name])
    # the natural gradients of the variational parameters do not depend on whether the hyper-parameters are traced
    ref = make_model(p, kname, dtype, False, False)
    torch.cuda.manual_seed(77)
    ref.elbo_and_grad(x, y, None if learn_noise else nb, **run)
    lim = 1e-8 if dname == "f64" else 2e-3
    assert relerr(mod.global_theta1.grad, ref.global_theta1.grad) < lim
    assert relerr(mod.global_theta2.grad, ref.global_theta2.grad) < lim
    # one Adam step on the hyper-parameters (svi_gp.py:254-262,327-329) moves both
    opt = torch.optim.Adam([mod.log_ell, mod.log_sig2], lr=1e-2)
    before = (float(mod.log_ell), float(mod.log_sig2))
    opt.step()
    assert float(mod.log_ell) != before[0] and float(mod.log_sig2) != before[1]


@pytest.mark.parametrize("dname", ["f64", "f32"])
def test_block_family_analytic_line_integrals_vs_oracle_autograd(dname):
    """BlockToeplitzGP (9 x 7 x 5 chunks of M' = 18 x 14 x 10: 8 blocks of 315) against the oracle's block ELBO on the same route"""
    p = problem("sqexp", family="block")
    dtype = DT[dname]
    mod = make_model(p, "sqexp", dtype, True, False, family="block")
    want = oracle_grads(p, "sqexp", "analytic", False, table_of(mod), family="block")
    x, y, nb = p["x"].to(DEV, dtype), p["y"].to(DEV, dtype), p["nb"].to(DEV, dtype)
    elbo = mod.elbo_and_grad(x, y, nb, maxiter_cg=60, integrated_obs=True, semi_integrated_estimator="analytic")
    (-elbo).backward()
    assert close(elbo, want["elbo"], ELBO_TOL[dname]), (float(elbo), want["elbo"])
    for name, par in (("g_log_sig2", mod.log_sig2), ("g_log_ell", mod.log_ell)):
        assert par.grad is not None and close(par.grad, want[name], HYPER_TOL[dname]), (name, float(par.grad), want[name])


# ---- refusals ----------------------------------------------------------------------------------------------------------
def test_refusals():
    from hipgp_b200 import kernels as hk
    from hipgp_b200.hipgp import MeanFieldToeplitzGP
    dtype = torch.float64
    xg = [torch.linspace(0.1, 1.0, 6, dtype=dtype), torch.linspace(-0.4, 0.4, 5, dtype=dtype)]
    x = torch.tensor([[0.5, 0.1], [0.8, -0.2]], dtype=dtype, device=DEV)
    # Gneiting: no closed-form hyper-parameter derivative
    mod = MeanFieldToeplitzGP(hk.Gneiting(dtype=dtype), xg, num_obs=10, sig2_init=1.0, ell_init=0.3, dtype=dtype,
                              learn_kernel=True).cuda_params(0)
    with pytest.raises(NotImplementedError, match="not for this kernel"):
        mod.elbo_and_grad(x, torch.zeros(2, 1, dtype=dtype, device=DEV), torch.ones(2, 1, dtype=dtype, device=DEV))
    # the doubly integrated diagonal with a per-axis ell and a gradient request
    s = torch.tensor(1.0, dtype=dtype, device=DEV, requires_grad=True)
    e = torch.tensor([0.3, 0.4], dtype=dtype, device=DEV, requires_grad=True)
    with pytest.raises(NotImplementedError, match="scalar ell"):
        hk.SqExp(dtype=dtype).k_doubly_diag(x, (s, e))
