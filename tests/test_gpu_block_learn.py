"""learn_kernel=True / learn_noise=True for the block-diagonal family (ziggy/hipgp.py:527-690 trained as in hipgp.py:214-218,
svi_gp.py:317-329): `BlockToeplitzGP.elbo_and_grad` keeps the ELBO estimate on the autograd tape down to log_sig2 / log_ell /
log_noise2, with knSkn_b = kn_b^T blockdiag(S) kn_b through the `_BlockKnSkn` node (hipgp_block_quadform_grad backward).

Checkers: torch autograd through the CPU oracle's block ELBO (oracle.ziggy_oracle.block_elbo_and_grad) in fp64 with the
solve as the reference's InvMatmul node (its flattened 1-D column gradient, which the library reproduces), and the
reference's own mean-field hyper-parameter gradients (tests/golden/learn_kernel_<dtype>.npz), which a block model with 1x1
blocks must reproduce."""
import os
from unittest import mock

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
DT = {"f32": torch.float32, "f64": torch.float64}
HYPER_TOL = {"f64": 1e-6, "f32": 5e-2}          # the tolerances of test_gpu_learn_kernel.py


def relerr(a, b):
    a = a.detach().cpu().numpy() if torch.is_tensor(a) else np.asarray(a)
    b = b.detach().cpu().numpy() if torch.is_tensor(b) else np.asarray(b)
    a = a.astype(np.float64); b = b.astype(np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def close(got, want, tol):
    return abs(float(got) - float(want)) <= tol * max(abs(float(want)), 1e-3)


def spd_blocks(gen, nblk, bs, skew=0.0):
    A = torch.randn(nblk, bs, bs, dtype=torch.float64, generator=gen)
    S = A @ A.transpose(1, 2) / bs + 0.5 * torch.eye(bs, dtype=torch.float64)
    if skew:
        K = torch.randn(nblk, bs, bs, dtype=torch.float64, generator=gen)
        S = S + skew * (K - K.transpose(1, 2))
    return S


def problem():
    """Matern-3/2 on a 12 x 9 grid (M' = 22 x 16), 11 x 4 chunks -> 8 blocks of 44; 16 observations"""
    gen = torch.Generator().manual_seed(4)
    xg = [torch.linspace(0, 1, 12, dtype=torch.float64), torch.linspace(-0.5, 0.5, 9, dtype=torch.float64)]
    x = torch.stack([torch.rand(16, dtype=torch.float64, generator=gen), torch.rand(16, dtype=torch.float64, generator=gen) - 0.5], 1)
    y = torch.randn(16, 1, dtype=torch.float64, generator=gen)
    nb = 0.3 + 0.2 * torch.rand(16, 1, dtype=torch.float64, generator=gen)
    theta1 = torch.randn(22 * 16, 1, dtype=torch.float64, generator=gen)
    theta2 = -0.5 * torch.linalg.inv(spd_blocks(gen, 8, 44))
    return dict(xg=xg, x=x, y=y, nb=nb, theta1=theta1, theta2=theta2, chunks=[11, 4], sig2=1.3, ell=0.25, noise2=0.2,
                nobs=1000, jitter=1e-3)


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


def oracle_grads(p, learn_noise, maxiter_cg=60):
    """fp64 CPU autograd of -ELBO through the oracle's block ELBO, with k_n on the reference's route (`ref_compute_kn`) and
    sig2, ell and the noise variance as leaves; returns the ELBO and the gradients with respect to their logarithms (the
    model's parameters)"""
    from oracle import ziggy_oracle as zo
    sig2 = torch.tensor(p["sig2"], dtype=torch.float64, requires_grad=True)
    ell = torch.tensor(p["ell"], dtype=torch.float64, requires_grad=True)
    noise2 = torch.tensor(p["noise2"], dtype=torch.float64, requires_grad=True)
    kfun = lambda a, b: zo.matern(a, b, sig2, ell, 1.5)
    blk_idx = zo.define_block_chunks([2 * len(g) - 2 for g in p["xg"]], p["chunks"])
    Knm = kfun(p["x"], zo.meshgrid_points(p["xg"]))
    Knn = sig2 * torch.ones(len(p["x"]), dtype=torch.float64)
    nb = torch.sqrt(noise2) * torch.ones_like(p["nb"]) if learn_noise else p["nb"]
    with mock.patch.object(zo, "compute_kn", ref_compute_kn):
        elbo, g1, g2, kn, qm, qS = zo.block_elbo_and_grad(p["xg"], kfun, blk_idx, Knm, Knn, p["y"], nb, p["theta1"], p["theta2"],
                                                         p["nobs"], maxiter_cg=maxiter_cg, jitter_val=p["jitter"])
    (-elbo).backward()                          # as the model's training step does (svi_gp.py:317-329)
    out = {"elbo": float(elbo.detach()), "g_log_sig2": float(sig2.grad) * p["sig2"], "g_log_ell": float(ell.grad) * p["ell"]}
    if learn_noise:
        out["g_log_noise2"] = float(noise2.grad) * p["noise2"]
    return out


def make_model(p, dtype, learn_kernel, learn_noise, parameterization="expectation-family"):
    from hipgp_b200 import kernels as hk
    from hipgp_b200.hipgp import BlockToeplitzGP
    mod = BlockToeplitzGP(hk.Matern(nu=1.5, dtype=dtype), [g.to(dtype) for g in p["xg"]], num_obs=p["nobs"], block_sizes=p["chunks"],
                          sig2_init=p["sig2"], ell_init=p["ell"], noise2_init=p["noise2"], dtype=dtype, jitter_val=p["jitter"],
                          learn_kernel=learn_kernel, learn_noise=learn_noise, parameterization=parameterization)
    if parameterization == "expectation-family":
        mod.global_theta1.data.copy_(p["theta1"].to(dtype)); mod.global_theta2.data.copy_(p["theta2"].to(dtype))
    return mod.cuda_params(0)


@pytest.mark.parametrize("dname", ["f64", "f32"])
@pytest.mark.parametrize("learn_noise", [False, True])
def test_hyperparameter_gradients_vs_oracle_autograd(dname, learn_noise):
    p = problem()
    want = oracle_grads(p, learn_noise)
    dtype = DT[dname]
    mod = make_model(p, dtype, True, learn_noise)
    x, y = p["x"].to(DEV, dtype), p["y"].to(DEV, dtype)
    nb = None if learn_noise else p["nb"].to(DEV, dtype)
    elbo = mod.elbo_and_grad(x, y, nb, maxiter_cg=60)
    assert elbo.requires_grad
    (-elbo).backward()
    tol = HYPER_TOL[dname]
    assert close(elbo, want["elbo"], 1e-8 if dname == "f64" else 2e-3), (float(elbo), want["elbo"])
    got = {"g_log_sig2": mod.log_sig2.grad, "g_log_ell": mod.log_ell.grad}
    if learn_noise:
        got["g_log_noise2"] = mod.log_noise2.grad
    for name, g in got.items():
        assert g is not None and close(g, want[name], tol), (name, float(g), want[name])
    # the natural gradients of the variational parameters do not depend on whether the hyper-parameters are traced
    ref = make_model(p, dtype, False, False)
    ref.elbo_and_grad(x, y, None if learn_noise else nb, maxiter_cg=60)
    lim = 1e-8 if dname == "f64" else 2e-3
    assert relerr(mod.global_theta1.grad, ref.global_theta1.grad) < lim
    assert relerr(mod.global_theta2.grad, ref.global_theta2.grad) < lim
    # one Adam step on the hyper-parameters (svi_gp.py:254-262,327-329) moves them
    opt = torch.optim.Adam([mod.log_ell, mod.log_sig2], lr=1e-2)
    before = (float(mod.log_ell), float(mod.log_sig2))
    opt.step()
    assert float(mod.log_ell) != before[0] and float(mod.log_sig2) != before[1]


@pytest.mark.parametrize("dname", ["f64", "f32"])
@pytest.mark.parametrize("tag", ["matern32", "sqexp_noise"])
def test_unit_blocks_match_reference_meanfield_gradients(tag, dname, golden_dir):
    """1x1 blocks make the block family the mean-field one: its hyper-parameter gradients must be the golden ones, which the
    UNMODIFIED reference's autograd produced for MeanFieldToeplitzGP.  (The block KL adds a 1e-4 jitter, so the ELBO values
    differ slightly; the KL does not depend on the hyper-parameters.)"""
    from hipgp_b200 import kernels as hk
    from hipgp_b200.hipgp import BlockToeplitzGP
    g = np.load(os.path.join(golden_dir, "learn_kernel_%s.npz" % dname))
    dtype = DT[dname]
    sig2, ell, noise2, jitter, nobs = [float(t) for t in g[tag + "_params"]]
    xg = [torch.linspace(lo, hi, int(m), dtype=dtype) for lo, hi, m in g[tag + "_grids"]]
    kern = hk.SqExp(dtype=dtype) if tag.startswith("sqexp") else hk.Matern(nu=1.5, dtype=dtype)
    learn_noise = tag.endswith("noise")
    mod = BlockToeplitzGP(kern, xg, num_obs=int(nobs), block_sizes=[1, 1], sig2_init=sig2, ell_init=ell, noise2_init=noise2,
                          dtype=dtype, jitter_val=jitter, learn_kernel=True, learn_noise=learn_noise)
    assert mod.block_size == 1
    theta2 = torch.from_numpy(g[tag + "_theta2"]).reshape(-1)
    mod.global_theta1.data.copy_(torch.from_numpy(g[tag + "_theta1"]))
    mod.global_theta2.data.copy_(theta2[mod.block_idx[:, 0]].reshape(-1, 1, 1))
    mod = mod.cuda_params(0)
    x = torch.from_numpy(g[tag + "_x"]).to(DEV); y = torch.from_numpy(g[tag + "_y"]).to(DEV)
    nb = None if learn_noise else torch.from_numpy(g[tag + "_noise_std"]).to(DEV)
    elbo = mod.elbo_and_grad(x, y, nb, maxiter_cg=60)
    (-elbo).backward()
    tol = HYPER_TOL[dname]
    names = [("g_log_sig2", mod.log_sig2), ("g_log_ell", mod.log_ell)] + ([("g_log_noise2", mod.log_noise2)] if learn_noise else [])
    for name, par in names:
        want = float(g[tag + "_" + name])
        assert par.grad is not None and close(par.grad, want, tol), (name, float(par.grad), want)
    # the ELBO up to the two KL terms: the mean-field KL of the same q(u) replaces the jittered block KL
    with torch.no_grad():
        qm, qS = mod.standard_variational_params()
        kl_mf = .5 * (qS.sum() + (qm * qm).sum() - torch.log(qS).sum() - qm.numel())
        mf_elbo = float(elbo) + (float(mod.get_kl_to_prior(qm, qS)) - float(kl_mf)) / nobs
    assert abs(mf_elbo - float(g[tag + "_elbo"])) <= (1e-8 if dname == "f64" else 2e-3) * abs(float(g[tag + "_elbo"]))


def test_knSkn_node_vs_torch_autograd():
    """the node's kn and S gradients against torch autograd of sum_b g_b kn_b . gather_bmm(S, kn)_b, non-symmetric S, fp64;
    65-point blocks (a full and a one-row tile) and 70 rows (two tiles of right-hand sides)"""
    from hipgp_b200.hipgp import _BlockKnSkn
    from hipgp_b200.util import define_block_chunks
    from oracle import ziggy_oracle as zo
    idx, _, _ = define_block_chunks([torch.arange(26), torch.arange(20)], [13, 5])
    gen = torch.Generator().manual_seed(9)
    nblk, bs = idx.shape
    kn = torch.randn(70, nblk * bs, dtype=torch.float64, generator=gen)
    S = torch.randn(nblk, bs, bs, dtype=torch.float64, generator=gen)
    g = torch.randn(70, dtype=torch.float64, generator=gen)
    knd = kn.to(DEV).requires_grad_(True); Sd = S.to(DEV).requires_grad_(True)
    out = _BlockKnSkn.apply(knd, Sd, idx.to(DEV))
    (out * g.to(DEV)).sum().backward()
    knc = kn.clone().requires_grad_(True); Sc = S.clone().requires_grad_(True)
    outc = torch.sum(knc * zo.block_diag_multiply(idx, Sc, knc), dim=-1)
    (outc * g).sum().backward()
    assert relerr(out, outc) < 1e-12
    assert relerr(knd.grad, knc.grad) < 1e-12
    assert relerr(Sd.grad, Sc.grad) < 1e-12


@pytest.mark.parametrize("dname", ["f64", "f32"])
def test_knSkn_node_kn_gradient_at_config3_shape(dname):
    """the 13 x 13 chunks of the 300 x 300 grid (2116 blocks of 169) with 40 rows against a fp64 torch gather + bmm"""
    from hipgp_b200.plan import block_quadform_grad
    from hipgp_b200.util import define_block_chunks
    dtype = DT[dname]
    idx, _, _ = define_block_chunks([torch.arange(598), torch.arange(598)], [13, 13])
    idxd = idx.to(DEV)
    gen = torch.Generator(device=DEV); gen.manual_seed(2)
    nblk, bs = idx.shape
    kn = torch.randn(40, nblk * bs, device=DEV, dtype=dtype, generator=gen)
    S = torch.randn(nblk, bs, bs, device=DEV, dtype=dtype, generator=gen)
    g = torch.randn(40, device=DEV, dtype=dtype, generator=gen)
    got = block_quadform_grad(S, kn, g, idxd)
    Sd = S.double()
    prod = torch.matmul(Sd + Sd.transpose(1, 2), kn.double()[:, idxd][..., None]).flatten(start_dim=1)
    want = g.double()[:, None] * prod[:, torch.argsort(idxd.flatten())]
    assert relerr(got, want) < (1e-5 if dname == "f32" else 1e-10)


def test_elbo_standard_parameterisation_and_batch_an():
    """`elbo()` for the block family: global_m / global_S gradients (S not symmetric) against autograd of a fp64 torch restatement
    on the model's own kn; `compute_batch_an` against the oracle's block ELBO terms"""
    from oracle import ziggy_oracle as zo
    p = problem()
    dtype = torch.float64
    mod = make_model(p, dtype, False, False, parameterization="standard")
    gen = torch.Generator().manual_seed(6)
    m0 = torch.randn(22 * 16, 1, dtype=dtype, generator=gen)
    S0 = spd_blocks(gen, 8, 44, skew=0.01)
    mod.global_m.data.copy_(m0.to(DEV)); mod.global_S.data.copy_(S0.to(DEV))
    x, y, nb = p["x"].to(DEV), p["y"].to(DEV), p["nb"].to(DEV)
    elbo = mod.elbo(x, y, nb, maxiter_cg=60)
    elbo.backward()
    with torch.no_grad():
        Knm, Knn = mod._make_grams(x)
        kn = mod.compute_kn(Knm, maxiter_cg=60).cpu()
    idx = mod.block_idx.numpy()
    m = m0.clone().requires_grad_(True); S = S0.clone().requires_grad_(True)
    ivar = 1 / p["nb"].squeeze() ** 2
    knSkn = torch.sum(kn * zo.block_diag_multiply(idx, S, kn), dim=-1)
    batch_an = -0.5 * ivar * ((kn.matmul(m).squeeze() - p["y"].squeeze()) ** 2 + Knn.reshape(-1).cpu() - torch.sum(kn * kn, -1) + knSkn) \
        - torch.log(p["nb"]).squeeze() - 0.5 * np.log(2 * np.pi)
    want = torch.mean(batch_an) - zo.block_kl_to_standard(m, S) / p["nobs"]
    want.backward()
    assert abs(float(elbo) - float(want)) <= 1e-10 * abs(float(want))
    assert relerr(mod.global_m.grad, m.grad) < 1e-10
    assert relerr(mod.global_S.grad, S.grad) < 1e-10
    # compute_batch_an (expectation-family model) against the oracle's block statistics
    mod2 = make_model(p, dtype, False, False)
    with torch.no_grad():
        an = mod2.compute_batch_an(x, y, nb, maxiter_cg=60)
    kfun = lambda a, b: zo.matern(a, b, p["sig2"], p["ell"], 1.5)
    Knm_o = kfun(p["x"], zo.meshgrid_points(p["xg"]))
    Knn_o = p["sig2"] * torch.ones(16, dtype=dtype)
    _, _, _, kn_o, qm_o, qS_o = zo.block_elbo_and_grad(p["xg"], kfun, idx, Knm_o, Knn_o, p["y"], p["nb"], p["theta1"], p["theta2"],
                                                        p["nobs"], maxiter_cg=60, jitter_val=p["jitter"])
    knSkn_o = torch.sum(kn_o * zo.block_diag_multiply(idx, qS_o, kn_o), dim=-1)
    an_o = -0.5 * ivar * ((kn_o.matmul(qm_o).squeeze() - p["y"].squeeze()) ** 2 + Knn_o - torch.sum(kn_o * kn_o, -1) + knSkn_o) \
        - torch.log(p["nb"]).squeeze() - 0.5 * np.log(2 * np.pi)
    assert relerr(an, an_o) < 1e-8
