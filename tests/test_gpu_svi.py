"""GPU parity of the mean-field natural-gradient step / predict (hipgp.py:194-276,416-446) against the golden vectors of
the unmodified reference, the shard-additivity of its statistics, and the begin/step PCG with a caller-owned stop rule."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DT = {"f32": torch.float32, "f64": torch.float64}
DEV = "cuda:0"


def relerr(a, b):
    if isinstance(a, torch.Tensor):
        a = a.detach().cpu().numpy()
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def make_model(g, dtype):
    from hipgp_b200 import hipgp as hh, kernels as hk
    xgrids = [torch.linspace(lo, hi, int(m), dtype=dtype) for lo, hi, m in g["grids"]]
    mod = hh.MeanFieldToeplitzGP(hk.Matern(nu=1.5, dtype=dtype), xgrids, num_obs=int(g["params"][3]),
                                 sig2_init=float(g["params"][0]), ell_init=float(g["params"][1]), dtype=dtype,
                                 jitter_val=float(g["params"][2])).cuda_params(0)
    mod.global_theta1.data.copy_(torch.from_numpy(g["theta1"])); mod.global_theta2.data.copy_(torch.from_numpy(g["theta2"]))
    return mod


@pytest.mark.parametrize("dname", ["f32", "f64"])
def test_meanfield_step_vs_reference(dname, golden_dir):
    g = np.load(os.path.join(golden_dir, "svi_step_%s.npz" % dname))
    dtype = DT[dname]
    tol = 1e-6 if dname == "f64" else 2e-3
    mod = make_model(g, dtype)
    x = torch.from_numpy(g["x"]).to(DEV); y = torch.from_numpy(g["y"]).to(DEV); nb = torch.from_numpy(g["noise_std"]).to(DEV)
    elbo = mod.elbo_and_grad(x, y, nb, maxiter_cg=20)
    assert abs(float(elbo) - float(g["elbo"])) <= tol * abs(float(g["elbo"]))
    assert relerr(mod.global_theta1.grad, g["g1"]) < tol
    assert relerr(mod.global_theta2.grad, g["g2"]) < tol
    mu, sig = mod.predict(x, maxiter_cg=50)
    assert not mu.is_cuda and relerr(mu, g["mu"]) < tol and relerr(sig, g["sig"]) < tol
    # one optimiser step exactly as svigp_fit does (SGD on theta with grad = -natural gradient, svi_gp.py:248,329)
    opt = torch.optim.SGD([mod.global_theta1, mod.global_theta2], lr=1e-2)
    opt.step()
    want1 = g["theta1"] - 1e-2 * g["g1"]
    assert relerr(mod.global_theta1.data, want1) < tol


def test_shard_additivity_of_statistics(golden_dir):
    """The packed all-reduce is exact because the statistics are sums over observations: two half-batches add up to
    the full batch (what N ranks compute, emulated on one GPU)."""
    from hipgp_b200.plan import meanfield_colstats, meanfield_rowstats
    torch.manual_seed(0)
    B, E = 10, 5000
    kn = torch.randn(B, E, dtype=torch.float64, device=DEV)
    w1 = torch.randn(B, dtype=torch.float64, device=DEV); w2 = torch.rand(B, dtype=torch.float64, device=DEV)
    qm = torch.randn(E, dtype=torch.float64, device=DEV); qS = torch.rand(E, dtype=torch.float64, device=DEV)
    dm, lam = meanfield_colstats(kn, w1, w2)
    dm2 = sum(meanfield_colstats(kn[s], w1[s], w2[s])[0] for s in (slice(0, 4), slice(4, 10)))
    lam2 = sum(meanfield_colstats(kn[s], w1[s], w2[s])[1] for s in (slice(0, 4), slice(4, 10)))
    assert relerr(dm2, dm.cpu().numpy()) < 1e-13 and relerr(lam2, lam.cpu().numpy()) < 1e-13
    assert relerr(dm, (w1[:, None] * kn).sum(0).cpu().numpy()) < 1e-13
    rs = meanfield_rowstats(kn, qm, qS)
    assert relerr(rs[0], (kn @ qm).cpu().numpy()) < 1e-12
    assert relerr(rs[1], (kn * kn).sum(1).cpu().numpy()) < 1e-12
    assert relerr(rs[2], (kn * kn * qS).sum(1).cpu().numpy()) < 1e-12


def test_begin_step_pcg_matches_fused_solve(golden_dir):
    """hipgp_pcg_begin/step with the stop rule evaluated by the caller reproduces hipgp_pcg (same iterates, same count);
    a minibatch split in two shards with the GLOBAL rule stops both shards at the unsharded iteration."""
    from hipgp_b200.plan import Plan
    from hipgp_b200 import dist as hdist
    g = np.load(os.path.join(golden_dir, "toeplitz_2d_25x25_matern52_f64.npz"), allow_pickle=True)
    plan = Plan([25, 25], torch.float64, DEV).set_first_row(torch.from_numpy(g["column"]).to(DEV))
    v = torch.from_numpy(g["v"]).to(DEV)
    x_ref, info = plan.pcg(v, maxiter=500, tol=1e-10, return_info=True)
    x, it = hdist.sharded_pcg(plan, v, maxiter=500, tol=1e-10)
    assert it == info["iters"] and relerr(x, x_ref.cpu().numpy()) < 1e-14
    # two shards, global rule: iterate both until max over shards < tol
    plans = [Plan([25, 25], torch.float64, DEV).set_first_row(torch.from_numpy(g["column"]).to(DEV)) for _ in range(2)]
    xs = [plans[0].pcg_begin(v[:1]), plans[1].pcg_begin(v[1:])]
    for it2 in range(1, 501):
        mx = max(plans[0].pcg_step(1)[2], plans[1].pcg_step(1)[2])
        if mx < 1e-10:
            break
    assert it2 == info["iters"]
    assert relerr(torch.cat(xs), x_ref.cpu().numpy()) < 1e-12


@pytest.mark.parametrize("exchange", ["peer", "nccl"])
@pytest.mark.parametrize("dname,nranks", [("f64", 2), ("f64", 4), ("f32", 2), ("f32", 4)])
def test_slab_decomposed_matvec_emulated(dname, nranks, exchange):
    """Grid-sharded (slab) K and C^-1 matvecs: all ranks emulated on one GPU, the all-to-all done by tensor shuffling;
    must equal the undecomposed plan and the CPU oracle."""
    from hipgp_b200.slab import SlabToeplitz
    from hipgp_b200.plan import Plan
    from hipgp_b200 import _lib as L, kernels as hk
    from oracle import ziggy_oracle as zo
    dtype = DT[dname]
    dims = (16, 12, 20)
    xg = [torch.linspace(0, 1 + d, m, dtype=dtype, device=DEV) for d, m in enumerate(dims)]
    col = hk.first_row(xg, hk.Matern(nu=1.5, dtype=dtype), (1.0, 0.4), jitter=1e-2)
    slab = SlabToeplitz(dims, col, dtype, DEV, emulate_ranks=nranks, exchange=exchange)
    full = Plan(dims, dtype, DEV).set_first_row(col)
    torch.manual_seed(0)
    v = torch.randn(1, int(np.prod(dims)), dtype=dtype, device=DEV)
    n0 = dims[0] // nranks
    slabs = [v.view(dims)[r * n0:(r + 1) * n0].contiguous() for r in range(nranks)]
    ora = zo.OracleToeplitz([g.cpu() for g in xg], lambda x, y: zo.matern(x, y, 1.0, 0.4, 1.5), jitter_val=1e-2)
    tol = 1e-10 if dname == "f64" else 1e-5
    for mode, ref in ((L.MV_K, ora.matmul_K(v.cpu())), (L.MV_CINV, ora.matmul_Cinv(v.cpu()))):
        got = torch.cat(slab.matvec(mode, slabs)).reshape(1, -1)
        assert relerr(got, full.matvec(mode, v).cpu().numpy()) < tol
        assert relerr(got, ref.numpy()) < (tol if mode == L.MV_K else 50 * tol)


@pytest.mark.parametrize("precond", [True, False])
def test_slab_solver_device_side_stopping_rule(precond):
    """SlabToeplitz.solve keeps the reference's break (cg.py:66-67) as a device-side flag: on one rank it must stop at the
    iteration the plan's PCG stops and return the same iterate, also when the host only looks every 5 iterations."""
    from hipgp_b200.slab import SlabToeplitz
    from hipgp_b200.plan import Plan
    from hipgp_b200 import kernels as hk
    dtype = torch.float64
    dims = (12, 10, 14)
    xg = [torch.linspace(0, 1 + d, m, dtype=dtype, device=DEV) for d, m in enumerate(dims)]
    col = hk.first_row(xg, hk.Matern(nu=1.5, dtype=dtype), (1.0, 0.15), jitter=1e-2)   # oracle: 21 preconditioned / 114 plain iterations
    slab = SlabToeplitz(dims, col, dtype, DEV, rank=0, nranks=1)
    full = Plan(dims, dtype, DEV).set_first_row(col)
    torch.manual_seed(1)
    b = torch.randn(1, int(np.prod(dims)), dtype=dtype, device=DEV)
    x_ref, info = full.pcg(b, maxiter=400, tol=1e-8, precond=precond, return_info=True)
    x = slab.solve(b, do_precond=precond, maxiter=400, tol=1e-8)
    assert 3 < info["iters"] < 200
    assert abs(slab.last_iters - info["iters"]) <= 1
    assert relerr(x, x_ref.cpu().numpy()) < 1e-9
    # stopping early must not depend on how often the host looks
    x1 = slab.solve(b, do_precond=precond, maxiter=400, tol=1e-8, check_every=1)
    assert torch.equal(x1, x)


def test_batch_predict_streams_the_same_batches(golden_dir):
    """batch_predict (svi_gp.py:78-97): same batches as the reference's batch_indices (bit-exact slices), each predicted
    exactly as predict() does, one D2H copy at the end."""
    from oracle import ziggy_oracle as zo
    g = np.load(os.path.join(golden_dir, "svi_step_f64.npz"))
    mod = make_model(g, torch.float64)
    x = torch.from_numpy(g["x"]).to(DEV)
    n = x.shape[0]
    for bs in (7, n, n + 3, 1):
        if bs == 1 and n > 40:
            continue
        mu, sig = mod.batch_predict(x, bs, verbose=False, maxiter_cg=50)
        assert not mu.is_cuda and mu.shape == (n, 1) and sig.shape == (n, 1)
        parts = [mod.predict(x[b], maxiter_cg=50) for b in zo.batch_indices(n, bs)]
        assert torch.equal(mu, torch.cat([p[0] for p in parts])) and torch.equal(sig, torch.cat([p[1] for p in parts]))


def test_misaligned_rows_take_the_scalar_path():
    """Vectors whose rows are not 16-byte aligned (a row-offset view of an odd-length batch) must give the same matvec
    and PCG results as aligned copies: the row kernels fall back from 16-byte chunks to element accesses."""
    from hipgp_b200.plan import Plan
    from hipgp_b200 import _lib as L, kernels as hk
    for dtype, tol in ((torch.float32, 1e-6), (torch.float64, 1e-13)):
        dims = (33, 35)
        xg = [torch.linspace(0, 1, m, dtype=dtype, device=DEV) for m in dims]
        plan = Plan(list(dims), dtype, DEV).set_first_row(hk.first_row(xg, hk.Matern(nu=2.5, dtype=dtype), (1.0, 0.2), jitter=1e-2))
        M = dims[0] * dims[1]
        big = torch.randn(4 * M + 1, dtype=dtype, device=DEV)
        v_mis = big[1:1 + 3 * M].view(3, M)                 # data_ptr offset by one element
        assert v_mis.data_ptr() % 16 != 0
        v_al = v_mis.clone()
        for mode in (L.MV_K, L.MV_CINV, L.MV_RT):
            assert relerr(plan.matvec(mode, v_mis), plan.matvec(mode, v_al).cpu().numpy()) < tol
        assert relerr(plan.pcg(v_mis, maxiter=15, tol=1e-12), plan.pcg(v_al, maxiter=15, tol=1e-12).cpu().numpy()) < 100 * tol
