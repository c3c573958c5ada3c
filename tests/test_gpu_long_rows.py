"""GPU checks of the four-step path along the LAST axis of 2-D and 3-D grids (long1d_kernels.cuh / long1d_api.inl with the
column passes of the leading axes in between).

The last axis leaves the one-block row pass where a 1-D grid of the same length would: on sm_100a, for both dtypes, from
m = 4097 for the narrow embedding (K, C^-1) and from m = 2732 for the wide one (R^T, R).  Checked:
  * both sides of each switch: launches per matvec and the result;
  * user sizes: K against the dense fp64 formula crop IFFT_N(max(Re FFT_N C, 1e-6) FFT_N pad v), || R^T v ||^2 = v^T K v,
    R R^T v = K v, fp32 against fp64;
  * a row of a batch against a one-row call (packed pairs);
  * PCG against the oracle, and the asynchronous host solve against the device solve;
  * one mean-field natural-gradient step against the oracle's;
  * the refusals."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def relerr(a, b):
    a = torch.as_tensor(a).double().cpu(); b = torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / max(float(b.norm()), 1e-300))


def first_col(dims):
    g = np.meshgrid(*[np.linspace(0.0, 1.0 + 0.3 * d, m) for d, m in enumerate(dims)], indexing="ij")
    r = np.sqrt(sum((x - x.flat[0]) ** 2 for x in g))
    ell = 3.0 / max(dims)
    col = (1 + np.sqrt(5) * r / ell + 5 * r ** 2 / (3 * ell ** 2)) * np.exp(-np.sqrt(5) * r / ell)
    col = col.reshape(-1).copy(); col[0] += 1e-3
    return col


def dense_K(col, dims, v):
    """the reference formula crop IFFT_N( max(Re FFT_N C, 1e-6) * FFT_N pad v ), N = 2m - 2 per axis, in fp64 (torch.fft on
    the device: the user sizes are too big for a quick numpy evaluation)"""
    D = len(dims)
    Cc = torch.from_numpy(col).to(DEV, torch.float64).reshape(dims)
    for d in range(D):
        Cc = torch.cat([Cc, Cc.narrow(d, 1, dims[d] - 2).flip(d)], dim=d)
    Dg = torch.fft.fftn(Cc).real.clamp(min=1e-6)
    x = torch.zeros((v.shape[0],) + tuple(Cc.shape), dtype=torch.float64, device=DEV)
    x[(slice(None),) + tuple(slice(0, k) for k in dims)] = v.to(DEV, torch.float64).reshape((v.shape[0],) + tuple(dims))
    ax = tuple(range(1, D + 1))
    y = torch.fft.ifftn(Dg * torch.fft.fftn(x, dim=ax), dim=ax).real
    return y[(slice(None),) + tuple(slice(0, k) for k in dims)].reshape(v.shape[0], -1)


def _free():
    import gc
    gc.collect(); torch.cuda.empty_cache()


def make_plan(dims, dt, col=None):
    from hipgp_b200.plan import Plan
    col = first_col(dims) if col is None else col
    return Plan(list(dims), dt, DEV).set_first_row(torch.from_numpy(col).to(DEV, dt)), col


@pytest.mark.parametrize("dt", [torch.float64, torch.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("lead", [(5,), (2, 3)], ids=["2d", "3d"])
def test_switch(lead, dt):
    """the last m on the row pass takes 3 (2-D) / 5 (3-D) launches per matvec, the first m on the four-step path 5 / 7;
    both are right"""
    from hipgp_b200 import _lib as L
    tol = 1e-10 if dt == torch.float64 else 1e-5
    row, four = (3, 5) if len(lead) == 1 else (5, 7)
    for mode, ms in ((L.MV_K, (4096, 4097)), (L.MV_RT, (2731, 2732))):
        for m, launches in zip(ms, (row, four)):
            dims = lead + (m,)
            plan, col = make_plan(dims, dt)
            v = torch.from_numpy(np.random.default_rng(m).standard_normal((3, int(np.prod(dims))))).to(DEV, dt)
            plan.matvec(mode, v)
            n0 = plan.launch_count()
            out = plan.matvec(mode, v)
            assert plan.launch_count() - n0 == launches, (dims, mode)
            Kv = plan.matvec(L.MV_K, v)
            if mode == L.MV_K:
                assert relerr(out, dense_K(col, dims, v)) < tol, dims
            else:
                vKv = (v.double() * Kv.double()).sum(1)
                assert float(((out.double() ** 2).sum(1) - vKv).abs().max() / vKv.abs().max()) < 10 * tol, dims
                assert relerr(plan.matvec(L.MV_R, out), Kv) < 10 * tol, dims
            del plan, v, out, Kv
    _free()


@pytest.mark.parametrize("dims", [(3000, 3000), (64, 20000), (8, 8, 5000)], ids=lambda d: "x".join(map(str, d)))
def test_user_sizes(dims):
    from hipgp_b200 import _lib as L
    B = 2
    M = int(np.prod(dims))
    v64 = torch.from_numpy(np.random.default_rng(1).standard_normal((B, M)))
    ref = dense_K(first_col(dims), dims, v64)
    out = {}
    for dname, dt, tol in (("f64", torch.float64, 1e-10), ("f32", torch.float32, 1e-5)):
        plan, col = make_plan(dims, dt)
        Ln, Lw = plan.embedding()
        assert Ln[-1] >= 2 * dims[-1] - 1 and Lw[-1] >= 3 * dims[-1] - 3
        v = v64.to(DEV, dt)
        Kv = plan.matvec(L.MV_K, v)
        RTv = plan.matvec(L.MV_RT, v)
        RRTv = plan.matvec(L.MV_R, RTv)
        assert relerr(Kv, ref) < tol, dname
        vKv = (v.double() * Kv.double()).sum(1)
        assert float(((RTv.double() ** 2).sum(1) - vKv).abs().max() / vKv.abs().max()) < 10 * tol, dname
        assert relerr(RRTv, Kv) < 10 * tol, dname
        out[dname] = (Kv.double().cpu(), RTv.double().cpu())
        del plan, v, Kv, RTv, RRTv
        _free()
    assert relerr(out["f32"][0], out["f64"][0]) < 1e-5 and relerr(out["f32"][1], out["f64"][1]) < 1e-5
    del ref
    _free()


def test_batch_composition():
    """packed pairs: the rounding of a row depends on its partner, so a row of a batch matches a one-row call to rounding"""
    from hipgp_b200 import _lib as L
    dims, B, dt = (64, 20000), 5, torch.float32
    plan, _ = make_plan(dims, dt)
    g = torch.Generator(device=DEV); g.manual_seed(3)
    v = torch.randn(B, int(np.prod(dims)), device=DEV, dtype=dt, generator=g)
    for mode in (L.MV_K, L.MV_CINV, L.MV_RT):
        out = plan.matvec(mode, v)
        for i in (0, 3, B - 1):
            one = plan.matvec(mode, v[i:i + 1].contiguous())[0]
            assert float((out[i] - one).double().norm() / one.double().norm()) < 1e-6, (mode, i)


def test_pcg_vs_oracle_and_host_solves():
    """(20, 5000), fp64: after the same number of PCG iterations the device iterate equals the oracle's, and so do the callback
    counts and the recurrence residual; the asynchronous host solve gives the device solve's bits"""
    from oracle import ziggy_oracle as zo
    m0, m1, iters, B = 20, 5000, 5, 2
    ora = zo.OracleToeplitz([torch.linspace(0, 1, m0, dtype=torch.float64), torch.linspace(0, 4, m1, dtype=torch.float64)],
                            lambda x, y: zo.matern(x, y, 1.0, 0.05, 2.5), jitter_val=1e-3)
    torch.manual_seed(42)
    v = torch.randn(B, m0 * m1, dtype=torch.float64)
    n_ref = [0]
    x_ref = ora.solve(v, do_precond=True, maxiter=iters, tol=1e-12, callback=lambda n, x: n_ref.__setitem__(0, n_ref[0] + 1))
    plan, _ = make_plan((m0, m1), torch.float64, col=ora.column.reshape(-1).numpy())
    n_dev = [0]
    x, info = plan.pcg(v.to(DEV), maxiter=iters, tol=1e-12, callback=lambda n, xx: n_dev.__setitem__(0, n_dev[0] + 1), return_info=True)
    assert n_dev[0] == n_ref[0] == info["callbacks"] == iters and info["iters"] == iters
    assert relerr(x, x_ref) < 1e-9
    P = ora.matmul_Cinv
    r = v.clone(); z = P(r); p = z
    for _ in range(iters):                 # the oracle's recurrence (cg.py:44-80), for its residual
        rs = (r * z).sum(1); Ap = ora.matmul_K(p); a = rs / (p * Ap).sum(1)
        r = r - a[:, None] * Ap; z = P(r); p = z + ((z * r).sum(1) / rs)[:, None] * p
    assert np.allclose(info["resid"], r.norm(dim=1).numpy(), rtol=1e-6, atol=1e-9 * float(v.norm(dim=1).max()))
    # a solve that converges: the host-buffer asynchronous solve against the device solve, bit for bit
    xd, infod = plan.pcg(v.to(DEV), maxiter=200, tol=1e-6, return_info=True)
    assert 0 < infod["iters"] < 200
    b_host = v.clone().pin_memory(); x_host = torch.zeros_like(v).pin_memory()
    plan.pcg_host_submit(b_host, x_host, 0, maxiter=200, tol=1e-6)
    assert plan.pcg_host_wait(0) == infod["iters"]
    assert torch.equal(x_host, xd.cpu())


def test_meanfield_step_vs_oracle():
    """one mean-field natural-gradient step (learn_kernel=False) on a (30, 3000) inducing grid against the oracle's
    restatement of the reference's step; then predict runs"""
    from hipgp_b200 import hipgp as hh, kernels as hk
    from oracle import ziggy_oracle as zo
    dtype = torch.float64
    grids = [(-2.0, 1.0, 30), (10.0, 40.0, 3000)]
    xg = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in grids]
    mod = hh.MeanFieldToeplitzGP(hk.Matern(nu=1.5, dtype=dtype), xg, num_obs=300, sig2_init=0.8, ell_init=0.6, dtype=dtype,
                                 jitter_val=1e-3, learn_kernel=False).cuda_params(0)
    g = torch.Generator(); g.manual_seed(5)
    lo = torch.tensor([a[0] for a in grids], dtype=dtype); hi = torch.tensor([a[1] for a in grids], dtype=dtype)
    xb = lo + (hi - lo) * torch.rand(8, 2, dtype=dtype, generator=g)
    yb = torch.randn(8, 1, dtype=dtype, generator=g); nb = 0.2 + 0.1 * torch.rand(8, 1, dtype=dtype, generator=g)
    th1 = mod.global_theta1.data.clone().cpu(); th2 = mod.global_theta2.data.clone().cpu()
    elbo = mod.elbo_and_grad(xb.to(DEV), yb.to(DEV), nb.to(DEV), maxiter_cg=15)
    kfun = lambda x, y: zo.matern(x, y, 0.8, 0.6, 1.5)
    Knm = kfun(xb, zo.meshgrid_points(xg)); Knn = torch.full((8,), 0.8, dtype=dtype)
    e2, g1, g2 = zo.meanfield_elbo_and_grad(xg, kfun, Knm, Knn, yb, nb, th1, th2, 300, maxiter_cg=15, jitter_val=1e-3)
    assert abs(float(elbo) - float(e2)) < 1e-8 * abs(float(e2)), (float(elbo), float(e2))
    assert relerr(mod.global_theta1.grad, g1) < 1e-8
    assert relerr(mod.global_theta2.grad, g2) < 1e-8
    mu, sig = mod.predict(xb.to(DEV), maxiter_cg=20)
    assert torch.isfinite(mu).all() and torch.isfinite(sig).all()
    del mod
    _free()


def test_refusals():
    """the gradient entry points, learn_kernel=True and the slab decomposition raise a RuntimeError naming the limitation"""
    from hipgp_b200 import hipgp as hh, kernels as hk
    from hipgp_b200.slab import SlabToeplitz
    dims = (4, 5000)
    plan, col = make_plan(dims, torch.float64)
    M, E = int(np.prod(dims)), int(np.prod([2 * m - 2 for m in dims]))
    v = torch.ones(1, M, dtype=torch.float64, device=DEV)
    with pytest.raises(RuntimeError, match="last axis is too long"):
        plan.toeplitz_quadform(v, v)
    with pytest.raises(RuntimeError, match="last axis is too long"):
        plan.rt_column_grad(v, torch.ones(1, E, dtype=torch.float64, device=DEV))
    torch.cuda.synchronize()
    assert torch.isfinite(plan.matvec(0, v)).all()       # the plan still works
    xg = [torch.linspace(0, 1, 4, dtype=torch.float64), torch.linspace(0, 10, 5000, dtype=torch.float64)]
    mod = hh.MeanFieldToeplitzGP(hk.Matern(nu=1.5, dtype=torch.float64), xg, num_obs=100, sig2_init=0.8, ell_init=0.6,
                                 dtype=torch.float64, learn_kernel=True).cuda_params(0)
    x = torch.rand(4, 2, dtype=torch.float64, device=DEV) * torch.tensor([1.0, 10.0], dtype=torch.float64, device=DEV)
    with pytest.raises(RuntimeError, match="last axis is too long"):      # (the hyper-parameter gradients, in backward)
        elbo = mod.elbo_and_grad(x, torch.randn(4, 1, dtype=torch.float64, device=DEV), 0.3 * torch.ones(4, 1, dtype=torch.float64, device=DEV))
        (-elbo).backward()
    d3 = (4, 2, 5000)
    with pytest.raises(RuntimeError, match="last axis is too long"):
        SlabToeplitz(d3, torch.from_numpy(first_col(d3)).to(DEV), torch.float64, DEV, emulate_ranks=2)
