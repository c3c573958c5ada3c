"""GPU checks of the four-step path for long 1-D grids (long1d_kernels.cuh / long1d_api.inl).

A 1-D embedding takes the path when its row pass would not fit shared memory.  On sm_100a that is, for both dtypes,
m >= 4097 for the narrow embedding (K, C^-1: today's length would be 16384, whose fp64 set-up row does not fit) and
m >= 2732 for the wide one (R^T, R).  The operators are checked through the same properties as tests/test_gpu_sizes.py:
  * K v and the C^-1 block against a dense FFT evaluation of the reference formula in numpy fp64;
  * || R^T v ||^2 = v^T K v  and  R R^T v = K v;
  * fp32 against fp64;
plus the Bluestein DCT-I set-up, PCG against the oracle, gram_solve at M = 10^6 and the refusals."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
# (largest m on the row pass, smallest m on the four-step path) per embedding
SWITCH = {"narrow": (4096, 4097), "wide": (2731, 2732)}


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def first_col(dims):
    g = np.meshgrid(*[np.linspace(0.0, 1.0 + 0.3 * d, m) for d, m in enumerate(dims)], indexing="ij")
    r = np.sqrt(sum((x - x.flat[0]) ** 2 for x in g))
    ell = 3.0 / max(dims)
    col = (1 + np.sqrt(5) * r / ell + 5 * r ** 2 / (3 * ell ** 2)) * np.exp(-np.sqrt(5) * r / ell)
    col = col.reshape(-1).copy(); col[0] += 1e-3
    return col


def dense_apply(col, dims, v, f):
    """reference formula: crop IFFT_N( f(max(Re FFT_N C, 1e-6)) * FFT_N pad v ), N = 2m-2 per axis (numpy fp64)"""
    D = len(dims)
    Cc = col.reshape(dims)
    for d in range(D):
        if dims[d] > 1:
            sl = [slice(None)] * D; sl[d] = slice(dims[d] - 2, 0, -1)
            Cc = np.concatenate([Cc, Cc[tuple(sl)]], axis=d)
    Dg = np.maximum(np.fft.fftn(Cc).real, 1e-6)
    x = np.zeros((v.shape[0],) + Cc.shape)
    x[(slice(None),) + tuple(slice(0, k) for k in dims)] = v.reshape((v.shape[0],) + tuple(dims))
    ax = tuple(range(1, D + 1))
    y = np.fft.ifftn(f(Dg) * np.fft.fftn(x, axes=ax), axes=ax).real
    return y[(slice(None),) + tuple(slice(0, k) for k in dims)].reshape(v.shape[0], -1)


def _free():
    import gc
    gc.collect(); torch.cuda.empty_cache()


@pytest.mark.parametrize("dt", [torch.float64, torch.float32], ids=["f64", "f32"])
def test_switch(dt):
    """the last m on the row pass takes 2 launches per matvec, the first m on the four-step path 3; both are right"""
    from hipgp_b200.plan import Plan
    from hipgp_b200 import _lib as L
    tol = 1e-10 if dt == torch.float64 else 1e-5
    for emb, mode in (("narrow", L.MV_K), ("wide", L.MV_RT)):
        for m, launches in zip(SWITCH[emb], (2, 3)):
            col = first_col((m,))
            plan = Plan([m], dt, DEV).set_first_row(torch.from_numpy(col).to(DEV, dt))
            v64 = np.random.default_rng(m).standard_normal((3, m))
            v = torch.from_numpy(v64).to(DEV, dt)
            plan.matvec(mode, v)
            n0 = plan.launch_count()
            out = plan.matvec(mode, v)
            assert plan.launch_count() - n0 == launches, (emb, m)
            f = (lambda d: d) if mode == L.MV_K else np.sqrt
            if mode == L.MV_K:
                assert relerr(out.cpu().numpy(), dense_apply(col, (m,), v.double().cpu().numpy(), f)) < tol, (emb, m)
            else:
                Kv = plan.matvec(L.MV_K, v).double()
                vKv = (v.double() * Kv).sum(1)
                assert float(((out.double() ** 2).sum(1) - vKv).abs().max() / vKv.abs().max()) < 10 * tol, (emb, m)


@pytest.mark.parametrize("m,B", [(4097, 3), (100000, 2), (1000000, 3)])
def test_operator_properties(m, B):
    from hipgp_b200.plan import Plan
    from hipgp_b200 import _lib as L
    dims = (m,)
    col = first_col(dims)
    rng = np.random.default_rng(1)
    v64 = rng.standard_normal((B, m))
    out = {}
    for dname, dt, tol in (("f64", torch.float64, 1e-10), ("f32", torch.float32, 1e-5)):
        plan = Plan([m], dt, DEV).set_first_row(torch.from_numpy(col).to(DEV, dt))
        v = torch.from_numpy(v64).to(DEV, dt)
        Kv = plan.matvec(L.MV_K, v)
        Pv = plan.matvec(L.MV_CINV, v)
        RTv = plan.matvec(L.MV_RT, v)
        RRTv = plan.matvec(L.MV_R, RTv)
        vin = v.double().cpu().numpy()
        assert relerr(Kv.cpu().numpy(), dense_apply(col, dims, vin, lambda d: d)) < tol
        Dsp = plan.spectrum(L.SPEC_D)
        ptol = tol if dname == "f64" else 1e-5 + 0.5 * float(Dsp.max() / Dsp.min()) * 2.0 ** -24
        perr = relerr(Pv.cpu().numpy(), dense_apply(col, dims, vin, lambda d: 1.0 / d))
        assert perr < ptol, (perr, ptol)
        vKv = (v.double() * Kv.double()).sum(1)
        assert float(((RTv.double() ** 2).sum(1) - vKv).abs().max() / vKv.abs().max()) < 10 * tol
        assert relerr(RRTv.cpu().numpy(), Kv.cpu().numpy()) < 10 * tol
        out[dname] = (Kv.double().cpu().numpy(), RTv.double().cpu().numpy())
        del plan, v, Kv, Pv, RTv, RRTv
    assert relerr(out["f32"][0], out["f64"][0]) < 1e-5 and relerr(out["f32"][1], out["f64"][1]) < 1e-5
    _free()


@pytest.mark.parametrize("m", [100000, 1000000])
def test_setup_spectrum(m):
    """the Bluestein DCT-I set-up against Re FFT_N of the embedding (N = 2m - 2: 199998 = 2 * 3 * 33333, not smooth)"""
    from hipgp_b200.plan import Plan
    from hipgp_b200 import _lib as L
    col = first_col((m,))
    plan = Plan([m], torch.float64, DEV).set_first_row(torch.from_numpy(col).to(DEV))
    raw = np.fft.fft(np.concatenate([col, col[m - 2:0:-1]])).real
    ref = np.maximum(raw, 1e-6)
    got = plan.spectrum(L.SPEC_D).cpu().numpy()
    assert np.abs(got - ref).max() / np.abs(ref).max() < 1e-12
    # (a raw eigenvalue within rounding of the clamp could go either way)
    near = int((np.abs(raw - 1e-6) < 1e-12 * np.abs(raw).max()).sum())
    assert abs(plan.num_clamped - int((raw < 1e-6).sum())) <= near


def test_pcg_iterates_vs_oracle():
    """m = 10^5, fp64, lengthscale 100 grid steps: after the same number of PCG iterations the device iterate equals the oracle's, and so do the
    callback counts (cg.py:70-78) and the recurrence residual"""
    from hipgp_b200.plan import Plan
    from oracle import ziggy_oracle as zo
    m, iters = 100000, 5
    ora = zo.OracleToeplitz([torch.linspace(0, 4, m, dtype=torch.float64)], lambda x, y: zo.matern(x, y, 1.0, 4e-3, 2.5), jitter_val=1e-3)
    torch.manual_seed(42)
    v = torch.randn(2, m, dtype=torch.float64)
    n_ref = [0]
    x_ref = ora.solve(v, do_precond=True, maxiter=iters, tol=1e-12, callback=lambda n, x: n_ref.__setitem__(0, n_ref[0] + 1))
    plan = Plan([m], torch.float64, DEV).set_first_row(ora.column.to(DEV))
    n_dev = [0]
    x, info = plan.pcg(v.to(DEV), maxiter=iters, tol=1e-12, callback=lambda n, xx: n_dev.__setitem__(0, n_dev[0] + 1), return_info=True)
    assert n_dev[0] == n_ref[0] == info["callbacks"] == iters and info["iters"] == iters
    assert relerr(x.cpu().numpy(), x_ref.numpy()) < 1e-9
    P = ora.matmul_Cinv
    r = v.clone(); z = P(r); p = z
    for _ in range(iters):                 # the oracle's recurrence (cg.py:44-80), for its residual
        rs = (r * z).sum(1); Ap = ora.matmul_K(p); a = rs / (p * Ap).sum(1)
        r = r - a[:, None] * Ap; z = P(r); p = z + ((z * r).sum(1) / rs)[:, None] * p
    assert np.allclose(info["resid"], r.norm(dim=1).numpy(), rtol=1e-6, atol=1e-9 * float(v.norm(dim=1).max()))


def test_gram_solve_harness_shape():
    """gram_solve at M = 10^6, fp32, 200 right-hand sides on the fused route (the reference harness shape): R^T of the
    solve comes back, and the true residual ||b - K x|| of a few rows, with K the numpy fp64 formula, is what the
    solver's K says it is and is small"""
    from hipgp_b200 import toeplitz_expanded
    from oracle import ziggy_oracle as zo
    M, B, dt = 1000000, 200, torch.float32
    x1 = torch.linspace(0, 1, M, device=DEV, dtype=dt)
    ell = 2.5 / (M - 1)
    kfun = lambda x, y: zo.matern(x, y, 1.0, ell, 2.5)
    g = torch.Generator(device=DEV); g.manual_seed(7)
    b = torch.randn(B, M, device=DEV, dtype=dt, generator=g)
    K = toeplitz_expanded.ToeplitzMatmul([x1], kfun, batch_shape=(B,))
    x = toeplitz_expanded.gram_solve([x1], kfun, b, K_matmul=K, maxiter=60, tol=1e-3, mult_RT=False)
    kn = toeplitz_expanded.gram_solve([x1], kfun, b, K_matmul=K, maxiter=60, tol=1e-3, mult_RT=True)
    assert x.shape == (B, M) and kn.shape == (B, 2 * M - 2)
    rows = [0, 101, B - 1]
    want = K(x[rows].contiguous(), multiply_type="RTv")        # (other pair partners: equal to rounding, not bitwise)
    assert float(((kn[rows] - want).double().norm(dim=1) / want.double().norm(dim=1)).max()) < 1e-5
    col = K.K.reshape(-1).double().cpu().numpy()                 # the Toeplitz first column the plan was built from
    xr = x[rows].double().cpu().numpy(); br = b[rows].double().cpu().numpy()
    res_np = np.linalg.norm(br - dense_apply(col, (M,), xr, lambda d: d), axis=1)
    res_dev = (b[rows] - K(x[rows].contiguous(), multiply_type="gram")).double().norm(dim=1).cpu().numpy()
    assert np.all(res_np < 1e-2 * np.linalg.norm(br, axis=1)), res_np
    assert np.allclose(res_np, res_dev, rtol=0.1, atol=1e-4 * np.linalg.norm(br, axis=1).max())
    del x, kn, b, K
    _free()


def test_batch_composition():
    """packed pairs: the rounding of a row depends on its partner, so a row of a batch matches a one-row call to rounding"""
    from hipgp_b200.plan import Plan
    from hipgp_b200 import _lib as L
    m, B, dt = 100000, 5, torch.float32
    plan = Plan([m], dt, DEV).set_first_row(torch.from_numpy(first_col((m,))).to(DEV, dt))
    g = torch.Generator(device=DEV); g.manual_seed(3)
    v = torch.randn(B, m, device=DEV, dtype=dt, generator=g)
    for mode in (L.MV_K, L.MV_CINV, L.MV_RT):
        out = plan.matvec(mode, v)
        for i in (0, 3, B - 1):
            one = plan.matvec(mode, v[i:i + 1].contiguous())[0]
            assert float((out[i] - one).double().norm() / one.double().norm()) < 1e-6, (mode, i)


def test_refusals():
    """the gradient entry points raise a RuntimeError naming the limitation on a long plan"""
    from hipgp_b200.plan import Plan
    m = 5000
    plan = Plan([m], torch.float64, DEV).set_first_row(torch.from_numpy(first_col((m,))).to(DEV))
    v = torch.ones(1, m, dtype=torch.float64, device=DEV)
    with pytest.raises(RuntimeError, match="long 1-D plans"):
        plan.toeplitz_quadform(v, v)
    with pytest.raises(RuntimeError, match="long 1-D plans"):
        plan.rt_column_grad(v, torch.ones(1, 2 * m - 2, dtype=torch.float64, device=DEV))
    torch.cuda.synchronize()
    assert torch.isfinite(plan.matvec(0, v)).all()       # the plan still works
