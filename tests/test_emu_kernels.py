"""CPU execution of the CUDA kernel sources (g++ -DHIPGP_EMU build, tests/emu_build.py) against the golden vectors.
This checks index arithmetic, barriers, digit-reversed layouts, mixed-radix stages and the fused PCG bookkeeping
without a GPU.  Sizes are tiny because every CUDA thread is an OS thread here.  It is a checker for the kernel
sources; the product never loads this library."""
import ctypes as C
import os

import numpy as np
import pytest

from hipgp_b200 import _lib as L
import emu_build

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def rel(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


@pytest.fixture(scope="module")
def lib():
    return emu_build.load()


def make_plan(lib, g, dt):
    m = np.array([int(x[2]) for x in g["grids"]], dtype=np.int64)
    plan = C.c_void_p()
    assert lib.hipgp_plan_create(len(m), m.ctypes.data_as(L._pi64), L.F32 if dt == np.float32 else L.F64, 0, C.byref(plan)) == 0
    col = np.ascontiguousarray(g["column"].astype(dt).reshape(-1))
    ncl = C.c_int64()
    assert lib.hipgp_plan_set_first_row(plan, ptr(col), 1e-6, C.byref(ncl), None) == 0, lib.hipgp_last_error()
    return plan


@pytest.mark.parametrize("case,dname", [("1d_m100_sqexp", "f64"), ("1d_m2", "f64"), ("2d_17x40_matern32", "f32"),
                                        ("2d_33x20_gneiting", "f64"), ("3d_6x9x12_matern12", "f64")])
def test_matvecs(lib, case, dname):
    g = np.load(os.path.join(GOLD, "toeplitz_%s_%s.npz" % (case, dname)), allow_pickle=True)
    dt = np.float32 if dname == "f32" else np.float64
    tol = 1e-5 if dname == "f32" else 1e-10
    plan = make_plan(lib, g, dt)
    E = g["D"].size
    D = np.zeros(E, dtype=dt)
    assert lib.hipgp_plan_spectrum(plan, 0, ptr(D), None) == 0
    assert np.abs(D - g["D"].reshape(-1)).max() / np.abs(g["D"]).max() < tol
    v = np.ascontiguousarray(g["v"][:2]); w = np.ascontiguousarray(g["w"][:2])
    B, M = v.shape
    for mode, name, inp, osz in ((0, "Kv", v, M), (1, "Cinv_v", v, M), (2, "RT_v", v, E), (3, "R_w", w, M)):
        out = np.zeros((B, osz), dtype=dt)
        assert lib.hipgp_matvec(plan, mode, ptr(inp), ptr(out), B, None) == 0, lib.hipgp_last_error()
        # fp32 preconditioner: explicit first-order bound 1e-5 + kappa(D) 2^-24 (see tests/test_gpu_toeplitz.py)
        lim = 1e-5 + float(D.max() / D.min()) * 2.0 ** -24 if (name == "Cinv_v" and dname == "f32") else tol
        assert rel(out, g[name][:2]) < lim, (name, rel(out, g[name][:2]))
    lib.hipgp_plan_destroy(plan)


def test_pcg_iteration_bookkeeping(lib):
    """PCG / CG callback counts and iterates against the reference on the 1-D case (7 / 20 iterations)."""
    g = np.load(os.path.join(GOLD, "toeplitz_1d_m100_sqexp_f64.npz"), allow_pickle=True)
    plan = make_plan(lib, g, np.float64)
    v = np.ascontiguousarray(g["v"]); B, M = v.shape
    for tag, prec in (("pcg", 1), ("cg", 0)):
        maxiter, tol = g["solve_%s_args" % tag]
        x = np.zeros((B, M)); it = C.c_int(); ncb = C.c_int(); res = np.zeros(B)
        seen = []
        cb = L.ITER_CB(lambda n, xp, user: seen.append(n))
        assert lib.hipgp_pcg(plan, ptr(v), ptr(x), B, int(maxiter), float(tol), prec, C.byref(it), C.byref(ncb),
                             res.ctypes.data_as(L._pd), cb, None, None) == 0, lib.hipgp_last_error()
        assert ncb.value == int(g["solve_%s_ncb" % tag]) == len(seen)
        assert seen == list(range(len(seen)))
        assert rel(x, g["solve_%s" % tag]) < 1e-9
    lib.hipgp_plan_destroy(plan)


def test_kxu_kernels(lib):
    g = np.load(os.path.join(GOLD, "kernels_f64.npz"))
    sig2, ell = [float(t) for t in g["sig2_ell"]]
    ids = {"sqexp": 0, "matern12": 1, "matern32": 2, "matern52": 3, "gneiting": 4}
    for D in (2, 3):
        grid = g["grid_d%d" % D]
        m = np.array([int(r[2]) for r in grid], dtype=np.int64)
        axes = np.concatenate([np.linspace(lo, hi, int(n)) for lo, hi, n in grid])
        x = np.ascontiguousarray(g["x_d%d" % D])
        B, M = x.shape[0], int(np.prod(m))
        ellv = (C.c_double * 1)(ell)
        for kname, kid in ids.items():
            out = np.zeros((B, M))
            assert lib.hipgp_kxu(L.F64, kid, L.KXU_POINT, sig2, ellv, 1, 1.0, ptr(x), B, D, m.ctypes.data_as(L._pi64),
                                 ptr(axes), None, 0, ptr(out), None) == 0, lib.hipgp_last_error()
            assert rel(out, g["fwd_%s_d%d" % (kname, D)]) < 1e-12, kname
        al = np.ascontiguousarray(g["semimc_alphas"])
        out = np.zeros((B, M))
        assert lib.hipgp_kxu(L.F64, 3, L.KXU_SEMI_MC, sig2, ellv, 1, 1.0, ptr(x), B, D, m.ctypes.data_as(L._pi64), ptr(axes),
                             ptr(al), al.size, ptr(out), None) == 0
        assert rel(out, g["semimc_matern52_d%d" % D]) < 1e-12
        out = np.zeros((B, M))
        assert lib.hipgp_kxu(L.F64, 0, L.KXU_SEMI_ANALYTIC, sig2, ellv, 1, 1.0, ptr(x), B, D, m.ctypes.data_as(L._pi64),
                             ptr(axes), None, 0, ptr(out), None) == 0
        assert rel(out, g["semi_sqexp_d%d" % D]) < 1e-10
        tab = g["table_sqexp"]
        out = np.zeros(B)
        xz = x.copy(); xz[1] = 0.
        assert lib.hipgp_doubly_diag(L.F64, ptr(xz), B, D, sig2, ellv, 1, ptr(np.ascontiguousarray(tab[0])),
                                     ptr(np.ascontiguousarray(tab[1])), ptr(np.ascontiguousarray(tab[2])), tab.shape[1],
                                     ptr(out), None) == 0
        assert rel(out, g["ddiag0_sqexp_d%d" % D]) < 1e-12
    # errors come back as status + message, never as exceptions across the ABI
    assert lib.hipgp_kxu(L.F64, 2, L.KXU_SEMI_ANALYTIC, sig2, ellv, 1, 1.0, ptr(x), B, 3, m.ctypes.data_as(L._pi64),
                         ptr(axes), None, 0, ptr(out), None) != 0
    assert b"SqExp only" in lib.hipgp_last_error()


def test_vec_kernels(lib):
    rng = np.random.default_rng(0)
    B, M = 3, 5000
    a = rng.standard_normal((B, M)); b = rng.standard_normal((B, M))
    out = np.zeros(B)
    assert lib.hipgp_vec_dot(L.F64, ptr(a), ptr(b), ptr(out), B, M, None) == 0
    assert np.allclose(out, (a * b).sum(1), rtol=1e-12)
    x = rng.standard_normal((B, M)); r = rng.standard_normal((B, M)); p = rng.standard_normal((B, M)); Ap = rng.standard_normal((B, M))
    rs = rng.random(B) + 1; pAp = rng.random(B) + 1; rr = np.zeros(B)
    x0, r0 = x.copy(), r.copy()
    assert lib.hipgp_vec_xr_update(L.F64, ptr(x), ptr(r), ptr(p), ptr(Ap), ptr(rs), ptr(pAp), ptr(rr), B, M, None) == 0
    al = (rs / pAp)[:, None]
    assert np.allclose(x, x0 + al * p) and np.allclose(r, r0 - al * Ap) and np.allclose(rr, (r * r).sum(1))
    p0 = p.copy()
    assert lib.hipgp_vec_p_update(L.F64, ptr(p), ptr(x), ptr(rs), ptr(pAp), B, M, None) == 0
    assert np.allclose(p, x + al * p0)


@pytest.mark.parametrize("tag,dname", [("1d", "f64"), ("2d", "f64"), ("2d", "f32"), ("3d", "f64"), ("2d_odd", "f64"),
                                      ("3d", "f32"), ("2d_odd", "f32"), ("1d", "f32")])
def test_toeplitz_quadform(lib, tag, dname):
    """hipgp_toeplitz_quadform (forward passes, real spectrum product, one inverse, carry-pattern gather) against the
    reference's sym_toeplitz_derivative_quadratic_form on flattened 1-/2-/3-D grid vectors (golden, gpt_toeplitz.py:169-209)."""
    g = np.load(os.path.join(GOLD, "quadform_%s.npz" % dname))
    dt = np.float32 if dname == "f32" else np.float64
    dims = np.array(g[tag + "_dims"], dtype=np.int64)
    M = int(np.prod(dims))
    plan = C.c_void_p()
    assert lib.hipgp_plan_create(len(dims), dims.ctypes.data_as(L._pi64), L.F32 if dt == np.float32 else L.F64, 0, C.byref(plan)) == 0
    col = np.zeros(M, dtype=dt); col[0] = 1.0              # any first row: the form does not depend on it
    ncl = C.c_int64()
    assert lib.hipgp_plan_set_first_row(plan, ptr(col), 1e-6, C.byref(ncl), None) == 0, lib.hipgp_last_error()
    u = np.ascontiguousarray(g[tag + "_u"].astype(dt)); v = np.ascontiguousarray(g[tag + "_v"].astype(dt))
    out = np.zeros(M, dtype=dt)
    assert lib.hipgp_toeplitz_quadform(plan, ptr(u), ptr(v), u.shape[0], 1.0, ptr(out), None) == 0, lib.hipgp_last_error()
    assert rel(out, g[tag + "_quad"]) < (1e-5 if dname == "f32" else 1e-10), rel(out, g[tag + "_quad"])
    # scale and the empty sum
    assert lib.hipgp_toeplitz_quadform(plan, ptr(u), ptr(v), 1, -2.0, ptr(out), None) == 0
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
    from oracle import ziggy_oracle as zo
    ref1 = -2.0 * zo.sym_toeplitz_derivative_quadratic_form(u[0].astype(np.float64), v[0].astype(np.float64))
    assert rel(out, ref1) < (1e-5 if dname == "f32" else 1e-10)
    assert lib.hipgp_toeplitz_quadform(plan, None, None, 0, 1.0, ptr(out), None) == 0 and not out.any()
    lib.hipgp_plan_destroy(plan)


@pytest.mark.parametrize("dname", ["f32", "f64"])
def test_block_kernels(lib, dname):
    """hipgp_block_lam / hipgp_block_diag_multiply against the reference's get_lam / block_diag_multiply outputs
    (hipgp.py:640-685, golden); chunked accumulation over the minibatch rows is exercised by the emulated launch too."""
    g = np.load(os.path.join(GOLD, "block_step_%s.npz" % dname))
    dt = np.float32 if dname == "f32" else np.float64
    code = L.F32 if dname == "f32" else L.F64
    tol = 1e-5 if dname == "f32" else 1e-10
    idx = np.ascontiguousarray(g["block_idx"].astype(np.int64))
    nblk, bs = idx.shape
    kn = np.ascontiguousarray(g["kn"].astype(dt)); B, E = kn.shape
    w = np.ascontiguousarray((1.0 / g["noise_std"].reshape(-1) ** 2).astype(dt))
    lam = np.zeros((nblk, bs, bs), dtype=dt)
    assert lib.hipgp_block_lam(code, ptr(kn), ptr(w), ptr(idx), B, E, nblk, bs, 500 / 8, 1.0, ptr(lam), None) == 0, lib.hipgp_last_error()
    assert rel(lam, g["lam"]) < tol
    S = np.ascontiguousarray(g["qS"].astype(dt))
    out = np.zeros_like(kn)
    assert lib.hipgp_block_diag_multiply(code, ptr(S), ptr(kn), ptr(idx), B, E, nblk, bs, ptr(out), None) == 0, lib.hipgp_last_error()
    assert rel(out, g["Sv"]) < tol
    # argument checks: the index must tile M'
    assert lib.hipgp_block_lam(code, ptr(kn), ptr(w), ptr(idx), B, E, nblk, bs - 1, 1.0, 1.0, ptr(lam), None) != 0
    assert lib.hipgp_block_diag_multiply(code, ptr(S), ptr(kn), None, B, E, nblk, bs, ptr(out), None) != 0
    # empty minibatch: lam = diag * I, multiply is a no-op
    assert lib.hipgp_block_lam(code, None, None, ptr(idx), 0, E, nblk, bs, 3.0, 2.0, ptr(lam), None) == 0
    assert np.array_equal(lam, np.broadcast_to(2.0 * np.eye(bs, dtype=dt), lam.shape))


def test_toeplitz_quadform_lane_layout(lib):
    """fp32 on a 30x60 grid: both embedding lengths (64, 128) are in the emulation build's specialised list, so the
    forward spectra are in the fp32 LANE layout (re0, re1, im0, im1) and corr_accumulate_kernel's layout switch is taken."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
    from oracle import ziggy_oracle as zo
    dims = np.array([30, 60], dtype=np.int64); M = 1800
    plan = C.c_void_p()
    assert lib.hipgp_plan_create(2, dims.ctypes.data_as(L._pi64), L.F32, 0, C.byref(plan)) == 0
    Ln = (C.c_int64 * 2)(); Lw = (C.c_int64 * 2)()
    assert lib.hipgp_plan_embedding(plan, Ln, Lw) == 0 and list(Ln) == [64, 128]
    col = np.zeros(M, dtype=np.float32); col[0] = 1.0
    assert lib.hipgp_plan_set_first_row(plan, ptr(col), 1e-6, None, None) == 0, lib.hipgp_last_error()
    rng = np.random.default_rng(4)
    u = rng.standard_normal((2, M)).astype(np.float32); v = rng.standard_normal((2, M)).astype(np.float32)
    out = np.zeros(M, dtype=np.float32)
    assert lib.hipgp_toeplitz_quadform(plan, ptr(u), ptr(v), 2, 1.0, ptr(out), None) == 0, lib.hipgp_last_error()
    want = zo.sym_toeplitz_derivative_quadratic_form(u.T.astype(np.float64), v.T.astype(np.float64))
    assert rel(out, want) < 1e-5, rel(out, want)
    lib.hipgp_plan_destroy(plan)


def _numpy_matvec(col2d, v, which):
    """crop IFFT(f(D) * FFT pad v) in fp64, D = max(Re FFT(even embedding), 1e-6) (toeplitz_tensor.py:21-33,70-83,114-125)."""
    m0, m1 = col2d.shape
    c = np.concatenate([col2d, col2d[-2:0:-1]], axis=0)
    c = np.concatenate([c, c[:, -2:0:-1]], axis=1)
    D = np.maximum(np.fft.fft2(c).real, 1e-6)
    f = D if which == 0 else 1.0 / D
    out = []
    for row in v:
        x = np.zeros(c.shape); x[:m0, :m1] = row.reshape(m0, m1)
        out.append(np.fft.ifft2(f * np.fft.fft2(x)).real[:m0, :m1].reshape(-1))
    return np.stack(out)


@pytest.mark.parametrize("dt,B", [(np.float32, 1), (np.float32, 3), (np.float64, 2)])
def test_block_local_column_pass_2048(lib, dt, B):
    """The block-local column kernel (cols_blk_kernel.cuh) at the config-2 column length (1000 -> 2048 points): warp-owned
    blocks between the first forward and the last inverse stage, shared-memory twiddle tables (fp32), several tiles per
    persistent CTA, a partial last tile, both dtypes."""
    m0, m1 = 1000, 9
    x0 = np.linspace(0, 4, m0)[:, None]; x1 = np.linspace(-2, 2, m1)[None, :]
    r = np.sqrt((x0 - x0[0, 0]) ** 2 + (x1 - x1[0, 0]) ** 2) / 0.05
    col = (1 + np.sqrt(5) * r + 5 * r * r / 3) * np.exp(-np.sqrt(5) * r)
    col[0, 0] += 1e-3
    m = np.array([m0, m1], dtype=np.int64)
    plan = C.c_void_p()
    assert lib.hipgp_plan_create(2, m.ctypes.data_as(L._pi64), L.F32 if dt == np.float32 else L.F64, 0, C.byref(plan)) == 0
    Ln = np.zeros(2, dtype=np.int64); Lw = np.zeros(2, dtype=np.int64)
    assert lib.hipgp_plan_embedding(plan, Ln.ctypes.data_as(L._pi64), Lw.ctypes.data_as(L._pi64)) == 0
    assert Ln[0] == 2048
    colf = np.ascontiguousarray(col.astype(dt).reshape(-1))
    ncl = C.c_int64()
    assert lib.hipgp_plan_set_first_row(plan, ptr(colf), 1e-6, C.byref(ncl), None) == 0, lib.hipgp_last_error()
    rng = np.random.RandomState(5)
    v = np.ascontiguousarray(rng.randn(B, m0 * m1).astype(dt))
    tol = 1e-5 if dt == np.float32 else 1e-10
    for mode in (0, 1):
        out = np.zeros_like(v)
        assert lib.hipgp_matvec(plan, mode, ptr(v), ptr(out), B, None) == 0, lib.hipgp_last_error()
        ref = _numpy_matvec(colf.astype(np.float64).reshape(m0, m1), v.astype(np.float64), mode)
        lim = tol if mode == 0 else (2e-4 if dt == np.float32 else 1e-9)   # C^-1 amplifies the fp32 rounding of the small eigenvalues
        assert rel(out, ref) < lim, (mode, rel(out, ref))
    lib.hipgp_plan_destroy(plan)


@pytest.mark.parametrize("dims", [(14, 11), (6, 5, 4), (7,)])
def test_rt_column_gradient_against_autograd_of_the_reference_formula(lib, dims):
    """hipgp_rt_column_grad (learn_kernel=True: d/d column of sum G . R^T v through D^(1/2) with torch.clamp's gradient) against
    torch autograd through the reference formula toeplitz_tensor.py:21-33,85-97; cases whose wide embedding is shorter than
    2N - 1 (where a symmetrised correlation would alias) and clamped eigenvalues."""
    import torch
    rng = np.random.RandomState(0)
    grids = np.meshgrid(*[np.arange(m) * 0.6 for m in dims], indexing="ij")
    col = np.exp(-sum(g ** 2 for g in grids) / 3.0).reshape(-1); col[0] += 1e-3
    M = int(np.prod(dims)); E = int(np.prod([2 * m - 2 for m in dims])); B = 3
    v = rng.randn(B, M); G = rng.randn(B, E)
    cc = torch.tensor(col, requires_grad=True)
    Cm = cc.view(dims)
    for d in range(len(dims)):
        idx = [slice(None)] * len(dims); idx[d] = slice(1, -1)
        Cm = torch.cat([Cm, torch.flip(Cm[tuple(idx)], [d])], dim=d)
    D = torch.fft.fftn(Cm).real.clamp(min=1e-6)
    pad = torch.zeros((B,) + tuple(Cm.shape), dtype=torch.float64)
    pad[(slice(None),) + tuple(slice(0, m) for m in dims)] = torch.tensor(v).view((-1,) + tuple(dims))
    ax = tuple(range(1, 1 + len(dims)))
    y = torch.fft.ifftn(torch.sqrt(D) * torch.fft.fftn(pad, dim=ax), dim=ax).real.reshape(B, -1)
    (y * torch.tensor(G)).sum().backward()
    m = np.array(dims, dtype=np.int64)
    plan = C.c_void_p()
    assert lib.hipgp_plan_create(len(dims), m.ctypes.data_as(L._pi64), L.F64, 0, C.byref(plan)) == 0
    ncl = C.c_int64()
    assert lib.hipgp_plan_set_first_row(plan, ptr(np.ascontiguousarray(col)), 1e-6, C.byref(ncl), None) == 0
    out = np.zeros(M)
    assert lib.hipgp_rt_column_grad(plan, ptr(np.ascontiguousarray(v)), ptr(np.ascontiguousarray(G)), B, 1.0, ptr(out), None) == 0, lib.hipgp_last_error()
    assert rel(out, cc.grad.numpy()) < 1e-10
    lib.hipgp_plan_destroy(plan)


@pytest.mark.parametrize("dims,nranks,dname,chunks,peer", [((16, 12, 20), 2, "f64", 1, False), ((8, 6, 10), 4, "f32", 2, False),
                                                          ((12, 10, 14), 3, "f64", 1, True)])
def test_slab_stages_equal_the_undecomposed_matvec(lib, dims, nranks, dname, chunks, peer):
    """SURVEY 8(e2): the three local stages of the grid-sharded matvec (also for a rank count that divides neither embedding
    length) with the all-to-all done in numpy -- or by the packing kernels' own stores into the other ranks' buffers
    (`peer`) -- equal the one-plan matvec."""
    import sys
    sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "scripts", "dev"))
    import emu_slab
    assert emu_slab.run(dims, nranks, np.float64 if dname == "f64" else np.float32, chunks, peer)


def test_async_host_solve_entry_points(lib):
    """hipgp_pcg_host_submit / _wait (two slots) return what hipgp_pcg returns, with its iteration count."""
    g = np.load(os.path.join(GOLD, "toeplitz_1d_m100_sqexp_f64.npz"), allow_pickle=True)
    plan = make_plan(lib, g, np.float64)
    v = np.ascontiguousarray(g["v"]); B, M = v.shape
    maxiter, tol = g["solve_pcg_args"]
    want = np.zeros((B, M)); it = C.c_int(); ncb = C.c_int()
    assert lib.hipgp_pcg(plan, ptr(v), ptr(want), B, int(maxiter), float(tol), 1, C.byref(it), C.byref(ncb), None, L.ITER_CB(0), None, None) == 0
    xs = [np.zeros((B, M)), np.zeros((B, M))]
    for slot in (0, 1):
        assert lib.hipgp_pcg_host_submit(plan, ptr(v), ptr(xs[slot]), B, int(maxiter), float(tol), 1, slot, None) == 0, lib.hipgp_last_error()
    for slot in (0, 1):
        n = C.c_int()
        assert lib.hipgp_pcg_host_wait(plan, slot, C.byref(n)) == 0, lib.hipgp_last_error()
        assert n.value == it.value
        assert np.array_equal(xs[slot], want)
    assert lib.hipgp_pcg_host_wait(plan, 0, None) != 0          # nothing pending
    assert lib.hipgp_pcg_host_submit(plan, ptr(v), ptr(xs[0]), B, int(maxiter), float(tol), 1, 2, None) != 0   # bad slot
    lib.hipgp_plan_destroy(plan)


@pytest.mark.parametrize("dims", [(3,), (4,), (5,), (8,), (65,), (130,), (5, 6), (33, 3), (4, 7, 3)])
def test_spectrum_setup_equals_the_fft_of_the_even_extension(lib, dims):
    """Set-up DCT-I (reflection-folded contraction, odd and even extents, unpaired middle input, extents down to 3): the spectrum
    the plan reports is Re FFT of the circulant embedding of the first row (toeplitz_tensor.py:21-33), clamped at 1e-6; and the
    K matvec on a unit vector returns the first row itself."""
    rng = np.random.default_rng(sum(dims))
    g = np.meshgrid(*[np.linspace(0, 1 + d, k) for d, k in enumerate(dims)], indexing="ij")
    r = np.sqrt(sum((x - x.flat[0]) ** 2 for x in g))
    col = (np.exp(-0.5 * (r / 0.35) ** 2)).reshape(-1); col[0] += 1e-3
    emb = col.reshape(dims)
    for ax in range(len(dims)):                                          # even extension per axis (circulant_embed)
        mid = np.flip(emb, axis=ax)
        sl = [slice(None)] * len(dims); sl[ax] = slice(1, -1)
        emb = np.concatenate([emb, mid[tuple(sl)]], axis=ax)
    want = np.maximum(np.real(np.fft.fftn(emb)), 1e-6).reshape(-1)
    plan = C.c_void_p(); mm = np.array(dims, dtype=np.int64)
    assert lib.hipgp_plan_create(len(dims), mm.ctypes.data_as(L._pi64), L.F64, 0, C.byref(plan)) == 0
    ncl = C.c_int64()
    assert lib.hipgp_plan_set_first_row(plan, ptr(np.ascontiguousarray(col)), 1e-6, C.byref(ncl), None) == 0, lib.hipgp_last_error()
    D = np.zeros(want.size)
    assert lib.hipgp_plan_spectrum(plan, 0, ptr(D), None) == 0, lib.hipgp_last_error()
    assert np.abs(D - want).max() / np.abs(want).max() < 1e-12
    corner = np.real(np.fft.fftn(emb))[tuple(slice(0, k) for k in dims)]          # the M distinct values (DCT-I of the column)
    assert ncl.value == int(np.sum(corner < 1e-6))
    if ncl.value == 0:
        e0 = np.zeros((1, col.size)); e0[0, 0] = 1.0
        out = np.zeros((1, col.size))
        assert lib.hipgp_matvec(plan, 0, ptr(e0), ptr(out), 1, None) == 0, lib.hipgp_last_error()
        assert rel(out[0], col) < 1e-12
    lib.hipgp_plan_destroy(plan)


def test_empty_shard_statistics_are_zero_not_uninitialised(lib):
    """A rank whose shard of the minibatch is empty (3 observations on 8 GPUs) all-reduces its column statistics like everybody
    else: hipgp_meanfield_colstats must WRITE zeros for B = 0 (the buffers come from torch.empty), and the row-wise entry points
    must accept B = 0 as a no-op."""
    E = 37
    dm = np.full(E, 7.0); lam = np.full(E, 7.0)
    kn = np.zeros((1, E)); w = np.zeros(1)
    assert lib.hipgp_meanfield_colstats(L.F64, ptr(kn), ptr(w), ptr(w), 0, E, ptr(dm), ptr(lam), None) == 0, lib.hipgp_last_error()
    assert not dm.any() and not lam.any()
    out = np.full(3, 7.0)
    assert lib.hipgp_meanfield_rowstats(L.F64, ptr(kn), ptr(kn), ptr(kn), 0, E, ptr(out), None) == 0
    assert lib.hipgp_vec_dot(L.F64, ptr(kn), ptr(kn), out.ctypes.data_as(L._pd), 0, E, None) == 0
    assert (out == 7.0).all()
