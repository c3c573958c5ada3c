"""Generates the committed golden vectors under tests/golden/ by running the UNMODIFIED reference
(<checkout>/ziggy) under oracle/ref_shim.py.  Runs only where a reference checkout is available (it is not part of
this repository).  Re-run with:  python tests/golden/make_golden.py  (checkout located as in oracle/make_ref.py)

Every array here is an output of reference code on seeded inputs; nothing is produced by this repo's
own implementation.  Files:

  toeplitz_<case>_<dtype>.npz  ToeplitzTensor (toeplitz_tensor.py): column, D, the four matvecs, _solve
  cfg1_<dtype>.npz             run_solve_kn_experiment.py:27-73 (gram_solve CG vs PCG, 25x25 / 50x50 / 100x100)
  kernels_<dtype>.npz          kernels.py forward/diag/k_semi/k_semi_mc/k_doubly_diag,
                               exact_gp_1d_derivatives.py:9-38
  compute_kn_<dtype>.npz       hipgp.py:117-146 + svi_gp.py:48-76 through MeanFieldToeplitzGP
  quadform_<dtype>.npz         gpt_toeplitz.py:169-209 on flattened 1-/2-/3-D grid vectors, and the column / right-hand-side
                               gradients of InvMatmul.backward (_inv_matmul.py:28-64) through ToeplitzTensor.inv_matmul
  block_step_<dtype>.npz       BlockToeplitzGP (hipgp.py:527-690): define_block_chunks (util.py:79-126) index maps in 2-D and 3-D,
                               get_lam, block_diag_multiply, compute_knSkn, elbo_and_grad (block branch :251-261), predict
  learn_kernel_<dtype>.npz     learn_kernel=True / learn_noise=True: MeanFieldToeplitzGP.elbo_and_grad followed by (-elbo).backward() as
                               svigp_fit does (svi_gp.py:317-329): the autograd gradients of log_sig2, log_ell, log_noise2 (through
                               kernels.py, ToeplitzTensor.__init__, InvMatmul, _matmul_by_RT), and the column gradient of R^T alone
  bidiag_<dtype>.npz           misc/bidiag.py:5-148 (Golub-Kahan bidiagonalisation solve c = K^{-1/2} b) over ToeplitzMatmul's R^T / R
                               matvecs, closures as in run_pcg_vs_cholesky.py:105-108; 1-D and 2-D grids
  notebook_counts.npz          preconditioner-analysis.ipynb saved outputs (raw lines 101-103,142-144,183-185,224-226)
"""
import os
import sys
import warnings

import numpy as np
import torch

warnings.filterwarnings("ignore")
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from oracle import ref_shim  # noqa: E402

ref_shim.import_reference()
from ziggy import kernels as zk  # noqa: E402
from ziggy import hipgp as zh  # noqa: E402
from ziggy import exact_gp_1d_derivatives as zd  # noqa: E402
from ziggy.misc.toeplitz_tensor import ToeplitzTensor  # noqa: E402
from ziggy.misc import toeplitz_expanded  # noqa: E402

DT = {"f32": torch.float32, "f64": torch.float64}

_KERNELS = {}


def get_kernel(name, dtype):
    key = (name, dtype)
    if key not in _KERNELS:
        if name == "sqexp":
            _KERNELS[key] = zk.SqExp(dtype=dtype)
        elif name.startswith("matern"):
            _KERNELS[key] = zk.Matern(nu={"matern12": .5, "matern32": 1.5, "matern52": 2.5}[name], dtype=dtype)
        elif name == "gneiting":
            _KERNELS[key] = zk.Gneiting(dtype=dtype)
    return _KERNELS[key]


TOEPLITZ_CASES = {
    # name: (grids as (lo, hi, m) per dim, kernel, sig2, ell, jitter, B)
    "1d_m100_sqexp": ([(0., 2., 100)], "sqexp", 1.0, 0.05, 1e-3, 3),
    "1d_m2": ([(0., 1., 2)], "matern32", 1.0, 0.5, 1e-3, 2),
    "2d_25x25_matern52": ([(0., 4., 25), (-2., 2., 25)], "matern52", 1.0, 0.3, 1e-3, 4),
    "2d_17x40_matern32": ([(-5.7, 1.8, 17), (50., 55.5, 40)], "matern32", 1.3, 0.6, 1e-3, 3),
    "2d_33x20_gneiting": ([(0., 1., 33), (0., 1., 20)], "gneiting", 0.7, 0.15, 1e-3, 2),
    "3d_10x10x5_sqexp": ([(-.25, .25, 10), (-.25, .25, 10), (-.05, .05, 5)], "sqexp", 0.1, 0.06, 1e-3, 3),
    "3d_6x9x12_matern12": ([(0., 1., 6), (0., 2., 9), (0., 3., 12)], "matern12", 1.0, 0.4, 1e-2, 2),
}


def make_toeplitz():
    for case, (grids, kname, sig2, ell, jitter, B) in TOEPLITZ_CASES.items():
        for dname, dtype in DT.items():
            torch.manual_seed(1234)
            xgrids = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in grids]
            kern = get_kernel(kname, dtype)
            kfun = lambda x, y: kern.forward(x, y, params=(sig2, ell))
            tt = ToeplitzTensor(xgrids, kfun, batch_shape=None, jitter_val=jitter)
            M = int(tt.M)
            E = int(np.prod(tt.C.shape))
            v = torch.randn(B, M, dtype=dtype)
            w = torch.randn(B, E, dtype=dtype)
            tt.set_batch_shape(v.shape[:-1])
            out = dict(
                grids=np.array(grids, dtype=np.float64), kernel=kname, sig2=sig2, ell=ell, jitter=jitter,
                column=tt.column.numpy(), D=tt.D[..., 0].numpy(), v=v.numpy(), w=w.numpy(),
                Kv=tt._matmul_by_K(v).numpy(), Cinv_v=tt._matmul_by_Cinv(v).numpy(),
                RT_v=tt._matmul_by_RT(v).numpy(), R_w=tt._matmul_by_R(w).numpy(),
            )
            for tag, prec, maxiter, tol in [("pcg", True, 20, 1e-8), ("cg", False, 20, 1e-8),
                                            ("pcg_conv", True, 500, 1e-10 if dname == "f64" else 1e-5)]:
                xs = []
                x = tt._solve(v, do_precond=prec, maxiter=maxiter, tol=tol,
                              callback=lambda n, xx: xs.append(xx.clone()))
                out["solve_%s" % tag] = x.numpy()
                out["solve_%s_ncb" % tag] = len(xs)
                out["solve_%s_args" % tag] = np.array([maxiter, tol])
                if tag == "pcg" and len(xs) > 0:
                    out["solve_pcg_x3"] = xs[min(2, len(xs) - 1)].numpy()   # iterate after <=3 callbacks
            np.savez_compressed(os.path.join(HERE, "toeplitz_%s_%s.npz" % (case, dname)), **out)
            print("toeplitz", case, dname, "M", M, "E", E, "ncb", out["solve_pcg_ncb"], out["solve_pcg_conv_ncb"])


def make_cfg1():
    """run_solve_kn_experiment.py:27-73, verbatim call pattern (seed once, three grids in order)."""
    for dname, dtype in DT.items():
        torch.manual_seed(42)
        kern = zk.Matern(nu=2.5, length_scale=.5) if dname == "f32" else zk.Matern(nu=2.5, length_scale=.5, dtype=dtype)
        out = {}
        for m in (25, 50, 100):
            x1 = torch.linspace(0, 4, m, dtype=dtype)
            x2 = torch.linspace(-2, 2, m, dtype=dtype)
            xgrids = [x1, x2]
            vec = torch.randn(1, m * m, dtype=dtype)
            kernel = lambda x, y: kern.forward(x, y, params=(1, .1))
            res = {}
            for tag, prec in (("cg", False), ("pcg", True)):
                cnt = [0]

                def cb(n, x):
                    cnt[0] += 1
                r = toeplitz_expanded.gram_solve(xgrids, kernel, vec, do_precond=prec, tol=1e-10, maxiter=2000,
                                                 callback=cb, mult_RT=False)
                res[tag] = (r.numpy(), cnt[0])
            rt = toeplitz_expanded.gram_solve(xgrids, kernel, vec, do_precond=True, tol=1e-10, maxiter=2000,
                                              mult_RT=True)
            out["vec_%d" % m] = vec.numpy()
            out["x_cg_%d" % m], out["ncb_cg_%d" % m] = res["cg"]
            out["x_pcg_%d" % m], out["ncb_pcg_%d" % m] = res["pcg"]
            out["rt_pcg_%d" % m] = rt.numpy()
            print("cfg1", dname, m, "cg", res["cg"][1], "pcg", res["pcg"][1])
        np.savez_compressed(os.path.join(HERE, "cfg1_%s.npz" % dname), **out)


def make_kernels():
    for dname, dtype in DT.items():
        torch.manual_seed(7)
        out = {}
        g1 = torch.linspace(-.25, .25, 8, dtype=dtype)
        g2 = torch.linspace(-.25, .25, 6, dtype=dtype)
        g3 = torch.linspace(-.05, .05, 5, dtype=dtype)
        for D, grids in ((1, [g1]), (2, [g1, g2]), (3, [g1, g2, g3])):
            xxs = torch.meshgrid(*grids)
            u = torch.stack([x.reshape(-1) for x in xxs], dim=-1)
            lo = torch.tensor([g[0] for g in grids], dtype=dtype)
            hi = torch.tensor([g[-1] for g in grids], dtype=dtype)
            x = lo + (hi - lo) * torch.rand(7, D, dtype=dtype) * 1.1
            x[0] = u[3]                               # an observation exactly on a grid point
            out["grid_d%d" % D] = np.array([(float(g[0]), float(g[-1]), len(g)) for g in grids])
            out["x_d%d" % D] = x.numpy()
            sig2, ell = 0.8, 0.11
            for kname in ("sqexp", "matern12", "matern32", "matern52", "gneiting"):
                kern = get_kernel(kname, dtype)
                out["fwd_%s_d%d" % (kname, D)] = kern.forward(x, u, params=(sig2, ell)).numpy()
                out["diag_%s_d%d" % (kname, D)] = kern.diag(x, params=(sig2, ell)).numpy()
                if D > 1:
                    torch.manual_seed(99)
                    out["semimc_%s_d%d" % (kname, D)] = kern.k_semi_mc(u, x, (sig2, ell), npts=6).transpose(0, 1).numpy()
                    torch.manual_seed(99)
                    npts = 6
                    out["semimc_alphas"] = (torch.arange(npts, dtype=dtype) / npts
                                            + torch.rand(1, dtype=dtype) * (1. / npts)).numpy()
                    out["ddiag_%s_d%d" % (kname, D)] = kern.k_doubly_diag(x, (sig2, ell)).numpy()
                    xz = x.clone(); xz[1] = 0.
                    out["ddiag0_%s_d%d" % (kname, D)] = kern.k_doubly_diag(xz, (sig2, ell)).numpy()
                out["table_%s" % kname] = np.stack([kern.diag_interp.distance_grid.numpy(),
                                                    kern.diag_interp.slopes.numpy(),
                                                    kern.diag_interp.knn.numpy()])
            if D > 1:
                kern = get_kernel("sqexp", dtype)
                out["semi_sqexp_d%d" % D] = kern.k_semi(u, x, (sig2, ell)).transpose(0, 1).numpy()
                ellv = torch.tensor([0.11, 0.2, 0.07][:D], dtype=dtype)
                out["ellv_d%d" % D] = ellv.numpy()
                out["fwd_sqexp_ellv_d%d" % D] = kern.forward(x, u, params=(sig2, ellv)).numpy()
                out["fwd_gneiting_ellv_d%d" % D] = get_kernel("gneiting", dtype).forward(x, u, params=(sig2, ellv)).numpy()
                out["semi_sqexp_ellv_d%d" % D] = kern.k_semi(u, x, (sig2, ellv)).transpose(0, 1).numpy()
        # 1-D derivative kernels
        u = torch.linspace(0., 2., 9, dtype=dtype)
        x = 2 * torch.rand(5, dtype=dtype)
        out["deriv_u"] = u.numpy(); out["deriv_x"] = x.numpy()
        out["deriv_k"] = zd.k(x, u, 0.9, 0.3).numpy()
        out["deriv_kprime"] = zd.kprime(x, u, 0.9, 0.3).numpy()
        out["deriv_kprime_double_full"] = zd.kprime_double_full(x, u, 0.9, 0.3).numpy()
        out["deriv_kprime_double_1d"] = np.array(zd.kprime_double_1d(x, 0.9, 0.3))
        out["sig2_ell"] = np.array([0.8, 0.11])
        np.savez_compressed(os.path.join(HERE, "kernels_%s.npz" % dname), **out)
        print("kernels", dname)


def make_compute_kn():
    for dname, dtype in DT.items():
        out = {}
        for tag, kname, grids, integ, est in [
            ("point2d", "matern32", [(-5.7, 1.8, 14), (50., 55.5, 11)], False, None),
            ("semi3d", "sqexp", [(-.25, .25, 8), (-.25, .25, 7), (-.05, .05, 5)], True, "analytic"),
            ("mc3d", "matern52", [(-.25, .25, 8), (-.25, .25, 7), (-.05, .05, 5)], True, "mc-biased"),
        ]:
            torch.manual_seed(5)
            xgrids = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in grids]
            kern = get_kernel(kname, dtype)
            ell = 0.7 if tag == "point2d" else 0.08
            mod = zh.MeanFieldToeplitzGP(kern, xgrids, num_obs=100, sig2_init=0.9, ell_init=ell, dtype=dtype,
                                         jitter_val=1e-3)
            lo = torch.tensor([g[0] for g in grids], dtype=dtype)
            hi = torch.tensor([g[1] for g in grids], dtype=dtype)
            xb = lo + (hi - lo) * torch.rand(6, len(grids), dtype=dtype)
            torch.manual_seed(77)
            Knm, Knn = mod._make_grams(xb, integrated_obs=integ,
                                       semi_integrated_estimator=est or "analytic", semi_integrated_samps=5)
            torch.manual_seed(77)
            alphas = (torch.arange(5, dtype=dtype) / 5 + torch.rand(1, dtype=dtype) * (1. / 5))
            with torch.no_grad():
                kn = mod.compute_kn(Knm, maxiter_cg=20)
            out["%s_grids" % tag] = np.array(grids)
            out["%s_x" % tag] = xb.numpy()
            out["%s_Knm" % tag] = Knm.detach().numpy()
            out["%s_Knn" % tag] = Knn.detach().numpy()
            out["%s_kn" % tag] = kn.detach().numpy()
            out["%s_alphas" % tag] = alphas.numpy()
            out["%s_params" % tag] = np.array([float(mod.sig2), float(mod.ell), 1e-3])
            out["%s_table" % tag] = np.stack([kern.diag_interp.distance_grid.numpy(),
                                              kern.diag_interp.slopes.numpy(), kern.diag_interp.knn.numpy()])
            print("compute_kn", dname, tag, tuple(kn.shape))
        np.savez_compressed(os.path.join(HERE, "compute_kn_%s.npz" % dname), **out)


def make_svi_step():
    """MeanFieldToeplitzGP.elbo_and_grad / predict (hipgp.py:194-276,416-446) on a small 2-D problem."""
    for dname, dtype in DT.items():
        torch.manual_seed(11)
        grids = [(-5.7, 1.8, 14), (50., 55.5, 11)]
        xgrids = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in grids]
        kern = get_kernel("matern32", dtype)
        mod = zh.MeanFieldToeplitzGP(kern, xgrids, num_obs=500, sig2_init=0.9, ell_init=0.7, dtype=dtype, jitter_val=1e-3)
        lo = torch.tensor([g[0] for g in grids], dtype=dtype); hi = torch.tensor([g[1] for g in grids], dtype=dtype)
        xb = lo + (hi - lo) * torch.rand(8, 2, dtype=dtype)
        yb = torch.randn(8, 1, dtype=dtype)
        nb = 0.3 + 0.1 * torch.rand(8, 1, dtype=dtype)
        th1 = mod.global_theta1.data.clone(); th2 = mod.global_theta2.data.clone()
        elbo = mod.elbo_and_grad(xb, yb, nb, maxiter_cg=20)
        mu, sig = mod.predict(xb, maxiter_cg=50)
        np.savez_compressed(os.path.join(HERE, "svi_step_%s.npz" % dname), grids=np.array(grids), x=xb.numpy(), y=yb.numpy(),
                            noise_std=nb.numpy(), theta1=th1.numpy(), theta2=th2.numpy(), elbo=float(elbo),
                            g1=mod.global_theta1.grad.numpy(), g2=mod.global_theta2.grad.numpy(), mu=mu.numpy(), sig=sig.numpy(),
                            params=np.array([0.9, 0.7, 1e-3, 500]))
        print("svi_step", dname, float(elbo))


def make_learn_kernel():
    """Hyper-parameter gradients of the reference (hipgp.py:208-218, svi_gp.py:317-329) on a small 2-D problem, plus the
    gradient of sum(G * R^T v) with respect to the Toeplitz column (autograd through toeplitz_tensor.py:21-33,85-97)."""
    for dname, dtype in DT.items():
        out = {}
        for tag, kname, learn_noise in (("matern32", "matern32", False), ("sqexp_noise", "sqexp", True), ("matern52", "matern52", False)):
            torch.manual_seed(31)
            grids = [(-5.7, 1.8, 14), (50., 55.5, 11)]
            xgrids = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in grids]
            kern = get_kernel(kname, dtype)
            mod = zh.MeanFieldToeplitzGP(kern, xgrids, num_obs=500, sig2_init=0.9, ell_init=0.7, noise2_init=0.2, dtype=dtype, jitter_val=1e-3,
                                         learn_kernel=True, learn_noise=learn_noise)
            lo = torch.tensor([g[0] for g in grids], dtype=dtype); hi = torch.tensor([g[1] for g in grids], dtype=dtype)
            xb = lo + (hi - lo) * torch.rand(8, 2, dtype=dtype)
            yb = torch.randn(8, 1, dtype=dtype)
            nb = None if learn_noise else 0.3 + 0.1 * torch.rand(8, 1, dtype=dtype)
            th1 = mod.global_theta1.data.clone(); th2 = mod.global_theta2.data.clone()
            elbo = mod.elbo_and_grad(xb, yb, nb, maxiter_cg=60)
            (-elbo).backward()
            out[tag + "_grids"] = np.array(grids); out[tag + "_x"] = xb.numpy(); out[tag + "_y"] = yb.numpy()
            if nb is not None:
                out[tag + "_noise_std"] = nb.numpy()
            out[tag + "_theta1"] = th1.numpy(); out[tag + "_theta2"] = th2.numpy(); out[tag + "_elbo"] = float(elbo)
            out[tag + "_g_log_sig2"] = float(mod.log_sig2.grad); out[tag + "_g_log_ell"] = float(mod.log_ell.grad)
            if learn_noise:
                out[tag + "_g_log_noise2"] = float(mod.log_noise2.grad)
            out[tag + "_g1"] = mod.global_theta1.grad.detach().numpy(); out[tag + "_g2"] = mod.global_theta2.grad.detach().numpy()
            out[tag + "_params"] = np.array([0.9, 0.7, 0.2, 1e-3, 500])
            print("learn_kernel", dname, tag, float(elbo), float(mod.log_sig2.grad), float(mod.log_ell.grad))
        # R^T column gradient alone, 2-D and 3-D, with clamped eigenvalues in the SqExp case
        for tag, grids, kname, sig2, ell in (("rt2d", [(0., 1., 9), (0., 2., 12)], "matern32", 1.2, 0.4),
                                             ("rt3d", [(0., 1., 5), (0., 1., 4), (0., 2., 6)], "sqexp", 0.8, 0.5)):
            torch.manual_seed(32)
            xgrids = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in grids]
            kern = get_kernel(kname, dtype)
            kfun = lambda x, y: kern.forward(x, y, params=(sig2, ell))
            tt = ToeplitzTensor(xgrids=xgrids, kernel=kfun, batch_shape=None, jitter_val=1e-3)
            col = tt.column.detach().clone().requires_grad_(True)
            # rebuild the spectrum from a column that is on the tape, exactly as toeplitz_tensor.py:19-33 does
            C = tt.circulant_embed(col.view(tt.dims)); Cc = tt.make_complex(C)
            D = torch.fft(Cc, signal_ndim=tt.ndim)
            D0 = D[..., 0].clamp(min=1e-6)
            tt.D_sqrt = torch.stack([torch.sqrt(D0), torch.zeros_like(D0)], dim=-1)
            M = int(np.prod(tt.dims)); E = int(np.prod(tt.C.shape))
            v = torch.randn(3, M, dtype=dtype); G = torch.randn(3, E, dtype=dtype)
            tt.set_batch_shape((3,))
            y = tt._matmul_by_RT(v)
            (y * G).sum().backward()
            out[tag + "_grids"] = np.array(grids); out[tag + "_column"] = tt.column.detach().numpy(); out[tag + "_v"] = v.numpy()
            out[tag + "_G"] = G.numpy(); out[tag + "_gcol"] = col.grad.numpy(); out[tag + "_nclamped"] = int((D[..., 0] < 1e-6).sum())
            print("rt column grad", dname, tag, "clamped", out[tag + "_nclamped"], float(col.grad.norm()))
        np.savez_compressed(os.path.join(HERE, "learn_kernel_%s.npz" % dname), **out)


def make_bidiag():
    """bidiag_solve (bidiag.py:129-148) with A = R^T, A* = R of ToeplitzMatmul (toeplitz_expanded.py:163-187)."""
    from ziggy.misc import bidiag as zb
    for dname, dtype in DT.items():
        out = {}
        for tag, grids, kname, sig2, ell, nobs, max_iter in (("g1d", [(0., 5., 60)], "matern52", 0.1, 0.4, 3, 25),
                                                             ("g2d", [(0., 1., 9), (0., 2., 7)], "matern32", 1.0, 0.5, 2, 20)):
            torch.manual_seed(41)
            xgrids = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in grids]
            kern = get_kernel(kname, dtype)
            kfun = lambda x, y: kern.forward(x, y, params=(sig2, ell))
            M = int(np.prod([g[2] for g in grids])); Mp = int(np.prod([2 * g[2] - 2 for g in grids]))
            b = torch.randn(M, nobs, dtype=dtype)
            K_matmul = toeplitz_expanded.ToeplitzMatmul(xgrids, kfun, batch_shape=b.shape[-1:])
            A_matmul = lambda x: K_matmul(x.t(), multiply_type="RTv").t()
            Astar_matmul = lambda x: K_matmul(x.t(), multiply_type="Rv").t()
            U, V, al, be = zb.golub_kahan_bidiag(A_matmul, Astar_matmul, (Mp, M), max_iter, dtype, b.device, b, tol=1e-5, run_all=True)
            c = zb.bidiag_solve(A_matmul, Astar_matmul, (Mp, M), max_iter, dtype, b.device, b, tol=1e-5)
            out[tag + "_grids"] = np.array(grids); out[tag + "_params"] = np.array([sig2, ell, max_iter]); out[tag + "_b"] = b.numpy()
            out[tag + "_c"] = c.numpy(); out[tag + "_alphas"] = al.numpy(); out[tag + "_betas"] = be.numpy(); out[tag + "_V"] = V.numpy()
            print("bidiag", dname, tag, "J", al.shape[0], float(c.norm()))
        np.savez_compressed(os.path.join(HERE, "bidiag_%s.npz" % dname), **out)


def make_quadform():
    """sym_toeplitz_derivative_quadratic_form on seeded vectors, and autograd through the reference's InvMatmul."""
    from ziggy.misc.gpt_toeplitz import sym_toeplitz_derivative_quadratic_form as quad
    for dname, dtype in DT.items():
        torch.manual_seed(99)
        out = {}
        for tag, dims, S in (("1d", (100,), 3), ("2d", (17, 40), 3), ("3d", (6, 9, 12), 2), ("2d_odd", (5, 3), 4)):
            M = int(np.prod(dims))
            u = torch.randn(S, M, dtype=dtype); v = torch.randn(S, M, dtype=dtype)
            out[tag + "_dims"] = np.array(dims); out[tag + "_u"] = u.numpy(); out[tag + "_v"] = v.numpy()
            out[tag + "_quad"] = quad(u.t().contiguous(), v.t().contiguous()).numpy()
        # InvMatmul.backward on the 2d_17x40_matern32 Toeplitz case
        grids, kname, sig2, ell, jitter, B = TOEPLITZ_CASES["2d_17x40_matern32"]
        xgrids = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in grids]
        kern = get_kernel(kname, dtype)
        tt = ToeplitzTensor(xgrids, lambda x, y: kern.forward(x, y, params=(sig2, ell)), batch_shape=None, jitter_val=jitter)
        tt.column.requires_grad_(True)
        Rt = torch.randn(B, int(tt.M), dtype=dtype, requires_grad=True)
        wts = torch.randn(B, int(tt.M), dtype=dtype)
        maxiter, tol = 60, (1e-12 if dname == "f64" else 1e-6)
        sol = tt.inv_matmul(Rt, do_precond=True, maxiter=maxiter, tol=tol)
        (sol * wts).sum().backward()
        out.update(bw_R=Rt.detach().numpy(), bw_w=wts.numpy(), bw_solves=sol.detach().numpy(),
                   bw_column_grad=tt.column.grad.numpy(), bw_right_grad=Rt.grad.numpy(), bw_maxiter=maxiter, bw_tol=tol)
        np.savez_compressed(os.path.join(HERE, "quadform_%s.npz" % dname), **out)
        print("quadform", dname, {k: np.asarray(v).shape for k, v in out.items() if k.endswith("quad") or k.startswith("bw_c")})


def make_block_step():
    """BlockToeplitzGP natural-gradient step / predict and its block helpers on a small 2-D problem; index maps in 3-D."""
    from ziggy.misc import util as zutil
    for dname, dtype in DT.items():
        torch.manual_seed(21)
        grids = [(-5.7, 1.8, 14), (50., 55.5, 11)]
        xgrids = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in grids]
        kern = get_kernel("matern32", dtype)
        mod = zh.BlockToeplitzGP(kern, xgrids, num_obs=500, block_sizes=[13, 5], sig2_init=0.9, ell_init=0.7, dtype=dtype,
                                 jitter_val=1e-3)
        # a non-trivial (symmetric negative definite) theta2 so that the block algebra is exercised
        A = 0.05 * torch.randn(mod.num_blocks, mod.block_size, mod.block_size, dtype=dtype)
        mod.global_theta2.data = mod.global_theta2.data - A.matmul(A.transpose(-1, -2))
        lo = torch.tensor([g[0] for g in grids], dtype=dtype); hi = torch.tensor([g[1] for g in grids], dtype=dtype)
        xb = lo + (hi - lo) * torch.rand(8, 2, dtype=dtype)
        yb = torch.randn(8, 1, dtype=dtype)
        nb = 0.3 + 0.1 * torch.rand(8, 1, dtype=dtype)
        th1 = mod.global_theta1.data.clone(); th2 = mod.global_theta2.data.clone()
        elbo = mod.elbo_and_grad(xb, yb, nb, maxiter_cg=20)
        mu, sig = mod.predict(xb, maxiter_cg=50)
        with torch.no_grad():
            Knm, _ = mod._make_grams(xb)
            kn = mod.compute_kn(Knm, maxiter_cg=20)
            qm, qS = mod.standard_variational_params()
            lam = mod.get_lam(1 / nb ** 2, kn, bscale=500 / 8)
            Sv = mod.block_diag_multiply(qS, kn)
            knSkn = mod.compute_knSkn(kn, qS)
            kl = mod.get_kl_to_prior(qm, qS)
        idx3, _, _ = zutil.define_block_chunks([torch.arange(6), torch.arange(10), torch.arange(14)], [3, 5, 7])
        np.savez_compressed(os.path.join(HERE, "block_step_%s.npz" % dname), grids=np.array(grids), x=xb.numpy(), y=yb.numpy(),
                            noise_std=nb.numpy(), theta1=th1.numpy(), theta2=th2.numpy(), elbo=float(elbo),
                            g1=mod.global_theta1.grad.numpy(), g2=mod.global_theta2.grad.numpy(), mu=mu.numpy(), sig=sig.numpy(),
                            params=np.array([0.9, 0.7, 1e-3, 500]), block_sizes=np.array([13, 5]),
                            block_idx=mod.block_idx.numpy(), kn=kn.numpy(), qm=qm.numpy(), qS=qS.numpy(), lam=lam.numpy(),
                            Sv=Sv.numpy(), knSkn=knSkn.numpy(), kl=float(kl), block_idx_3d=idx3.numpy())
        print("block_step", dname, float(elbo), mod.block_idx.shape)


def make_notebook_counts():
    """Saved cell outputs of experiments-hip-gp/preconditioner-analysis.ipynb -- the only numbers the
    reference repo pins (unseeded RNG there => reproducible to a few iterations only)."""
    Ms = [10, 20, 40, 80, 100, 200, 300, 400, 500]
    np.savez(os.path.join(HERE, "notebook_counts.npz"), Ms=np.array(Ms),
             sqexp_cg=[2, 11, 55, 2000, 2000, 2000, 2000, 2000, 2000], sqexp_pcg=[1, 2, 4, 39, 42, 67, 87, 100, 102],
             matern52_cg=[3, 11, 37, 177, 319, 2000, 2000, 2000, 2000], matern52_pcg=[1, 2, 3, 6, 6, 12, 17, 25, 41],
             matern32_cg=[4, 11, 32, 104, 156, 591, 1327, 2000, 2000], matern32_pcg=[1, 2, 3, 4, 5, 6, 8, 9, 11],
             matern12_cg=[5, 11, 23, 45, 56, 111, 168, 224, 282], matern12_pcg=[1, 2, 3, 3, 3, 3, 3, 3, 4])


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "svi":
        make_svi_step()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "block":
        make_block_step()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "bidiag":
        make_bidiag()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "learn_kernel":
        make_learn_kernel()
        sys.exit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "quadform":
        make_quadform()
        sys.exit(0)
    make_notebook_counts()
    make_svi_step()
    make_toeplitz()
    make_kernels()
    make_compute_kn()
    make_cfg1()
    make_quadform()
    make_block_step()
    make_learn_kernel()
    make_bidiag()
