"""The UNMODIFIED reference running on top of the CUDA drop-ins (SURVEY.md section 8b: "the ziggy Python API stays a drop-in").

`hipgp_b200.install_as_ziggy()` registers this package's modules under the reference's module names; the reference's OWN
callers are then imported from the staged copy `oracle/_ref/ziggy` (oracle/make_ref.py; byte-identical to the reference
checkout, git-ignored; skipped where it is not staged):

  * `ziggy.hipgp.MeanFieldToeplitzGP` / `BlockToeplitzGP` (hipgp.py:449-690): `elbo_and_grad` + `predict` against the golden
    vectors generated from the reference running on its own torch implementation (tests/golden/make_golden.py);
  * `ziggy.misc.bidiag` (bidiag.py:5-148, unchanged) over the drop-in ToeplitzMatmul's R^T / R matvecs;
  * the body of `experiments-hip-gp/run_solve_kn_experiment.py:27-73` (config 1: seeded vectors, CG then PCG through
    `toeplitz_expanded.gram_solve`, callback counts 28/196/1978 and 6/19/89 in fp32).

Each case runs in a subprocess: the module substitution must happen before `ziggy` is imported and must not leak into the
other tests of this process."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.path.join(ROOT, "oracle", "_ref")

PRELUDE = r'''
import os, sys, types
sys.path.insert(0, %(root)r)
import numpy as np, torch
# the reference imports pyprind (progress bar) and calls torch.solve; nothing else of the legacy shim is needed because the
# FFT call sites live in the modules that are being replaced
if "pyprind" not in sys.modules:
    m = types.ModuleType("pyprind"); m.prog_bar = lambda it, *a, **k: it; sys.modules["pyprind"] = m
if not hasattr(torch, "solve"):
    torch.solve = lambda B, A: (torch.linalg.solve(A, B), None)
import hipgp_b200
hipgp_b200.install_as_ziggy()
sys.path.insert(0, %(ref)r)
import ziggy
assert os.path.realpath(os.path.dirname(ziggy.__file__)).startswith(os.path.realpath(%(ref)r)), ziggy.__file__
import ziggy.misc.toeplitz_tensor as ztt, ziggy.misc.toeplitz_expanded as zte, ziggy.kernels as zk
assert ztt.__name__.startswith("hipgp_b200") and zte.__name__.startswith("hipgp_b200") and zk.__name__.startswith("hipgp_b200")
GOLD = os.path.join(%(root)r, "tests", "golden")
DT = {"f32": torch.float32, "f64": torch.float64}
def relerr(a, b):
    if isinstance(a, torch.Tensor): a = a.detach().cpu().numpy()
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)
'''

MEANFIELD = PRELUDE + r'''
from ziggy import hipgp as zh                       # the reference's own model classes
assert zh.__file__.startswith(os.path.realpath(%(ref)r)) or os.path.realpath(zh.__file__).startswith(os.path.realpath(%(ref)r))
for dname in ("f64", "f32"):
    g = np.load(os.path.join(GOLD, "svi_step_%%s.npz" %% dname)); dtype = DT[dname]
    tol = 1e-6 if dname == "f64" else 2e-3
    xg = [torch.linspace(lo, hi, int(m), dtype=dtype) for lo, hi, m in g["grids"]]
    mod = zh.MeanFieldToeplitzGP(zk.Matern(nu=1.5, dtype=dtype), xg, num_obs=int(g["params"][3]), sig2_init=float(g["params"][0]),
                                 ell_init=float(g["params"][1]), dtype=dtype, jitter_val=float(g["params"][2]))
    mod.global_theta1.data.copy_(torch.from_numpy(g["theta1"])); mod.global_theta2.data.copy_(torch.from_numpy(g["theta2"]))
    mod = mod.cuda_params(0)
    x = torch.from_numpy(g["x"]).cuda(); y = torch.from_numpy(g["y"]).cuda(); nb = torch.from_numpy(g["noise_std"]).cuda()
    elbo = mod.elbo_and_grad(x, y, nb, maxiter_cg=20)
    assert abs(float(elbo) - float(g["elbo"])) <= tol * abs(float(g["elbo"])), (dname, float(elbo), float(g["elbo"]))
    assert relerr(mod.global_theta1.grad, g["g1"]) < tol and relerr(mod.global_theta2.grad, g["g2"]) < tol
    mu, sig = mod.predict(x, maxiter_cg=50)
    assert relerr(mu, g["mu"]) < tol and relerr(sig, g["sig"]) < tol, (dname, relerr(mu, g["mu"]), relerr(sig, g["sig"]))
print("DROPIN_OK")
'''

BLOCK = PRELUDE + r'''
from ziggy import hipgp as zh
for dname in ("f64", "f32"):
    g = np.load(os.path.join(GOLD, "block_step_%%s.npz" %% dname)); dtype = DT[dname]
    tol = 1e-6 if dname == "f64" else 2e-3
    xg = [torch.linspace(lo, hi, int(m), dtype=dtype) for lo, hi, m in g["grids"]]
    mod = zh.BlockToeplitzGP(zk.Matern(nu=1.5, dtype=dtype), xg, num_obs=int(g["params"][3]), block_sizes=[int(b) for b in g["block_sizes"]],
                             sig2_init=float(g["params"][0]), ell_init=float(g["params"][1]), dtype=dtype, jitter_val=float(g["params"][2]))
    assert np.array_equal(mod.block_idx.numpy(), g["block_idx"])
    mod.global_theta1.data.copy_(torch.from_numpy(g["theta1"])); mod.global_theta2.data.copy_(torch.from_numpy(g["theta2"]))
    mod = mod.cuda_params(0)
    x = torch.from_numpy(g["x"]).cuda(); y = torch.from_numpy(g["y"]).cuda(); nb = torch.from_numpy(g["noise_std"]).cuda()
    elbo = mod.elbo_and_grad(x, y, nb, maxiter_cg=20)
    assert abs(float(elbo) - float(g["elbo"])) <= tol * abs(float(g["elbo"])), (dname, float(elbo), float(g["elbo"]))
    assert relerr(mod.global_theta1.grad, g["g1"]) < tol and relerr(mod.global_theta2.grad, g["g2"]) < tol
    mu, sig = mod.predict(x, maxiter_cg=50)
    assert relerr(mu, g["mu"]) < tol and relerr(sig, g["sig"]) < tol
print("DROPIN_OK")
'''

SOLVE_KN = PRELUDE + r'''
# experiments-hip-gp/run_solve_kn_experiment.py:27-73, the reference script's own call pattern (its plotting tail needs
# matplotlib / seaborn, which are not installed): seed once, three grids in order, CG then PCG through gram_solve
from ziggy.kernels import Matern
from ziggy.misc import toeplitz_expanded
src = open(os.path.join(%(ref)r, "experiments-hip-gp", "run_solve_kn_experiment.py")).read()
assert "toeplitz_expanded.gram_solve(xgrids, kernel, vec," in src and "torch.manual_seed(42)" in src
device = torch.device("cuda")
for dname, want_cg, want_pcg in (("f32", (28, 196, 1978), (6, 19, 89)), ("f64", None, None)):
    g = np.load(os.path.join(GOLD, "cfg1_%%s.npz" %% dname)); dtype = DT[dname]
    kern = Matern(nu=2.5, length_scale=.5) if dname == "f32" else Matern(nu=2.5, length_scale=.5, dtype=dtype)
    for i, m in enumerate((25, 50, 100)):
        x1 = torch.linspace(0, 4, m, device=device, dtype=dtype); x2 = torch.linspace(-2, 2, m, device=device, dtype=dtype)
        xgrids = [x1, x2]
        vec = torch.from_numpy(g["vec_%%d" %% m]).to(device)      # = torch.randn(1, M) after manual_seed(42) on the CPU generator
        kernel = lambda x, y: kern.forward(x, y, params=(1, .1))
        res = {}
        for tag, prec in (("cg", False), ("pcg", True)):
            xs = []
            r = toeplitz_expanded.gram_solve(xgrids, kernel, vec, do_precond=prec, tol=1e-10, maxiter=2000,
                                             callback=lambda n, x: xs.append(n), mult_RT=False)
            res[tag] = (r, len(xs))
        ncg, npcg = int(g["ncb_cg_%%d" %% m]), int(g["ncb_pcg_%%d" %% m])
        if want_cg is not None:
            assert (ncg, npcg) == (want_cg[i], want_pcg[i])
        # same bars as tests/test_gpu_api.py::test_cfg1_gram_solve: fp64 counts within max(1, 2 %%) and iterates to 1e-6; fp32 counts
        # in a band (the count is decided by when the recurrence residual underflows tol while the true residual has stalled)
        if dname == "f64":
            for tag, want in (("cg", ncg), ("pcg", npcg)):
                assert abs(res[tag][1] - want) <= max(1, int(0.02 * want)), (dname, m, tag, res[tag][1], want)
                assert relerr(res[tag][0], g["x_%%s_%%d" %% (tag, m)]) < 1e-6
        else:
            for tag, want in (("cg", ncg), ("pcg", npcg)):
                assert abs(res[tag][1] - want) <= max(2, int(0.25 * want)), (dname, m, tag, res[tag][1], want)
        rt = toeplitz_expanded.gram_solve(xgrids, kernel, vec, do_precond=True, tol=1e-10, maxiter=2000, mult_RT=True)
        assert tuple(rt.shape) == (1, (2 * m - 2) ** 2)
        assert relerr(rt, g["rt_pcg_%%d" %% m]) < (1e-6 if dname == "f64" else 5e-2)
print("DROPIN_OK")
'''


BIDIAG = PRELUDE + r'''
# SURVEY.md 8f rank 4: the Golub-Kahan bidiagonalisation route to K^{-1/2} b (ziggy/misc/bidiag.py:5-148) is generic host
# code over two matvec closures; it runs UNCHANGED (imported from the staged reference) on the structured CUDA matvecs
# R^T / R of the drop-in ToeplitzMatmul, closures as in run_pcg_vs_cholesky.py:105-108.
from ziggy.misc import bidiag as zb
assert os.path.realpath(zb.__file__).startswith(os.path.realpath(%(ref)r))
for dname in ("f64", "f32"):
    g = np.load(os.path.join(GOLD, "bidiag_%%s.npz" %% dname)); dtype = DT[dname]
    for tag, kern in (("g1d", zk.Matern(nu=2.5, dtype=dtype)), ("g2d", zk.Matern(nu=1.5, dtype=dtype))):
        sig2, ell, max_iter = [float(t) for t in g[tag + "_params"]]
        xgrids = [torch.linspace(lo, hi, int(m), dtype=dtype, device="cuda") for lo, hi, m in g[tag + "_grids"]]
        kfun = lambda x, y: kern.forward(x, y, params=(sig2, ell))
        b = torch.from_numpy(g[tag + "_b"]).cuda()
        M = b.shape[0]; Mp = int(np.prod([2 * len(x) - 2 for x in xgrids]))
        K_matmul = zte.ToeplitzMatmul(xgrids, kfun, batch_shape=b.shape[-1:])
        A_matmul = lambda x: K_matmul(x.t(), multiply_type="RTv").t()
        Astar_matmul = lambda x: K_matmul(x.t(), multiply_type="Rv").t()
        U, V, al, be = zb.golub_kahan_bidiag(A_matmul, Astar_matmul, (Mp, M), int(max_iter), dtype, b.device, b, tol=1e-5, run_all=True)
        c = zb.bidiag_solve(A_matmul, Astar_matmul, (Mp, M), int(max_iter), dtype, b.device, b, tol=1e-5)
        assert tuple(c.shape) == tuple(g[tag + "_c"].shape) and al.shape[0] == g[tag + "_alphas"].shape[0]
        if dname == "f64":
            assert relerr(al, g[tag + "_alphas"]) < 1e-8 and relerr(be, g[tag + "_betas"]) < 1e-8, (tag, relerr(al, g[tag + "_alphas"]))
            assert relerr(V, g[tag + "_V"]) < 1e-6 and relerr(c, g[tag + "_c"]) < 1e-6, (tag, relerr(c, g[tag + "_c"]))
        else:           # fp32: the Krylov basis loses digits with every re-orthogonalisation; the leading coefficients pin the matvecs
            assert relerr(al[:5], g[tag + "_alphas"][:5]) < 1e-4 and relerr(be[:5], g[tag + "_betas"][:5]) < 1e-3
            assert bool(torch.isfinite(c).all())
print("DROPIN_OK")
'''


def _run(script):
    if not os.path.isdir(os.path.join(REF, "ziggy")):
        pytest.skip("oracle/_ref not staged: needs the reference checkout (python oracle/make_ref.py)")
    r = subprocess.run([sys.executable, "-c", script % {"root": ROOT, "ref": REF}], capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "DROPIN_OK" in r.stdout, r.stdout[-3000:] + r.stderr[-6000:]


def test_reference_meanfield_model_on_cuda_dropins():
    _run(MEANFIELD)


def test_reference_block_model_on_cuda_dropins():
    _run(BLOCK)


def test_reference_solve_kn_experiment_on_cuda_dropins():
    _run(SOLVE_KN)


def test_reference_bidiag_solver_on_cuda_matvecs():
    _run(BIDIAG)
