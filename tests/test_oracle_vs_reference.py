"""Comparison of the CPU oracle (oracle/ziggy_oracle.py) with the UNMODIFIED reference on fresh seeds / shapes: always
against the stored outputs of those cases (tests/golden/fresh_oracle_vs_reference.npz, tests/golden/make_fresh_golden.py),
and live wherever the reference tree is reachable (the reference checkout oracle/make_ref.py locates, or the staged byte-identical
copy oracle/_ref, oracle/make_ref.py).  The live run is a subprocess so the legacy-API shim (oracle/ref_shim.py patches
torch.fft) never leaks into the other tests of this process."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SCRIPT = r'''
import sys
sys.path.insert(0, %(root)r)
import numpy as np, torch
from oracle import ref_shim
ref_shim.import_reference()
from ziggy.misc.toeplitz_tensor import ToeplitzTensor
from ziggy.misc import toeplitz_expanded
from ziggy import kernels as zk, hipgp as zh
from oracle import ziggy_oracle as zo

torch.manual_seed(20261018)
for dtype in (torch.float32, torch.float64):
    for dims, nu, ell in (((19, 23), 1.5, 0.4), ((7, 5, 9), 2.5, 0.6), ((31,), 0.5, 0.2)):
        xg = [torch.linspace(-1.0 - d, 2.0 + 0.5 * d, m, dtype=dtype) for d, m in enumerate(dims)]
        kern = zk.Matern(nu=nu, length_scale=ell, dtype=dtype)
        kfun = lambda x, y: kern.forward(x, y, params=(1.3, ell))
        ofun = lambda x, y: zo.matern(x, y, 1.3, ell, nu)
        ref = ToeplitzTensor(xgrids=xg, kernel=kfun, batch_shape=None, jitter_val=2e-3)
        ora = zo.OracleToeplitz(xg, ofun, jitter_val=2e-3)
        M = int(np.prod(dims)); E = int(np.prod(ref.C.shape))
        v = torch.randn(3, M, dtype=dtype); w = torch.randn(3, E, dtype=dtype)
        assert torch.equal(ref.column, ora.column) and torch.equal(ref.D, ora.D)
        ref.set_batch_shape((3,))
        for a, b in ((ref._matmul_by_K(v), ora.matmul_K(v)), (ref._matmul_by_Cinv(v), ora.matmul_Cinv(v)),
                     (ref._matmul_by_RT(v), ora.matmul_RT(v)), (ref._matmul_by_R(w), ora.matmul_R(w))):
            assert torch.equal(a, b), (dtype, dims)
        calls = [[], []]
        xr = ref._solve(v, do_precond=True, maxiter=40, tol=1e-9, callback=lambda n, x: calls[0].append(n))
        xo = ora.solve(v, do_precond=True, maxiter=40, tol=1e-9, callback=lambda n, x: calls[1].append(n))
        assert calls[0] == calls[1] and torch.equal(xr, xo), (dtype, dims)
        if len(dims) > 1:
            res = toeplitz_expanded.gram_solve(xg, kfun, v[:1], do_precond=True, tol=1e-9, maxiter=60, mult_RT=True)
            reso = zo.gram_solve(xg, ofun, v[:1], do_precond=True, tol=1e-9, maxiter=60, mult_RT=True)
            assert torch.equal(res, reso), (dtype, dims)
# one mean-field natural-gradient step of the reference's own model class against the oracle's restatement
dtype = torch.float64
grids = [(-2.0, 1.0, 9), (10.0, 12.5, 12)]
xg = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in grids]
kern = zk.Matern(nu=1.5, length_scale=0.6, dtype=dtype)
mod = zh.MeanFieldToeplitzGP(kern, xg, num_obs=300, sig2_init=0.8, ell_init=0.6, dtype=dtype, jitter_val=1e-3, learn_kernel=False)
lo = torch.tensor([g[0] for g in grids], dtype=dtype); hi = torch.tensor([g[1] for g in grids], dtype=dtype)
xb = lo + (hi - lo) * torch.rand(6, 2, dtype=dtype); yb = torch.randn(6, 1, dtype=dtype); nb = 0.2 + 0.1 * torch.rand(6, 1, dtype=dtype)
th1 = mod.global_theta1.data.clone(); th2 = mod.global_theta2.data.clone()
elbo = mod.elbo_and_grad(xb, yb, nb, maxiter_cg=15)
xin = zo.meshgrid_points(xg)
kfun = lambda x, y: zo.matern(x, y, 0.8, 0.6, 1.5)
Knm = kfun(xb, xin); Knn = torch.full((6,), 0.8, dtype=dtype)
e2, g1, g2 = zo.meanfield_elbo_and_grad(xg, kfun, Knm, Knn, yb, nb, th1, th2, 300, maxiter_cg=15, jitter_val=1e-3)
assert abs(float(elbo) - float(e2)) < 1e-12 * abs(float(e2)), (float(elbo), float(e2))
assert (mod.global_theta1.grad - g1).abs().max() < 1e-12 * g1.abs().max()
assert (mod.global_theta2.grad - g2).abs().max() < 1e-12 * g2.abs().max()
print("ORACLE_VS_REFERENCE_OK")
'''


def _compare_with_stored_fresh_cases():
    """the oracle on the stored inputs of the fresh cases: bit for bit, the mean-field step to 1e-12 relative"""
    import torch
    from oracle import ziggy_oracle as zo
    sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
    import make_fresh_golden as mf
    g = np.load(mf.OUT)
    for dname, dtype in mf.DT.items():
        for dims, nu, ell in mf.CASES:
            t = mf.case_tag(dname, dims)
            xg = mf.grids(dims, dtype)
            ofun = lambda x, y: zo.matern(x, y, 1.3, ell, nu)
            ora = zo.OracleToeplitz(xg, ofun, jitter_val=2e-3)
            v = torch.from_numpy(g[t + "_v"]); w = torch.from_numpy(g[t + "_w"])
            assert np.array_equal(ora.column.numpy(), g[t + "_column"]) and np.array_equal(ora.D.numpy(), g[t + "_D"]), t
            for got, key in ((ora.matmul_K(v), "_Kv"), (ora.matmul_Cinv(v), "_Cinv_v"), (ora.matmul_RT(v), "_RT_v"), (ora.matmul_R(w), "_R_w")):
                assert np.array_equal(got.numpy(), g[t + key]), (t, key)
            calls = []
            x = ora.solve(v, do_precond=True, maxiter=40, tol=1e-9, callback=lambda n, xx: calls.append(n))
            assert calls == g[t + "_calls"].tolist() and np.array_equal(x.numpy(), g[t + "_solve"]), t
            if len(dims) > 1:
                rt = zo.gram_solve(xg, ofun, v[:1], do_precond=True, tol=1e-9, maxiter=60, mult_RT=True)
                assert np.array_equal(rt.numpy(), g[t + "_gram_rt"]), t
    dtype = torch.float64
    xg = [torch.linspace(lo, hi, m, dtype=dtype) for lo, hi, m in mf.MF_GRIDS]
    kfun = lambda x, y: zo.matern(x, y, 0.8, 0.6, 1.5)
    xb = torch.from_numpy(g["mf_x"])
    Knm = kfun(xb, zo.meshgrid_points(xg)); Knn = torch.full((xb.shape[0],), 0.8, dtype=dtype)
    e2, g1, g2 = zo.meanfield_elbo_and_grad(xg, kfun, Knm, Knn, torch.from_numpy(g["mf_y"]), torch.from_numpy(g["mf_noise_std"]),
                                            torch.from_numpy(g["mf_theta1"]), torch.from_numpy(g["mf_theta2"]), 300, maxiter_cg=15,
                                            jitter_val=1e-3)
    elbo = float(g["mf_elbo"])
    assert abs(float(e2) - elbo) < 1e-12 * abs(elbo), (float(e2), elbo)
    assert np.abs(g1.numpy() - g["mf_g1"]).max() < 1e-12 * np.abs(g["mf_g1"]).max()
    assert np.abs(g2.numpy() - g["mf_g2"]).max() < 1e-12 * np.abs(g["mf_g2"]).max()


def test_oracle_matches_live_reference_on_fresh_inputs():
    sys.path.insert(0, ROOT)
    _compare_with_stored_fresh_cases()
    from oracle import ref_shim
    if ref_shim.reference_root() is None:
        return                     # the live run needs the reference tree; the stored comparison above has run
    r = subprocess.run([sys.executable, "-c", SCRIPT % {"root": ROOT}], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ORACLE_VS_REFERENCE_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


def test_staged_reference_is_unmodified():
    """oracle/_ref is byte-identical to the reference it was staged from."""
    sys.path.insert(0, ROOT)
    from oracle import make_ref
    if not os.path.isdir(os.path.join(make_ref.DST, "ziggy")):
        pytest.skip("oracle/_ref not staged")
    assert make_ref.verify() == []
    if make_ref.SRC and os.path.isdir(os.path.join(make_ref.SRC, "ziggy")):
        import hashlib
        for root, _d, files in os.walk(os.path.join(make_ref.SRC, "ziggy")):
            for f in files:
                if f.endswith(".py"):
                    p = os.path.join(root, f)
                    q = os.path.join(make_ref.DST, os.path.relpath(p, make_ref.SRC))
                    assert hashlib.sha256(open(p, "rb").read()).hexdigest() == hashlib.sha256(open(q, "rb").read()).hexdigest(), q


def test_install_as_ziggy_binds_the_dropins_into_the_reference_package():
    """hipgp_b200.install_as_ziggy(): the reference's own ziggy/hipgp.py imports this package's ToeplitzTensor, and all three
    import spellings used by the reference and its experiment scripts resolve to the drop-ins (no GPU needed: imports only)."""
    sys.path.insert(0, ROOT)
    from oracle import ref_shim
    root = ref_shim.reference_root()
    if root is None:
        pytest.skip("reference tree not present")
    code = r'''
import sys, types
sys.path.insert(0, %r)
m = types.ModuleType("pyprind"); m.prog_bar = lambda it, *a, **k: it; sys.modules["pyprind"] = m
import hipgp_b200
hipgp_b200.install_as_ziggy()
sys.path.insert(0, %r)
import ziggy.misc.toeplitz_tensor as ztt
from ziggy.misc import toeplitz_expanded, cg, _inv_matmul
from ziggy import kernels as zk
from ziggy import hipgp as zh, svi_gp
from ziggy.misc import util, stats                      # stay the reference's own
for mod in (ztt, toeplitz_expanded, cg, _inv_matmul, zk):
    assert mod.__name__.startswith("hipgp_b200"), mod.__name__
assert zh.ToeplitzTensor is ztt.ToeplitzTensor and zh.__name__ == "ziggy.hipgp" and util.__name__ == "ziggy.misc.util"
assert zh.MeanFieldToeplitzGP.__module__ == "ziggy.hipgp"
print("BOUND_OK")
''' % (ROOT, root)
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "BOUND_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
