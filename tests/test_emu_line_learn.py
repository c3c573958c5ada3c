"""CPU execution (g++ -DHIPGP_EMU build, tests/emu_build.py) of the hyper-parameter derivatives of line-integral observations:

  hipgp_kxu_param_grad, mode SEMI_ANALYTIC   d/d(sig2, ell_d) of sum G * K_xu for the analytic SqExp line integral
  hipgp_doubly_diag_param_grad               d/d(sig2, ell) of sum g * K_nn for the interpolated doubly integrated diagonal

checked against fp64 CPU-torch autograd through the oracle's formulas (oracle.semi_integrated_sqe, oracle.doubly_diag_interp)
on the same (dtype-rounded) inputs."""
import ctypes as C

import numpy as np
import pytest
import torch

from hipgp_b200 import _lib as L
import emu_build

DT = {"f32": np.float32, "f64": np.float64}
CODE = {"f32": L.F32, "f64": L.F64}


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def rel(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


@pytest.fixture(scope="module")
def lib():
    return emu_build.load()


def line_problem(dname):
    """rays from the origin to 5 points of a 12 x 10 x 9 grid box (1080 columns: two blocks of 1024, the second partial)"""
    rng = np.random.default_rng(3)
    dt = DT[dname]
    grids = [np.linspace(0.1, 1.0, 12), np.linspace(-0.5, 0.5, 10), np.linspace(0.2, 0.8, 9)]
    grids = [g.astype(dt) for g in grids]
    x = np.stack([rng.uniform(0.1, 1.0, 5), rng.uniform(-0.5, 0.5, 5), rng.uniform(0.2, 0.8, 5)], 1).astype(dt)
    u = np.stack([a.reshape(-1) for a in np.meshgrid(*grids, indexing="ij")], 1).astype(dt)
    G = rng.standard_normal((5, u.shape[0])).astype(dt)
    return grids, x, u, G


def want_semi_grad(x, u, G, sig2, ell):
    """fp64 autograd of sum G * semi_integrated_sqe(x, u) with Sinv = diag(1 / ell^2) (kernels.py:223-237)"""
    from oracle import ziggy_oracle as zo
    s = torch.tensor(sig2, dtype=torch.float64, requires_grad=True)
    e = torch.tensor(ell, dtype=torch.float64, requires_grad=True)
    D = x.shape[1]
    Sinv = torch.diag(torch.ones(D, dtype=torch.float64) / e ** 2) if e.dim() else torch.eye(D, dtype=torch.float64) / e ** 2
    K = zo.semi_integrated_sqe(torch.from_numpy(x.astype(np.float64)), torch.from_numpy(u.astype(np.float64)), s, Sinv)
    (K * torch.from_numpy(G.astype(np.float64))).sum().backward()
    return float(s.grad), e.grad.numpy()


def run_kxu_grad(lib, dname, x, G, sig2, ell, grids=None, ypts=None):
    dt = DT[dname]
    x = np.ascontiguousarray(x, dt); G = np.ascontiguousarray(G, dt)
    B, D = x.shape
    M = G.shape[1]
    ellv = np.atleast_1d(np.asarray(ell, np.float64))
    nbx = (M + 1023) // 1024
    partial = np.full((B, nbx, 4), np.nan)
    if grids is not None:
        marr = (C.c_int64 * D)(*[len(g) for g in grids])
        gcat = np.ascontiguousarray(np.concatenate(grids).astype(dt))
        args = (marr, ptr(gcat), None, 0)
    else:
        ypts = np.ascontiguousarray(ypts, dt)
        args = (None, None, ptr(ypts), ypts.shape[0])
    rc = lib.hipgp_kxu_param_grad(CODE[dname], L.K_SQEXP, L.KXU_SEMI_ANALYTIC, sig2, (C.c_double * len(ellv))(*ellv), len(ellv),
                                  ptr(x), B, D, *args, None, 0, ptr(G), ptr(partial), None)
    assert rc == 0, lib.hipgp_last_error()
    tot = partial.sum(axis=(0, 1))
    return tot[0], (tot[1:4].sum() if len(ellv) == 1 else tot[1:1 + D])


@pytest.mark.parametrize("dname", ["f32", "f64"])
@pytest.mark.parametrize("shape", ["grid", "points"])
@pytest.mark.parametrize("ell", [0.3, (0.3, 0.5, 0.9)], ids=["scalar", "per_axis"])
def test_analytic_line_integral_param_grad(lib, dname, shape, ell):
    """The kernel evaluates the derivative in fp64 whatever the input dtype, so fp32 inputs meet the fp64 bound of 1e-10 against
    fp64 autograd on the same rounded inputs."""
    grids, x, u, G = line_problem(dname)
    sig2 = 1.3
    if shape == "grid":
        got_s, got_e = run_kxu_grad(lib, dname, x, G, sig2, ell, grids=grids)
    else:
        got_s, got_e = run_kxu_grad(lib, dname, x, G, sig2, ell, ypts=u)
    want_s, want_e = want_semi_grad(x, u, G, sig2, ell)
    assert abs(got_s - want_s) <= 1e-10 * abs(want_s), (got_s, want_s)
    assert rel(got_e, want_e) < 1e-10, (got_e, want_e)


def test_analytic_param_grad_refuses_other_kernels(lib):
    grids, x, u, G = line_problem("f64")
    partial = np.zeros((5, 2, 4))
    marr = (C.c_int64 * 3)(*[len(g) for g in grids])
    gcat = np.ascontiguousarray(np.concatenate(grids))
    for kid in (L.K_MATERN32, L.K_GNEITING):
        rc = lib.hipgp_kxu_param_grad(L.F64, kid, L.KXU_SEMI_ANALYTIC, 1.0, (C.c_double * 1)(0.3), 1, ptr(x), 5, 3, marr, ptr(gcat),
                                      None, 0, None, 0, ptr(G), ptr(partial), None)
        assert rc != 0 and "SqExp only" in lib.hipgp_last_error().decode()
    assert not partial.any()


def diag_table(kname, dname):
    """the table KernelDoublyDiagInterpolator builds for the kernel (50 entries up to dmax = 5), in the interpolator's dtype"""
    from hipgp_b200 import kernels as hk
    tdt = torch.float32 if dname == "f32" else torch.float64
    kern = hk.SqExp(dtype=tdt) if kname == "sqexp" else hk.Matern(nu=1.5, dtype=tdt)
    di = kern.diag_interp
    return [t.numpy() for t in (di.distance_grid, di.slopes, di.knn)]


def diag_points(dname, ell):
    """|x| / ell from 0.05 to 6.5: every interval of the table and the extrapolation past dmax = 5 with the last slope"""
    rng = np.random.default_rng(8)
    r = np.concatenate([np.linspace(0.05, 6.5, 300), rng.uniform(0.0, 6.5, 40)]) * ell
    d = rng.standard_normal((len(r), 3))
    return (d / np.linalg.norm(d, axis=1, keepdims=True) * r[:, None]).astype(DT[dname])


def want_diag_grad(x, g, sig2, ell, table):
    from oracle import ziggy_oracle as zo
    s = torch.tensor(sig2, dtype=torch.float64, requires_grad=True)
    e = torch.tensor(ell, dtype=torch.float64, requires_grad=True)
    tab = [torch.from_numpy(t.astype(np.float64)) for t in table]
    out = zo.doubly_diag_interp(torch.from_numpy(x.astype(np.float64)), s, e, *tab)
    (out * torch.from_numpy(g.astype(np.float64))).sum().backward()
    return float(s.grad), float(e.grad)


def run_diag_grad(lib, dname, x, g, sig2, ell, table):
    dt = DT[dname]
    x = np.ascontiguousarray(x, dt); g = np.ascontiguousarray(g, dt)
    dg, sl, kn = [np.ascontiguousarray(t, dt) for t in table]
    B, D = x.shape
    partial = np.full(((B + 255) // 256, 2), np.nan)
    rc = lib.hipgp_doubly_diag_param_grad(CODE[dname], ptr(x), B, D, sig2, (C.c_double * 1)(ell), 1, ptr(dg), ptr(sl), ptr(kn),
                                          len(dg), ptr(g), ptr(partial), None)
    assert rc == 0, lib.hipgp_last_error()
    return partial.sum(axis=0)


@pytest.mark.parametrize("dname", ["f32", "f64"])
@pytest.mark.parametrize("kname", ["sqexp", "matern32"])
def test_doubly_diag_param_grad(lib, dname, kname):
    """340 points (two blocks of 256, the second partial).  fp32: the distance and the table lookup are evaluated in fp32 as in
    the forward, so the bound is fp32's."""
    ell, sig2 = 0.2, 1.3
    table = diag_table(kname, dname)
    x = diag_points(dname, ell)
    g = np.random.default_rng(9).standard_normal(len(x)).astype(DT[dname])
    got = run_diag_grad(lib, dname, x, g, sig2, ell, table)
    want = want_diag_grad(x, g, sig2, ell, table)
    tol = 1e-5 if dname == "f32" else 1e-12
    assert abs(got[0] - want[0]) <= tol * abs(want[0]), (got, want)
    assert abs(got[1] - want[1]) <= tol * abs(want[1]), (got, want)


def test_doubly_diag_param_grad_argument_errors(lib):
    table = [np.ascontiguousarray(t) for t in diag_table("sqexp", "f64")]
    dg, sl, kn = table
    x = np.ascontiguousarray(diag_points("f64", 0.2)[:10]); g = np.ones(10)
    partial = np.zeros((1, 2))
    f = lib.hipgp_doubly_diag_param_grad
    ell1, ell3 = (C.c_double * 1)(0.2), (C.c_double * 3)(0.2, 0.3, 0.4)

    def call(dtype=L.F64, xp=ptr(x), B=10, D=3, ell=ell1, n_ell=1, dgp=ptr(dg), ntab=len(dg), gp=ptr(g), pp=ptr(partial)):
        return f(dtype, xp, B, D, 1.0, ell, n_ell, dgp, ptr(sl), ptr(kn), ntab, gp, pp, None)
    for kw, what in ((dict(dtype=7), "dtype"), (dict(D=0), "ndim"), (dict(D=4), "ndim"), (dict(ell=ell3, n_ell=3), "scalar"),
                     (dict(ntab=0), "table"), (dict(B=-1), "negative"), (dict(xp=None), "null"), (dict(dgp=None), "null"),
                     (dict(gp=None), "null"), (dict(pp=None), "null")):
        assert call(**kw) != 0, kw
        assert what in lib.hipgp_last_error().decode(), (kw, lib.hipgp_last_error())
    assert not partial.any()
    # empty minibatch: success, partial untouched
    sentinel = np.full((1, 2), 3.5)
    assert call(B=0, pp=ptr(sentinel)) == 0, lib.hipgp_last_error()
    assert np.all(sentinel == 3.5)
