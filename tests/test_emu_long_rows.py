"""CPU execution of the four-step path along the LAST axis of 2-D and 3-D grids (long1d_kernels.cuh / long1d_api.inl with
the column passes of the leading axes in between), against numpy fp64 and the CPU oracle.

The library is built here on its own (same sources, g++ -DHIPGP_EMU -DHIPGP_DEV_SMALL) with the row-pass shared-memory
budget lowered to 4 KB, so that last axes of a few hundred points already leave the one-block row pass: the same switch
that sends last axes of m >= 2732 (R^T / R) and m >= 4097 (K / C^-1) to the four-step path on the device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from hipgp_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC_DIR = os.path.join(ROOT, "hipgp_b200", "csrc")
OUT = os.path.join(ROOT, "tests", "_emu", "libhipgp_emu_long_rows.so")
ROW_SMEM_MAX = 4096


def _build():
    srcs = [os.path.join(SRC_DIR, f) for f in os.listdir(SRC_DIR) if f.endswith((".cu", ".cuh", ".h", ".inl"))]
    srcs.append(os.path.join(ROOT, "include", "hipgp_b200.h"))
    if not os.path.exists(OUT) or any(os.path.getmtime(s) > os.path.getmtime(OUT) for s in srcs):
        os.makedirs(os.path.dirname(OUT), exist_ok=True)
        tmp = OUT + ".%d.tmp" % os.getpid()
        subprocess.run(["g++", "-O1", "-std=c++17", "-DHIPGP_EMU", "-DHIPGP_DEV_SMALL", "-DHIPGP_ROW_SMEM_MAX=%d" % ROW_SMEM_MAX,
                        "-x", "c++", "-fPIC", "-shared", "-pthread", os.path.join(SRC_DIR, "plan.cu"),
                        os.path.join(SRC_DIR, "fast_inst.cu"), "-o", tmp], check=True)
        os.replace(tmp, OUT)
    return OUT


@pytest.fixture(scope="module")
def lib():
    return L.declare(C.CDLL(_build()))


DTS = {"f64": (np.float64, L.F64, 1e-10), "f32": (np.float32, L.F32, 1e-5)}
# shape -> (launches per K / C^-1 matvec, per R^T / R matvec): the four-step path takes 5 (2-D) / 7 (3-D), the row pass 3 / 5.
# (3, 100): only the wide embedding (512) leaves the row pass, the narrow one (256) keeps it.
SHAPES = {(3, 100): (3, 5), (3, 200): (5, 5), (5, 300): (5, 5), (2, 3, 200): (7, 7), (3, 2, 300): (7, 7)}


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


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


def raw_spectrum(col, dims):
    """Re FFT_N of the even extension of the column, N = 2m - 2 per axis"""
    Cc = col.reshape(dims)
    for d in range(len(dims)):
        sl = [slice(None)] * len(dims); sl[d] = slice(dims[d] - 2, 0, -1)
        Cc = np.concatenate([Cc, Cc[tuple(sl)]], axis=d)
    return np.fft.fftn(Cc).real


def dense_apply(col, dims, v, f, n_in, n_out):
    """crop_{n_out} IFFT_N( f(max(Re FFT_N C, 1e-6)) * FFT_N pad_{n_in} v ) (numpy fp64)"""
    Dg = np.maximum(raw_spectrum(col, dims), 1e-6)
    D = len(dims)
    x = np.zeros((v.shape[0],) + Dg.shape)
    x[(slice(None),) + tuple(slice(0, k) for k in n_in)] = v.reshape((v.shape[0],) + tuple(n_in))
    ax = tuple(range(1, D + 1))
    y = np.fft.ifftn(f(Dg) * np.fft.fftn(x, axes=ax), axes=ax).real
    return y[(slice(None),) + tuple(slice(0, k) for k in n_out)].reshape(v.shape[0], -1)


class PlanNd:
    def __init__(self, lib, dims, dname, col=None):
        self.lib, self.dims = lib, tuple(dims)
        self.Nd = tuple(2 * m - 2 for m in dims)
        self.M, self.E = int(np.prod(dims)), int(np.prod(self.Nd))
        self.dt, code, self.tol = DTS[dname]
        h = C.c_void_p()
        assert lib.hipgp_plan_create(len(dims), (C.c_int64 * len(dims))(*dims), code, 0, C.byref(h)) == 0, lib.hipgp_last_error()
        self.h = h
        self.col = (first_col(dims) if col is None else col).astype(self.dt).astype(np.float64)
        c = self.col.astype(self.dt)
        n = C.c_int64()
        assert lib.hipgp_plan_set_first_row(h, ptr(c), 1e-6, C.byref(n), None) == 0, lib.hipgp_last_error()
        self.nclamped = n.value

    def __del__(self):
        self.lib.hipgp_plan_destroy(self.h)

    def launches(self):
        n = C.c_int64()
        self.lib.hipgp_plan_launch_count(self.h, C.byref(n))
        return n.value

    def mv(self, mode, v):
        v = np.ascontiguousarray(v, dtype=self.dt)
        out = np.zeros((v.shape[0], self.E if mode == L.MV_RT else self.M), self.dt)
        assert self.lib.hipgp_matvec(self.h, mode, ptr(v), ptr(out), v.shape[0], None) == 0, self.lib.hipgp_last_error()
        return out

    def embedding(self):
        Ln, Lw = (C.c_int64 * len(self.dims))(), (C.c_int64 * len(self.dims))()
        assert self.lib.hipgp_plan_embedding(self.h, Ln, Lw) == 0
        return list(Ln), list(Lw)


@pytest.mark.parametrize("dims", list(SHAPES), ids=lambda d: "x".join(map(str, d)))
def test_launch_counts_and_embedding(lib, dims):
    """launches per matvec on each side of the switch; the four-step last axis reports L1 * L2, the leading axes keep their
    lengths"""
    p = PlanNd(lib, dims, "f64")
    want_n, want_w = SHAPES[dims]
    v = np.ones((3, p.M)); w = np.ones((3, p.E))
    p.mv(L.MV_RT, v)                                      # (the first R^T builds the wide spectrum)
    for mode, inp, want in ((L.MV_K, v, want_n), (L.MV_CINV, v, want_n), (L.MV_RT, v, want_w), (L.MV_R, w, want_w)):
        n0 = p.launches(); p.mv(mode, inp)
        assert p.launches() - n0 == want, mode
    Ln, Lw = p.embedding()
    m = dims[-1]
    assert Ln[-1] >= 2 * m - 1 and Lw[-1] >= 3 * m - 3
    # (the lengths the same plan would get in 1-D, and the leading axes' lengths of a grid with a short last axis)
    q1 = PlanNd(lib, (m,), "f64")
    assert (Ln[-1], Lw[-1]) == (q1.embedding()[0][0], q1.embedding()[1][0])
    q2 = PlanNd(lib, dims[:-1] + (5,), "f64")
    assert (Ln[:-1], Lw[:-1]) == (q2.embedding()[0][:-1], q2.embedding()[1][:-1])


@pytest.mark.parametrize("dname", ["f64", "f32"])
@pytest.mark.parametrize("dims", list(SHAPES), ids=lambda d: "x".join(map(str, d)))
def test_operators_against_dense_formula(lib, dims, dname):
    p = PlanNd(lib, dims, dname)
    rng = np.random.default_rng(sum(dims))
    tol = p.tol
    Dg = np.maximum(raw_spectrum(p.col, dims), 1e-6)
    ptol = tol if dname == "f64" else 1e-5 + 0.5 * float(Dg.max() / Dg.min()) * 2.0 ** -24
    for B in (1, 2, 3):
        v = rng.standard_normal((B, p.M)).astype(p.dt).astype(np.float64)
        w = rng.standard_normal((B, p.E)).astype(p.dt).astype(np.float64)
        Kv = dense_apply(p.col, dims, v, lambda d: d, dims, dims)
        assert relerr(p.mv(L.MV_K, v), Kv) < tol, B
        assert relerr(p.mv(L.MV_CINV, v), dense_apply(p.col, dims, v, lambda d: 1.0 / d, dims, dims)) < ptol, B
        RTv = p.mv(L.MV_RT, v)
        assert relerr(RTv, dense_apply(p.col, dims, v, np.sqrt, dims, p.Nd)) < tol, B
        assert relerr(p.mv(L.MV_R, w), dense_apply(p.col, dims, w, np.sqrt, p.Nd, dims)) < tol, B
        vKv = (v * Kv).sum(1)
        assert np.abs((RTv.astype(np.float64) ** 2).sum(1) - vKv).max() / np.abs(vKv).max() < 10 * tol
        assert relerr(p.mv(L.MV_R, RTv), Kv) < 10 * tol
        # a row of a batch against a one-row call: packed pairs couple the rounding of partners, nothing else
        for mode in (L.MV_K, L.MV_RT):
            assert relerr(p.mv(mode, v[B - 1:B]), p.mv(mode, v)[B - 1:B]) < (1e-14 if dname == "f64" else 1e-6), (B, mode)


@pytest.mark.parametrize("dname", ["f64", "f32"])
@pytest.mark.parametrize("dims", [(3, 200), (2, 3, 200)], ids=lambda d: "x".join(map(str, d)))
def test_setup_spectrum(lib, dims, dname):
    """the set-up (tiled DCT-I per axis, spectra from the four-step forward) against Re FFT_N of the embedding"""
    p = PlanNd(lib, dims, dname)
    Dsp = np.zeros(p.E, p.dt)
    assert lib.hipgp_plan_spectrum(p.h, L.SPEC_D, ptr(Dsp), None) == 0, lib.hipgp_last_error()
    raw = raw_spectrum(p.col, dims).reshape(-1)
    ref = np.maximum(raw, 1e-6)
    assert np.abs(Dsp - ref).max() / np.abs(ref).max() < (1e-13 if dname == "f64" else 1e-6)
    assert p.nclamped == int((raw < 1e-6).sum())


def recurrence_residual(ora, b, precond, iters):
    """||r|| of the recurrence r -= alpha A p after `iters` iterations of the oracle's conj_grad2 (cg.py:44-80)"""
    P = ora.matmul_Cinv if precond else (lambda v: v)
    x = torch.zeros_like(b); r = b.clone(); z = P(r); p = z
    for _ in range(iters):
        rs = (r * z).sum(1); Ap = ora.matmul_K(p); alpha = rs / (p * Ap).sum(1)
        x = x + alpha[:, None] * p; r = r - alpha[:, None] * Ap
        z = P(r); p = z + ((z * r).sum(1) / rs)[:, None] * p
    return r.norm(dim=1).numpy()


def _oracle_2d(m0, m1, ell):
    from oracle import ziggy_oracle as zo
    dt = torch.float64
    return zo.OracleToeplitz([torch.linspace(0, 1, m0, dtype=dt), torch.linspace(0, 4, m1, dtype=dt)],
                             lambda x, y: zo.matern(x, y, 1.0, ell, 2.5), jitter_val=1e-3)


@pytest.mark.parametrize("precond", [1, 0])
@pytest.mark.parametrize("dname", ["f64", "f32"])
def test_pcg_against_oracle(lib, dname, precond):
    """PCG on a 2-D grid with a four-step last axis: iterate, callback count and recurrence residual against the oracle's
    conj_grad2, and compute_kn = R^T of the same solve"""
    m0, m1, B, iters = 3, 200, 3, 6
    ora = _oracle_2d(m0, m1, 0.5)
    torch.manual_seed(0)
    b = torch.randn(B, m0 * m1, dtype=torch.float64)
    n_ref = [0]
    x_ref = ora.solve(b, do_precond=bool(precond), maxiter=iters, tol=1e-14, callback=lambda n, x: n_ref.__setitem__(0, n_ref[0] + 1))
    p = PlanNd(lib, (m0, m1), dname, col=ora.column.reshape(-1).numpy())
    bb = np.ascontiguousarray(b.numpy().astype(p.dt)); x = np.zeros_like(bb)
    it, ncb = C.c_int(), C.c_int()
    resid = (C.c_double * B)()
    n_dev = [0]
    cb = L.ITER_CB(lambda n, xp, user: n_dev.__setitem__(0, n_dev[0] + 1))
    assert lib.hipgp_pcg(p.h, ptr(bb), ptr(x), B, iters, 1e-14, precond, C.byref(it), C.byref(ncb), resid, cb, None, None) == 0, \
        lib.hipgp_last_error()
    assert n_dev[0] == n_ref[0] == ncb.value == iters and it.value == iters
    assert relerr(x, x_ref.numpy()) < (1e-9 if dname == "f64" else 1e-3)
    if dname == "f64":
        atol = 1e-9 * float(b.norm(dim=1).max())
        assert np.allclose(np.asarray(resid[:]), recurrence_residual(ora, b, bool(precond), iters), rtol=1e-6, atol=atol)
    if precond:
        kn = np.zeros((B, p.E), p.dt)
        assert lib.hipgp_compute_kn(p.h, ptr(bb), ptr(kn), B, iters, 1e-14, None, None) == 0, lib.hipgp_last_error()
        assert np.array_equal(kn, p.mv(L.MV_RT, x))


def test_pcg_stops_like_the_fused_solver(lib):
    """a solve that converges stops at the same iteration, with the same callback count, as the oracle; the asynchronous host
    solve gives the same bits"""
    m0, m1, B = 3, 300, 2
    ora = _oracle_2d(m0, m1, 0.05)
    torch.manual_seed(1)
    b = torch.randn(B, m0 * m1, dtype=torch.float64)
    n_ref = [0]
    x_ref = ora.solve(b, do_precond=True, maxiter=200, tol=1e-8, callback=lambda n, x: n_ref.__setitem__(0, n_ref[0] + 1))
    p = PlanNd(lib, (m0, m1), "f64", col=ora.column.reshape(-1).numpy())
    bb = b.numpy().copy(); x = np.zeros_like(bb)
    it, ncb = C.c_int(), C.c_int()
    assert lib.hipgp_pcg(p.h, ptr(bb), ptr(x), B, 200, 1e-8, 1, C.byref(it), C.byref(ncb), None, L.ITER_CB(0), None, None) == 0
    assert 0 < it.value < 200 and ncb.value == n_ref[0] == it.value - 1
    assert relerr(x, x_ref.numpy()) < 1e-9
    xs = np.zeros_like(bb); its = C.c_int()
    assert lib.hipgp_pcg_host_submit(p.h, ptr(bb), ptr(xs), B, 200, 1e-8, 1, 0, None) == 0, lib.hipgp_last_error()
    assert lib.hipgp_pcg_host_wait(p.h, 0, C.byref(its)) == 0
    assert its.value == it.value and np.array_equal(xs, x)


def test_refusals(lib):
    """the gradient entry points and the slab decomposition raise on these plans, naming the limitation; the plan still works"""
    p = PlanNd(lib, (2, 3, 200), "f64")
    v = np.ones((1, p.M)); g = np.ones((1, p.E)); out = np.zeros(p.M)
    assert lib.hipgp_toeplitz_quadform(p.h, ptr(v), ptr(v), 1, 1.0, ptr(out), None) != 0
    assert "last axis is too long" in lib.hipgp_last_error().decode()
    assert lib.hipgp_rt_column_grad(p.h, ptr(v), ptr(g), 1, 1.0, ptr(out), None) != 0
    assert "last axis is too long" in lib.hipgp_last_error().decode()
    assert lib.hipgp_plan_set_slab(p.h, 0, 2) != 0
    assert "last axis is too long" in lib.hipgp_last_error().decode()
    # (3, 100): the narrow embedding keeps the row pass, so only the wide one refuses
    q = PlanNd(lib, (3, 100), "f64")
    v = np.ones((1, q.M)); g = np.ones((1, q.E)); out = np.zeros(q.M)
    assert lib.hipgp_toeplitz_quadform(q.h, ptr(v), ptr(v), 1, 1.0, ptr(out), None) == 0, lib.hipgp_last_error()
    assert lib.hipgp_rt_column_grad(q.h, ptr(v), ptr(g), 1, 1.0, ptr(out), None) != 0
    assert "last axis is too long" in lib.hipgp_last_error().decode()
    assert relerr(p.mv(L.MV_K, np.ones((1, p.M))), dense_apply(p.col, p.dims, np.ones((1, p.M)), lambda d: d, p.dims, p.dims)) < 1e-10
