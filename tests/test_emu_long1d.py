"""CPU execution of the four-step path for long 1-D grids (long1d_kernels.cuh / long1d_api.inl) and its Bluestein DCT-I
set-up, against numpy fp64 and the CPU oracle.

The library is built here on its own (same sources, g++ -DHIPGP_EMU -DHIPGP_DEV_SMALL) with the row-pass shared-memory
budget lowered to 4 KB, so that 1-D embeddings of a few hundred points already leave the one-block row pass: the same
switch that sends m ~ 10^4 .. 10^6 grids to the four-step path on the device."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import torch

from hipgp_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC_DIR = os.path.join(ROOT, "hipgp_b200", "csrc")
OUT = os.path.join(ROOT, "tests", "_emu", "libhipgp_emu_long1d.so")
ROW_SMEM_MAX = 4096          # fp64 row pass fits up to H = 127, fp32 up to H = 255


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


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def first_col(m):
    r = np.linspace(0.0, 1.0, m)
    ell = 15.0 / m
    col = (1 + np.sqrt(5) * r / ell + 5 * r ** 2 / (3 * ell ** 2)) * np.exp(-np.sqrt(5) * r / ell)
    col[0] += 1e-3
    return col


def spectrum(col):
    m = col.size
    return np.maximum(np.fft.fft(np.concatenate([col, col[m - 2:0:-1]])).real, 1e-6)


def dense_apply(col, v, f, n_out):
    """crop IFFT_N( f(max(Re FFT_N C, 1e-6)) * FFT_N pad v ), N = 2m - 2 (numpy fp64)"""
    Dg = spectrum(col)
    x = np.zeros((v.shape[0], Dg.size)); x[:, :v.shape[1]] = v
    return np.fft.ifft(f(Dg) * np.fft.fft(x, axis=1), axis=1).real[:, :n_out]


class Plan1d:
    def __init__(self, lib, m, dname):
        self.lib, self.m, self.N = lib, m, 2 * m - 2
        self.dt, code, self.tol = DTS[dname]
        h = C.c_void_p()
        assert lib.hipgp_plan_create(1, (C.c_int64 * 1)(m), code, 0, C.byref(h)) == 0, lib.hipgp_last_error()
        self.h = h
        self.col = first_col(m)
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
        out = np.zeros((v.shape[0], self.N if mode == L.MV_RT else self.m), self.dt)
        assert self.lib.hipgp_matvec(self.h, mode, ptr(v), ptr(out), v.shape[0], None) == 0, self.lib.hipgp_last_error()
        return out


def test_switch(lib):
    """m = 100: the narrow embedding (256 = 2 x 128, a specialised row length) stays on the row pass, two launches per
    matvec; its wide one (512) and both embeddings of m = 200 take the four-step path, three launches per matvec."""
    for m, k_launches, rt_launches in ((100, 2, 3), (200, 3, 3)):
        p = Plan1d(lib, m, "f64")
        v = np.ones((1, m))
        for mode, want in ((L.MV_K, k_launches), (L.MV_RT, rt_launches)):
            p.mv(mode, v)                       # (the first R^T builds the wide spectrum)
            n0 = p.launches(); p.mv(mode, v)
            assert p.launches() - n0 == want, (m, mode)
        Ln, Lw = (C.c_int64 * 1)(), (C.c_int64 * 1)()
        assert lib.hipgp_plan_embedding(p.h, Ln, Lw) == 0
        assert (Ln[0], Lw[0]) == {100: (256, 512), 200: (512, 1024)}[m]


@pytest.mark.parametrize("dname", ["f64", "f32"])
@pytest.mark.parametrize("m", [200, 300])
def test_matvecs_against_dense_formula(lib, m, dname):
    p = Plan1d(lib, m, dname)
    rng = np.random.default_rng(m)
    tol = p.tol
    Dg = spectrum(p.col)
    ptol = tol if dname == "f64" else 1e-5 + 0.5 * float(Dg.max() / Dg.min()) * 2.0 ** -24
    for B in (1, 2, 3, 5):
        v = rng.standard_normal((B, m)).astype(p.dt).astype(np.float64)
        Kv = dense_apply(p.col, v, lambda d: d, m)
        assert relerr(p.mv(L.MV_K, v), Kv) < tol, B
        assert relerr(p.mv(L.MV_CINV, v), dense_apply(p.col, v, lambda d: 1.0 / d, m)) < ptol, B
        RTv = p.mv(L.MV_RT, v)
        assert relerr(RTv, dense_apply(p.col, v, np.sqrt, p.N)) < tol, B
        w = rng.standard_normal((B, p.N)).astype(p.dt).astype(np.float64)
        assert relerr(p.mv(L.MV_R, w), np.fft.ifft(np.sqrt(Dg) * np.fft.fft(w, axis=1), axis=1).real[:, :m]) < tol, B
        vKv = (v * Kv).sum(1)
        assert np.abs((RTv.astype(np.float64) ** 2).sum(1) - vKv).max() / np.abs(vKv).max() < 10 * tol
        assert relerr(p.mv(L.MV_R, RTv), Kv) < 10 * tol
        # a row of a batch against a one-row call: packed pairs couple the rounding of partners, nothing else
        assert relerr(p.mv(L.MV_K, v[B - 1:B]), p.mv(L.MV_K, v)[B - 1:B]) < (1e-14 if dname == "f64" else 1e-6)


@pytest.mark.parametrize("dname", ["f64", "f32"])
@pytest.mark.parametrize("m", [200, 300])
def test_setup_spectrum(lib, m, dname):
    """the Bluestein DCT-I set-up (N = 2m - 2 = 398, 598: not 2^a 3^b 5^c) against Re FFT_N of the embedding"""
    p = Plan1d(lib, m, dname)
    Dsp = np.zeros(p.N, p.dt)
    assert lib.hipgp_plan_spectrum(p.h, L.SPEC_D, ptr(Dsp), None) == 0, lib.hipgp_last_error()
    ref = spectrum(p.col.astype(p.dt).astype(np.float64))
    assert np.abs(Dsp - ref).max() / np.abs(ref).max() < (1e-13 if dname == "f64" else 1e-6)
    assert p.nclamped == int((np.fft.fft(np.concatenate([p.col, p.col[m - 2:0:-1]])).real < 1e-6).sum())


def recurrence_residual(ora, b, precond, iters):
    """||r|| of the recurrence r -= alpha A p after `iters` iterations of the oracle's conj_grad2 (cg.py:44-80)"""
    P = ora.matmul_Cinv if precond else (lambda v: v)
    x = torch.zeros_like(b); r = b.clone(); z = P(r); p = z
    for _ in range(iters):
        rs = (r * z).sum(1); Ap = ora.matmul_K(p); alpha = rs / (p * Ap).sum(1)
        x = x + alpha[:, None] * p; r = r - alpha[:, None] * Ap
        z = P(r); p = z + ((z * r).sum(1) / rs)[:, None] * p
    return r.norm(dim=1).numpy()


@pytest.mark.parametrize("precond", [1, 0])
@pytest.mark.parametrize("dname", ["f64", "f32"])
def test_pcg_against_oracle(lib, dname, precond):
    """PCG on the four-step path: iterate, callback count and recurrence residual against the oracle's conj_grad2"""
    from oracle import ziggy_oracle as zo
    m, B, iters = 200, 3, 6
    dt = torch.float64
    ora = zo.OracleToeplitz([torch.linspace(0, 4, m, dtype=dt)], lambda x, y: zo.matern(x, y, 1.0, 0.5, 2.5), jitter_val=1e-3)
    torch.manual_seed(0)
    b = torch.randn(B, m, dtype=dt)
    n_ref = [0]
    x_ref = ora.solve(b, do_precond=bool(precond), maxiter=iters, tol=1e-14, callback=lambda n, x: n_ref.__setitem__(0, n_ref[0] + 1))
    npdt, code, _ = DTS[dname]
    h = C.c_void_p()
    assert lib.hipgp_plan_create(1, (C.c_int64 * 1)(m), code, 0, C.byref(h)) == 0
    col = ora.column.numpy().astype(npdt)
    assert lib.hipgp_plan_set_first_row(h, ptr(col), 1e-6, None, None) == 0, lib.hipgp_last_error()
    bb = b.numpy().astype(npdt); x = np.zeros_like(bb)
    it, ncb = C.c_int(), C.c_int()
    resid = (C.c_double * B)()
    n_dev = [0]
    cb = L.ITER_CB(lambda n, xp, user: n_dev.__setitem__(0, n_dev[0] + 1))
    assert lib.hipgp_pcg(h, ptr(bb), ptr(x), B, iters, 1e-14, precond, C.byref(it), C.byref(ncb), resid, cb, None, None) == 0, \
        lib.hipgp_last_error()
    lib.hipgp_plan_destroy(h)
    assert n_dev[0] == n_ref[0] == ncb.value == iters and it.value == iters
    assert relerr(x, x_ref.numpy()) < (1e-9 if dname == "f64" else 1e-3)
    if dname == "f64":   # (small against b: a 1e-9 relative difference of the iterates moves it by ~1e-9 ||b||)
        atol = 1e-9 * float(b.norm(dim=1).max())
        assert np.allclose(np.asarray(resid[:]), recurrence_residual(ora, b, bool(precond), iters), rtol=1e-6, atol=atol)


def test_pcg_stops_like_the_fused_solver(lib):
    """a solve that converges stops at the same iteration, with the same callback count, as the oracle"""
    from oracle import ziggy_oracle as zo
    m, B = 300, 2
    dt = torch.float64
    ora = zo.OracleToeplitz([torch.linspace(0, 4, m, dtype=dt)], lambda x, y: zo.matern(x, y, 1.0, 0.05, 2.5), jitter_val=1e-3)
    torch.manual_seed(1)
    b = torch.randn(B, m, dtype=dt)
    n_ref = [0]
    x_ref = ora.solve(b, do_precond=True, maxiter=200, tol=1e-8, callback=lambda n, x: n_ref.__setitem__(0, n_ref[0] + 1))
    h = C.c_void_p()
    assert lib.hipgp_plan_create(1, (C.c_int64 * 1)(m), L.F64, 0, C.byref(h)) == 0
    col = ora.column.numpy().copy()
    assert lib.hipgp_plan_set_first_row(h, ptr(col), 1e-6, None, None) == 0
    bb = b.numpy().copy(); x = np.zeros_like(bb)
    it, ncb = C.c_int(), C.c_int()
    assert lib.hipgp_pcg(h, ptr(bb), ptr(x), B, 200, 1e-8, 1, C.byref(it), C.byref(ncb), None, L.ITER_CB(0), None, None) == 0
    lib.hipgp_plan_destroy(h)
    assert 0 < it.value < 200 and ncb.value == n_ref[0] == it.value - 1
    assert relerr(x, x_ref.numpy()) < 1e-9


def test_refusals(lib):
    """the gradient entry points raise on a long plan instead of touching the row-pass geometry"""
    p = Plan1d(lib, 200, "f64")
    v = np.ones((1, 200)); g = np.ones((1, p.N)); out = np.zeros(200)
    assert lib.hipgp_toeplitz_quadform(p.h, ptr(v), ptr(v), 1, 1.0, ptr(out), None) != 0
    assert "long 1-D plans" in lib.hipgp_last_error().decode()
    assert lib.hipgp_rt_column_grad(p.h, ptr(v), ptr(g), 1, 1.0, ptr(out), None) != 0
    assert "long 1-D plans" in lib.hipgp_last_error().decode()


def test_tiled_dct_refuses_long_axes(lib):
    """an axis longer than 65536 points never reaches the tiled DCT-I kernel (its 32-bit cosine index would overflow)"""
    h = C.c_void_p()
    assert lib.hipgp_plan_create(2, (C.c_int64 * 2)(70000, 2), L.F64, 0, C.byref(h)) == 0
    col = np.zeros(140000); col[0] = 1.0
    assert lib.hipgp_plan_set_first_row(h, ptr(col), 1e-6, None, None) != 0
    assert "65536" in lib.hipgp_last_error().decode()
    lib.hipgp_plan_destroy(h)
