"""CPU execution (g++ -DHIPGP_EMU build, tests/emu_build.py) of hipgp_block_quadform_grad, the backward of the block family's
knSkn_b = kn_b^T blockdiag(S) kn_b:  dkn = g[:, None] * from_blocks((S + S^T) @ to_blocks(kn)),  checked against numpy on
the block_step golden inputs (65-point blocks: a full and a one-row tile), a non-symmetric S and a 3-D index map."""
import ctypes as C
import os

import numpy as np
import pytest

from hipgp_b200 import _lib as L
import emu_build

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = {"f32": 1e-5, "f64": 1e-10}
DT = {"f32": np.float32, "f64": np.float64}
CODE = {"f32": L.F32, "f64": L.F64}


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def rel(a, b):
    a = np.asarray(a, np.float64); b = np.asarray(b, np.float64)
    return np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-300)


def want_dkn(S, kn, g, idx):
    """numpy restatement in fp64: g[:, None] * from_blocks((S + S^T) @ to_blocks(kn))"""
    S = S.astype(np.float64); kn = kn.astype(np.float64)
    blk = kn[:, idx]                                                    # (B, nblk, bs)
    prod = np.einsum("kij,bkj->bki", S + S.transpose(0, 2, 1), blk)
    out = np.empty_like(kn)
    out[:, idx.reshape(-1)] = prod.reshape(kn.shape[0], -1)
    return g.astype(np.float64)[:, None] * out


@pytest.fixture(scope="module")
def lib():
    return emu_build.load()


def run(lib, dname, S, kn, g, idx):
    dt = DT[dname]
    S = np.ascontiguousarray(S.astype(dt)); kn = np.ascontiguousarray(kn.astype(dt)); g = np.ascontiguousarray(g.astype(dt))
    idx = np.ascontiguousarray(idx.astype(np.int64))
    B, E = kn.shape
    nblk, bs = idx.shape
    out = np.full_like(kn, np.nan)
    assert lib.hipgp_block_quadform_grad(CODE[dname], ptr(S), ptr(kn), ptr(g), ptr(idx), B, E, nblk, bs, ptr(out), None) == 0, \
        lib.hipgp_last_error()
    return out, want_dkn(S, kn, g, idx)


@pytest.mark.parametrize("dname", ["f32", "f64"])
def test_block_quadform_grad_golden_and_nonsymmetric(lib, dname):
    gd = np.load(os.path.join(GOLD, "block_step_%s.npz" % dname))
    idx = gd["block_idx"]; kn = gd["kn"]
    rng = np.random.default_rng(7)
    g = rng.standard_normal(kn.shape[0])
    # the golden (symmetric) qS, then a random non-symmetric S: the kernel must use S + S^T, not 2 S
    for S in (gd["qS"], rng.standard_normal(gd["qS"].shape)):
        got, want = run(lib, dname, S, kn, g, idx)
        assert rel(got, want) < TOL[dname], rel(got, want)


@pytest.mark.parametrize("dname", ["f32", "f64"])
def test_block_quadform_grad_3d_map(lib, dname):
    """the golden 3-D map (8 blocks of 105 = 2 row tiles, the second one partial) with 70 rows (two tiles of right-hand sides)"""
    idx = np.load(os.path.join(GOLD, "block_step_f64.npz"))["block_idx_3d"]
    rng = np.random.default_rng(11)
    nblk, bs = idx.shape
    kn = rng.standard_normal((70, nblk * bs)); g = rng.standard_normal(70)
    S = rng.standard_normal((nblk, bs, bs))
    got, want = run(lib, dname, S, kn, g, idx)
    assert rel(got, want) < TOL[dname], rel(got, want)


def test_block_quadform_grad_argument_errors(lib):
    gd = np.load(os.path.join(GOLD, "block_step_f64.npz"))
    idx = np.ascontiguousarray(gd["block_idx"]); kn = np.ascontiguousarray(gd["kn"]); S = np.ascontiguousarray(gd["qS"])
    B, E = kn.shape
    nblk, bs = idx.shape
    g = np.ones(B)
    out = np.zeros_like(kn)
    f = lib.hipgp_block_quadform_grad
    assert f(L.F64, ptr(S), ptr(kn), ptr(g), ptr(idx), B, E, nblk, bs - 1, ptr(out), None) != 0          # does not tile M'
    assert "num_blocks * block_size" in lib.hipgp_last_error().decode()
    assert f(L.F64, ptr(S), ptr(kn), ptr(g), None, B, E, nblk, bs, ptr(out), None) != 0                  # null index
    assert "null block index" in lib.hipgp_last_error().decode()
    assert f(L.F64, ptr(S), ptr(kn), ptr(g), ptr(idx), B, E, nblk, bs, ptr(kn), None) != 0               # dkn == kn
    assert "overlap" in lib.hipgp_last_error().decode()
    assert f(L.F64, ptr(S), ptr(kn), None, ptr(idx), B, E, nblk, bs, ptr(out), None) != 0                # null g
    assert f(L.F64, None, ptr(kn), ptr(g), ptr(idx), B, E, nblk, bs, ptr(out), None) != 0                # null S
    assert f(7, ptr(S), ptr(kn), ptr(g), ptr(idx), B, E, nblk, bs, ptr(out), None) != 0 and "dtype" in lib.hipgp_last_error().decode()
    assert not out.any()
    # empty minibatch: success, dkn untouched
    sentinel = np.full_like(kn, 3.5)
    assert f(L.F64, ptr(S), ptr(kn), ptr(g), ptr(idx), 0, E, nblk, bs, ptr(sentinel), None) == 0, lib.hipgp_last_error()
    assert np.all(sentinel == 3.5)
