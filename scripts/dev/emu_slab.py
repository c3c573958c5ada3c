"""Developer check: slab-decomposed matvec stages on the CPU emulation build vs the undecomposed plan (emulated ranks)."""
import ctypes as C, sys, os
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from hipgp_b200 import _lib as L
import emu_build
lib = emu_build.load()
def ptr(a): return a.ctypes.data_as(C.c_void_p)
def mkplan(dims, dt, col, slab=None, chunks=1):
    plan = C.c_void_p(); mm = np.array(dims, dtype=np.int64)
    assert lib.hipgp_plan_create(3, mm.ctypes.data_as(L._pi64), L.F32 if dt == np.float32 else L.F64, 0, C.byref(plan)) == 0
    if slab: assert lib.hipgp_plan_set_slab(plan, slab[0], slab[1]) == 0, lib.hipgp_last_error()
    if chunks > 1: assert lib.hipgp_plan_set_slab_chunks(plan, chunks) == 0, lib.hipgp_last_error()
    ncl = C.c_int64()
    assert lib.hipgp_plan_set_first_row(plan, ptr(col), 1e-6, C.byref(ncl), None) == 0, lib.hipgp_last_error()
    return plan
def run(dims, nranks, dt, chunks=1, peer=False):
    g = np.meshgrid(*[np.linspace(0, 1 + d, k) for d, k in enumerate(dims)], indexing="ij")
    r = np.sqrt(sum((x - x.flat[0]) ** 2 for x in g)); col = ((1 + np.sqrt(3) * r / 0.4) * np.exp(-np.sqrt(3) * r / 0.4)).reshape(-1); col[0] += 1e-2
    col = col.astype(dt)
    full = mkplan(dims, dt, col)
    plans = [mkplan(dims, dt, col, (rk, nranks), chunks) for rk in range(nranks)]
    a, b = C.c_int64(), C.c_int64()
    assert lib.hipgp_slab2_sizes(plans[0], C.byref(a), C.byref(b)) == 0, lib.hipgp_last_error(); slab_elems, exch = a.value, b.value
    rng = np.random.default_rng(0); M = int(np.prod(dims))
    v = rng.standard_normal((1, M)).astype(dt)
    n0 = dims[0] // nranks
    slabs = [np.ascontiguousarray(v.reshape(dims)[rk * n0:(rk + 1) * n0]).reshape(-1) for rk in range(nranks)]
    cdt = np.complex64 if dt == np.float32 else np.complex128
    def exchange(bufs):
        per = exch // chunks; blk = per // nranks
        return [np.concatenate([bufs[q][c * per + rk * blk:c * per + (rk + 1) * blk] for c in range(chunks) for q in range(nranks)]) for rk in range(nranks)]
    if peer:
        r1 = [C.c_void_p() for _ in plans]; r2 = [C.c_void_p() for _ in plans]
        for i, p in enumerate(plans): assert lib.hipgp_slab2_peer_alloc(p, C.byref(r1[i]), C.byref(r2[i]), None, None) == 0, lib.hipgp_last_error()
        a1 = (C.c_void_p * nranks)(*[x.value for x in r1]); a2 = (C.c_void_p * nranks)(*[x.value for x in r2])
        for p in plans: assert lib.hipgp_slab2_peer_set(p, a1, a2) == 0, lib.hipgp_last_error()
    ok = True
    for mode in (0, 1):
        ref = np.zeros((1, M), dtype=dt)
        assert lib.hipgp_matvec(full, mode, ptr(v), ptr(ref), 1, None) == 0
        if peer:
            for p, x in zip(plans, slabs): assert lib.hipgp_slab2_push_a(p, ptr(x), None) == 0, lib.hipgp_last_error()
            for p in plans: assert lib.hipgp_slab2_push_b(p, mode, -1, None) == 0, lib.hipgp_last_error()
            outs = []
            for p in plans:
                o = np.zeros(slab_elems, dtype=dt); assert lib.hipgp_slab2_finish(p, ptr(o), None) == 0, lib.hipgp_last_error(); outs.append(o)
            got = np.concatenate(outs).reshape(1, -1)
            e = np.linalg.norm(got - ref) / np.linalg.norm(ref)
            print(dims, nranks, dt.__name__, "peer exchange, chunks", chunks, "mode", mode, "err %.2e" % e); ok &= e < (1e-5 if dt == np.float32 else 1e-10)
            continue
        bufs = []
        for p, x in zip(plans, slabs):
            send = np.zeros(exch, dtype=cdt); assert lib.hipgp_slab2_stage_a(p, ptr(x), ptr(send), None) == 0, lib.hipgp_last_error(); bufs.append(send)
        bufs = exchange(bufs)
        for p, bb in zip(plans, bufs): assert lib.hipgp_slab2_stage_b(p, mode, ptr(bb), None) == 0, lib.hipgp_last_error()
        bufs = exchange(bufs)
        outs = []
        for p, bb in zip(plans, bufs):
            o = np.zeros(slab_elems, dtype=dt); assert lib.hipgp_slab2_stage_c(p, ptr(bb), ptr(o), None) == 0, lib.hipgp_last_error(); outs.append(o)
        got = np.concatenate(outs).reshape(1, -1)
        e = np.linalg.norm(got - ref) / np.linalg.norm(ref)
        print(dims, nranks, dt.__name__, "chunks", chunks, "mode", mode, "err %.2e" % e); ok &= e < (1e-5 if dt == np.float32 else 1e-10)
    return ok
if __name__ == "__main__":
    ok = run((16, 12, 20), 2, np.float64) & run((16, 12, 20), 4, np.float32) & run((12, 10, 14), 3, np.float64)
    ok &= run((16, 12, 20), 4, np.float32, 1, True) & run((12, 10, 14), 3, np.float64, 2, True)
    ok &= run((16, 12, 20), 2, np.float32, 2) & run((12, 10, 14), 3, np.float64, 3)
    sys.exit(0 if ok else 1)
