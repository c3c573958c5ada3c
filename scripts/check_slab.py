"""Run under torchrun (N >= 2): slab-decomposed K matvec and PCG vs the undecomposed plan on rank 0.
usage: check_slab.py [m0 m1 m2] [bench] [nccl]
  nccl: exchange through NCCL all-to-alls (two overlapped chunks) instead of the peer-memory stores"""
import os, sys, json
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
from hipgp_b200.slab import SlabToeplitz
from hipgp_b200.plan import Plan
from hipgp_b200 import _lib as L, kernels as hk
world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0")); local = int(os.environ.get("LOCAL_RANK", "0"))
torch.cuda.set_device(local); dev = torch.device("cuda", local)
os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
if world > 1:
    dist.init_process_group("nccl", device_id=dev)
args = [a for a in sys.argv[1:] if a not in ("bench", "nccl")]
dims = tuple(int(a) for a in args[:3]) if len(args) >= 3 else (64, 48, 40)
bench = "bench" in sys.argv
dtype = torch.float32 if bench else torch.float64
xg = [torch.linspace(0, 1, m, dtype=dtype, device=dev) for m in dims]
step = float(xg[0][1] - xg[0][0])
col = hk.first_row(xg, hk.Matern(nu=2.5, dtype=dtype), (1.0, 2.5 * step), jitter=1e-3)
slab = SlabToeplitz(dims, col, dtype, dev, exchange="nccl" if "nccl" in sys.argv else None)
n0 = dims[0] // world
gen = torch.Generator(device=dev); gen.manual_seed(42)
v = torch.randn(1, int(np.prod(dims)), dtype=dtype, device=dev, generator=gen)      # same on every rank
mine = v.view(dims)[rank * n0:(rank + 1) * n0].contiguous()
out = slab.matvec_K(mine)
x = slab.solve(mine, do_precond=True, maxiter=20, tol=1e-8)
if not bench:
    full = Plan(dims, dtype, dev).set_first_row(col)
    ref = full.matvec(L.MV_K, v).view(dims)[rank * n0:(rank + 1) * n0].reshape(-1)
    xr = full.pcg(v, maxiter=20, tol=1e-8).view(dims)[rank * n0:(rank + 1) * n0].reshape(-1)
    e = torch.stack([(out - ref).norm() / ref.norm(), (x.reshape(-1) - xr).norm() / xr.norm()])
    if world > 1: dist.all_reduce(e, op=dist.ReduceOp.MAX)
    if rank == 0:
        print("slab vs full: matvec rel err %.2e, PCG(20) rel err %.2e (world %d, grid %s)" % (e[0].item(), e[1].item(), world, dims))
        assert e[0].item() < 1e-12 and e[1].item() < 1e-8
else:
    def timed(fn, n):
        for _ in range(2): fn()
        torch.cuda.synchronize()
        if world > 1: dist.barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n): fn()
        e1.record(); torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / n], device=dev, dtype=torch.float64)
        if world > 1: dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return t.item()
    ms_mv = timed(lambda: slab.matvec_K(mine), 10)
    ms_pcg = timed(lambda: slab.solve(mine, do_precond=True, maxiter=20, tol=1e-8), 2)
    # where the time goes: per-class kernel times of one matvec (CUDA events around every launch), the barrier alone, host issue time
    import ctypes as C, time
    p0 = slab.plans[0]
    L.check(p0.lib, p0.lib.hipgp_plan_profile(p0._h, 1))
    slab.matvec_K(mine); torch.cuda.synchronize()
    cls = {}
    for i, nm in enumerate(("rows_fwd", "cols", "rows_inv", "push/pack")):
        ms = C.c_double(); n = C.c_int64()
        L.check(p0.lib, p0.lib.hipgp_plan_profile_read(p0._h, i, C.byref(ms), C.byref(n), 0))
        cls[nm] = (round(ms.value, 4), n.value)
    L.check(p0.lib, p0.lib.hipgp_plan_profile(p0._h, 0))
    tok = torch.zeros(1, device=dev)
    bar_ms = timed(lambda: dist.all_reduce(tok), 20) if world > 1 else 0.0
    torch.cuda.synchronize(); t0 = time.perf_counter()
    for _ in range(10): slab.matvec_K(mine)
    issue_ms = (time.perf_counter() - t0) / 10 * 1e3
    torch.cuda.synchronize()
    if rank == 0:
        print(json.dumps({"kernel_ms_by_class": cls, "allreduce_barrier_ms": bar_ms, "host_issue_ms_per_matvec": issue_ms, "exchange": slab.exchange}))
        M = int(np.prod(dims)); E_h = (2 * dims[0] - 2) * (2 * dims[1] - 2) * (dims[2] - 1 + 1)
        print(json.dumps({"bench": "slab_matvec", "grid": dims, "n_gpus": world, "dtype": "f32", "matvec_ms": ms_mv,
                          "pcg20_s": ms_pcg / 1e3, "alg_GBps": 4 * (2 * M + E_h) / ms_mv / 1e6,
                          "exchange_MB_per_rank_per_transpose": slab.exch_elems * 8 / 1e6}))
if world > 1: dist.destroy_process_group()
