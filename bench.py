#!/usr/bin/env python
"""bench.py -- headline benchmark of the HIP-GP structured-kernel hot path on B200.

Workload (BASELINE.json configs[1]): 2-D inducing grid 1000 x 1000 (M = 10^6), Matern-5/2, ell = 0.01,
jitter 1e-3, fp32; one STEP = one PCG solve K_uu^-1 b with the HIP-GP preconditioner exactly as the SVI
loop issues it (maxiter 20, tol 1e-8 -- it does not converge, so 20 iterations = 20 K-matvecs + 21
preconditioner matvecs + the fused vector updates) on B = 64 right-hand sides per GPU.

metric  : Toeplitz matvec GB/s = algorithmic bytes of the step's 41 structured matvecs,
          w (2 M B + E_h) each (SURVEY.md 8d contract figure, E_h = 1998*1000), divided by the step time.
          `pcg_solve_s` (the other half of BASELINE.json's metric) is reported beside it.
value   : inputs resident in HBM (plan.pcg on device tensors).
e2e     : the same steps through the C-ABI host entry points with HOST buffers: every step uploads its right-hand sides
          from pinned memory and downloads its solution inside the timed region.  The steps are a stream of batches through
          hipgp_pcg_host_submit / _wait with two in flight, so the copies of neighbouring steps run under the current solve.
          `one_synchronous_call_per_step` is the same through ONE blocking call per step (hipgp_pcg_host_pipelined: the
          right-hand sides travel as a small first group, the bulk, and a small last group).
roofline: per-kernel-class CUDA-event timing inside this script (a second pass of the same steps with the
          library's event hooks on); achieved = matvec algorithmic bytes / (sum of the three pass kernels'
          average durations); the dominant kernel and its share of the matvec are named.
cpu_baseline / --impl reference: the UNMODIFIED reference (`oracle/_ref/ziggy`, staged byte for byte by
          oracle/make_ref.py; ToeplitzTensor._solve under the legacy-torch shim oracle/ref_shim.py) on the host cores,
          same configuration, each step a bounded sample (8 of the step's 64 right-hand sides); falls back to the CPU
          oracle port (oracle/ziggy_oracle.py) when the staged reference is absent.

--dump-outputs DIR: after the timed steps, the solution the last timed step returned (B x M, fp32) is written as
          DIR/pcg_x_sample.npy at a fixed seeded sample of its grid points (all right-hand sides, DUMP_POINTS columns);
          the inputs are seeded, so two builds run with the same arguments can be compared output for output.  With
          N > 1 only rank 0 writes, so the file holds rank 0's right-hand sides (generator seed 42).

N > 1 (torchrun): right-hand sides are independent, so each rank solves its own B = 64 shard with no data-path
collective ("weak" scaling); time = max over ranks.  The two paths that DO need collectives are measured in the same run
and reported as extra keys: `svi_cfg3` (observation-sharded mean-field natural-gradient step, one packed all-reduce per
step) and `slab_cfg5` (512^3 grid sharded over the ranks, two all-to-all transposes per matvec).
"""
import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GRID = (1000, 1000)
ELL, SIG2, JITTER = 0.01, 1.0, 1e-3
MAXITER, TOL = 20, 1e-8
B_PER_GPU = 64
E2E_GROUP = int(os.environ.get("HIPGP_E2E_GROUP", "8"))     # right-hand sides in the first and the last group of the pipelined host solve
CPU_SAMPLE_B = 8       # right-hand sides per CPU step: ~7 s per step on 16 cores, so that --steps 20 --warmup 5 ends in ~3 minutes
N_MATVEC = 2 * MAXITER + 1
METRIC = "toeplitz_matvec_GBps_in_pcg_1e6grid"
DUMP_POINTS = 1 << 17  # grid points kept by --dump-outputs: 64 x 131072 fp32 = 32 MB


def workload_config():
    """identical in both arms (the driver compares it)"""
    return {"workload": "cfg2: 2D grid 1000x1000 (M=1e6), Matern-5/2 ell=0.01 jitter=1e-3, PCG maxiter=20 tol=1e-8 + HIP-GP preconditioner",
            "rhs_per_gpu_per_step": B_PER_GPU, "matvecs_per_step": N_MATVEC,
            "l2": "working set per GPU (5 vectors x 256 MB + 528 MB of half-spectra) exceeds the 126 MB L2; no flush needed"}


def alg_bytes_matvec(B, w=4):
    M = GRID[0] * GRID[1]
    E_h = (2 * GRID[0] - 2) * ((2 * GRID[1] - 2) // 2 + 1)
    return w * (2 * M * B + E_h)


def alg_bytes_pcg_iteration(B, w=4):
    """SURVEY.md 8d: w (13 M B + 2 E_h) -- both matvecs in / out plus the fully fused x, r, p updates and dots"""
    M = GRID[0] * GRID[1]
    E_h = (2 * GRID[0] - 2) * ((2 * GRID[1] - 2) // 2 + 1)
    return w * (13 * M * B + 2 * E_h)


def first_row(dtype, device):
    """k(u_0, u_.) for Matern-5/2 on linspace(0,4,1000) x linspace(-2,2,1000) (+ jitter at [0])."""
    import torch
    from hipgp_b200 import kernels as hk
    g1 = torch.linspace(0, 4, GRID[0], dtype=dtype, device=device)
    g2 = torch.linspace(-2, 2, GRID[1], dtype=dtype, device=device)
    return hk.first_row([g1, g2], hk.Matern(nu=2.5, dtype=dtype), (SIG2, ELL), jitter=JITTER)


def dump_outputs(path, x):
    """Writes the solution x (B, M) at the grid points np.random.default_rng(0).choice(M, DUMP_POINTS, replace=False),
    sorted, as path/pcg_x_sample.npy (B, DUMP_POINTS) in x's dtype."""
    import numpy as np
    import torch
    cols = np.sort(np.random.default_rng(0).choice(x.shape[1], min(DUMP_POINTS, x.shape[1]), replace=False))
    sample = x[:, torch.from_numpy(cols).to(x.device)].cpu().numpy()
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "pcg_x_sample.npy"), sample)


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.stop_flag, self.proc = index, [], False, None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.samples.append([t.strip() for t in line.split(",")])
        except Exception:
            pass

    def mark(self):
        return len(self.samples)

    def wait_running(self, timeout=5.0):
        t0 = time.time()
        while not self.samples and time.time() - t0 < timeout:
            time.sleep(0.01)

    def finish(self, lo=0, hi=None, lo_fallback=None, hi_fallback=None):
        """Samples [lo, hi) = the timed region; if that window holds fewer than 3 samples (a very short region) it is
        widened to [lo_fallback, hi_fallback) -- the same steps repeated under the same load -- and that is reported."""
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        window = "timed region"
        sel = self.samples[lo:hi]
        if len(sel) < 3 and lo_fallback is not None:
            sel = self.samples[lo_fallback:hi_fallback]
            window = "timed region + the e2e / roofline passes of the same step (timed region shorter than 3 sampling periods)"
        self.samples = sel
        self.window = window
        sm = sorted(int(float(s[0])) for s in self.samples if s and s[0].replace(".", "").isdigit())
        mx = [int(float(s[1])) for s in self.samples if len(s) > 1 and s[1].replace(".", "").isdigit()]
        reasons = set()
        for s in self.samples:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), s[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "window": getattr(self, "window", "")}


def host_threads():
    """threads for the CPU arm: the box's physical cores (what torch picks by default), within this process's affinity"""
    try:
        import psutil
        phys = psutil.cpu_count(logical=False) or os.cpu_count() or 1
    except Exception:
        phys = os.cpu_count() or 1
    try:
        phys = min(phys, len(os.sched_getaffinity(0)))
    except Exception:
        pass
    return max(1, int(phys))


# ---------------------------------------------------------------------------------------------------------------------
# CPU arm: the reference's own implementation of the path on the host cores
# ---------------------------------------------------------------------------------------------------------------------
def reference_step(B, threads):
    """Returns (step_fn, setup_seconds, kind).  kind = "reference": the unmodified ziggy.misc.toeplitz_tensor.ToeplitzTensor
    (its K matvec, its preconditioner, its conj_grad2) ; "port": the oracle restatement (staged reference absent)."""
    import torch
    torch.set_num_threads(threads)             # torchrun exports OMP_NUM_THREADS=1: the CPU arm still uses every core
    g1 = torch.linspace(0, 4, GRID[0]); g2 = torch.linspace(-2, 2, GRID[1])
    torch.manual_seed(42)
    v = torch.randn(B, GRID[0] * GRID[1])
    from oracle import ref_shim
    kind = "reference" if ref_shim.reference_root() is not None else "port"
    t0 = time.perf_counter()
    if kind == "reference":
        ref_shim.import_reference()
        from ziggy.misc.toeplitz_tensor import ToeplitzTensor
        from ziggy.kernels import Matern
        kern = Matern(nu=2.5, length_scale=ELL)
        kfun = lambda x, y: kern.forward(x, y, params=(SIG2, ELL))
        K = ToeplitzTensor(xgrids=[g1, g2], kernel=kfun, batch_shape=None, jitter_val=JITTER)
        solve = lambda: K._solve(v, do_precond=True, maxiter=MAXITER, tol=TOL)
    else:
        from oracle import ziggy_oracle as zo
        K = zo.OracleToeplitz([g1, g2], lambda x, y: zo.matern(x, y, SIG2, ELL, 2.5), jitter_val=JITTER)
        solve = lambda: K.solve(v, do_precond=True, maxiter=MAXITER, tol=TOL)
    t_setup = time.perf_counter() - t0

    def step():
        t = time.perf_counter()
        solve()
        return time.perf_counter() - t
    return step, t_setup, kind


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    B = args.cpu_sample_b
    cores = host_threads()
    step, t_setup, kind = reference_step(B, cores)
    for _ in range(args.warmup):
        step()
    ts = [step() for _ in range(args.steps)]
    t = sum(ts) / len(ts)
    val = N_MATVEC * alg_bytes_matvec(B) / t / 1e9
    line = {
        "impl": "reference", "metric": METRIC, "value": val, "unit": "GB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": t * 1e3,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "pcg_solve_s": t, "pcg_solve_s_per_rhs": t / B,
        "config": workload_config(),
        "cpu_baseline": {"value": val, "unit": "GB/s", "cores": cores, "kind": kind,
                         "sample": "%d of the step's %d right-hand sides x 20 PCG iterations on the full 10^6 grid per step (value = the sample's own "
                                   "algorithmic bytes / its time); spectrum set-up %.2f s not timed" % (B, B_PER_GPU, t_setup),
                         "what": ("unmodified reference: ziggy.misc.toeplitz_tensor.ToeplitzTensor._solve (oracle/_ref, torch CPU, all host threads)"
                                  if kind == "reference" else "CPU oracle port of the reference (oracle/ziggy_oracle.py; oracle/_ref not staged)")},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# The other BASELINE.json configurations, CPU (the reference itself, bounded samples) next to the GPU path at the full batch:
# (tag, grid, dtype, GPU right-hand sides, CPU sample, with R^T) -- op = PCG(20) + preconditioner [+ R^T = compute_kn, hipgp.py:139-146]
OTHER_CONFIGS = [("cfg1", (100, 100), "f32", 16, 16, False), ("cfg1", (100, 100), "f64", 16, 16, False),
                 ("cfg2", (1000, 1000), "f64", 16, 2, False),
                 ("cfg3", (300, 300), "f32", 200, 20, True),
                 ("cfg4", (128, 128, 64), "f32", 200, 1, True)]


def _other_grids(dims, dtype, device=None):
    import torch
    g = [torch.linspace(0, 1, m, dtype=dtype, device=device) for m in dims]
    return g, 2.5 / (dims[0] - 1)


def run_reference_other(args):
    """`--impl reference --other-configs`: one JSON list, the reference's ToeplitzTensor._solve (+ _matmul_by_RT) per config"""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    import torch
    cores = host_threads()
    torch.set_num_threads(cores)
    from oracle import ref_shim
    kind = "reference" if ref_shim.reference_root() is not None else "port"
    out = []
    for tag, dims, dn, _, Bc, with_rt in OTHER_CONFIGS:
        dtype = torch.float32 if dn == "f32" else torch.float64
        grids, ell = _other_grids(dims, dtype)
        torch.manual_seed(7)
        v = torch.randn(Bc, math.prod(dims), dtype=dtype)
        t0 = time.perf_counter()
        if kind == "reference":
            ref_shim.import_reference()
            from ziggy.misc.toeplitz_tensor import ToeplitzTensor
            from ziggy.kernels import Matern
            kern = Matern(nu=2.5, length_scale=ell)
            K = ToeplitzTensor(xgrids=grids, kernel=lambda x, y: kern.forward(x, y, params=(SIG2, ell)), batch_shape=None, jitter_val=JITTER)
            solve = lambda u: K._solve(u, do_precond=True, maxiter=MAXITER, tol=TOL)
            rt = lambda d: K._matmul_by_RT(d)
        else:
            from oracle import ziggy_oracle as zo
            K = zo.OracleToeplitz(grids, lambda x, y: zo.matern(x, y, SIG2, ell, 2.5), jitter_val=JITTER)
            solve = lambda u: K.solve(u, do_precond=True, maxiter=MAXITER, tol=TOL)
            rt = lambda d: K.matmul_RT(d)
        t_setup = time.perf_counter() - t0
        solve(v[:1])                                   # untimed first call
        t0 = time.perf_counter()
        d = solve(v)
        if with_rt:
            rt(d)
        t = time.perf_counter() - t0
        out.append({"config": tag, "grid": list(dims), "dtype": dn, "op": "PCG(20) + preconditioner" + (" + R^T (compute_kn)" if with_rt else ""),
                    "sample_rhs": Bc, "s": t, "s_per_rhs": t / Bc, "setup_s": t_setup, "cores": cores, "kind": kind})
    print(json.dumps(out), flush=True)


def other_configs_gpu(dev):
    """the same operations through the C ABI at the configuration's full batch (device-resident, CUDA events)"""
    import torch
    from hipgp_b200.plan import Plan
    from hipgp_b200 import _lib as L, kernels as hk
    out = {}
    for tag, dims, dn, Bg, _, with_rt in OTHER_CONFIGS:
        dtype = torch.float32 if dn == "f32" else torch.float64
        grids, ell = _other_grids(dims, dtype, dev)
        plan = Plan(list(dims), dtype, dev)
        plan.set_first_row(hk.first_row(grids, hk.Matern(nu=2.5, dtype=dtype), (SIG2, ell), jitter=JITTER))
        gen = torch.Generator(device=dev); gen.manual_seed(7)
        v = torch.randn(Bg, math.prod(dims), dtype=dtype, device=dev, generator=gen)

        def op():
            d = plan.pcg(v, maxiter=MAXITER, tol=TOL, precond=True)
            if with_rt:
                plan.matvec(L.MV_RT, d)
        op(); torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            op()
        e1.record(); torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / 3e3
        out[(tag, dn)] = {"rhs": Bg, "s": t, "s_per_rhs": t / Bg}
        del plan, v
        torch.cuda.empty_cache()
    return out


# ---------------------------------------------------------------------------------------------------------------------
# the two multi-GPU paths that need collectives (extra keys of the N > 1 line; also run at N = 1 as the reference point)
# ---------------------------------------------------------------------------------------------------------------------
def svi_cfg3_section(dev, world, rank, steps=20):
    """BASELINE config 3: 300x300 grid, Matern-3/2, 200-observation minibatches, mean-field natural-gradient step
    (K_xu on the fly -> 20-iteration PCG -> R^T -> fused statistics), observations of every minibatch sharded over the
    ranks, ONE packed all-reduce [data_dm; lam_sum; sum a_n] per step (hipgp.py:194-276)."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from hipgp_b200 import hipgp as hh, kernels as hk
    dtype = torch.float32
    bsz = 200
    xgrids = [torch.linspace(-5.7, 1.8, 300, dtype=dtype), torch.linspace(50, 55.5, 300, dtype=dtype)]
    mod = hh.MeanFieldToeplitzGP(hk.Matern(nu=1.5, dtype=dtype), xgrids, num_obs=2_000_000, sig2_init=1.0, ell_init=0.05,
                                 dtype=dtype, jitter_val=1e-3).cuda_params(dev.index)
    opt = torch.optim.SGD([mod.global_theta1, mod.global_theta2], lr=1e-4)
    rs = np.random.RandomState(42)

    def make_data(b):
        n = (steps + 3) * b
        X = torch.from_numpy(np.stack([rs.uniform(-5.7, 1.8, n), rs.uniform(50, 55.5, n)], 1)).to(dtype).pin_memory()
        Y = torch.from_numpy(rs.randn(n, 1)).to(dtype).pin_memory()
        NS = torch.full((n, 1), 0.3, dtype=dtype).pin_memory()
        return X, Y, NS

    def timed(shard, b, data):
        X, Y, NS = data

        def step(i):
            sl = slice(i * b, (i + 1) * b)
            xb = X[sl].to(dev, non_blocking=True); yb = Y[sl].to(dev, non_blocking=True); nb = NS[sl].to(dev, non_blocking=True)
            el = mod.elbo_and_grad(xb, yb, nb, maxiter_cg=20, shard=shard)
            opt.step()
            return el
        for i in range(3):
            step(i)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            step(3 + i)
        e1.record(); torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())
    data = make_data(bsz)
    ms_n = timed(True, bsz, data)          # the reference's minibatch of 200, sharded over the ranks (strong scaling of one step)
    out = {"ms_per_step": ms_n, "obs_per_s": bsz / (ms_n / 1e3), "batch_size": bsz, "maxiter_cg": 20, "steps": steps, "dtype": "f32",
           "allreduce_bytes": int((2 * mod.Mprime + 1) * 4) if world > 1 else 0, "n_gpus": world,
           "epoch_s_extrapolated_2M_obs": 2_000_000 / bsz * ms_n / 1e3}
    if world > 1:
        ms_1 = timed(False, bsz, data)     # every rank runs the WHOLE minibatch: the one-GPU step, measured in the same run
        out["ms_per_step_1gpu_same_run"] = ms_1
        out["speedup_vs_1gpu"] = ms_1 / ms_n
        out["efficiency_vs_n1"] = ms_1 / ms_n / world
        # weak scaling: 200 observations PER RANK per step (a minibatch of 200 x N): same kernels at the batch they are sized for
        ms_w = timed(True, bsz * world, make_data(bsz * world))
        out["weak"] = {"batch_size": bsz * world, "ms_per_step": ms_w, "obs_per_s": bsz * world / (ms_w / 1e3), "efficiency_vs_n1": ms_1 / ms_w}
        out["note"] = ("strong scaling of a 200-observation step leaves %d observations per rank: 126 pass-kernel launches of ~25 us each are "
                       "then bound by per-launch fixed costs (measured: GPU busy 3.36 of 3.48 ms at 25 observations on one GPU)" % (bsz // world))
    return out


def slab_cfg5_section(dev, world, rank):
    """BASELINE config 5: 512^3 grid (134M inducing points), K matvec and PCG(20) with the grid sharded over the ranks
    (slab decomposition along axis 0, two all-to-all transposes per matvec); strong scaling against the undecomposed
    one-GPU plan measured on rank 0 in the same run."""
    import torch
    import torch.distributed as dist
    from hipgp_b200.plan import Plan
    from hipgp_b200.slab import SlabToeplitz
    from hipgp_b200 import _lib as L, kernels as hk
    dtype = torch.float32
    dims = (512, 512, 512)
    xg = [torch.linspace(0, 1, m, dtype=dtype, device=dev) for m in dims]
    h = float(xg[0][1] - xg[0][0])
    col = hk.first_row(xg, hk.Matern(nu=2.5, dtype=dtype), (1.0, 2.5 * h), jitter=1e-3)

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    def timed(fn, n, warm=2):
        for _ in range(warm):
            fn()
        sync_all()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record(); torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1) / n], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    out = {"grid": list(dims), "n_gpus": world, "dtype": "f32"}
    # one-GPU reference point: the undecomposed plan (rank 0 measures, the others wait)
    one = torch.zeros(2, device=dev, dtype=torch.float64)
    if rank == 0:
        plan = Plan(list(dims), dtype, dev).set_first_row(col)
        v = torch.randn(1, dims[0] * dims[1] * dims[2], dtype=dtype, device=dev)
        for _ in range(2):
            plan.matvec(L.MV_K, v)
        torch.cuda.synchronize()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            plan.matvec(L.MV_K, v)
        e1.record(); torch.cuda.synchronize()
        one[0] = e0.elapsed_time(e1) / 5
        plan.pcg(v, maxiter=MAXITER, tol=TOL)
        torch.cuda.synchronize()
        e0.record(); plan.pcg(v, maxiter=MAXITER, tol=TOL); e1.record(); torch.cuda.synchronize()
        one[1] = e0.elapsed_time(e1) / 1e3
        del plan, v
        torch.cuda.empty_cache()
    if world > 1:
        dist.broadcast(one, src=0)
    out["matvec_ms_1gpu_undecomposed"] = float(one[0]); out["pcg20_s_1gpu_undecomposed"] = float(one[1])
    if world == 1:
        out["matvec_ms"] = float(one[0]); out["pcg20_s"] = float(one[1])
        return out
    try:
        slab = SlabToeplitz(dims, col, dtype, dev)
    except Exception as e:      # e.g. inter-process memory handles unavailable on this box: the NCCL exchange still works
        out["peer_exchange_error"] = repr(e)[:200]
        slab = SlabToeplitz(dims, col, dtype, dev, exchange="nccl")
    gen = torch.Generator(device=dev); gen.manual_seed(42 + rank)      # counter-based per-slab stream (SURVEY 8d)
    vs = torch.randn(slab.slab_elems, dtype=dtype, device=dev, generator=gen)
    out["matvec_ms"] = timed(lambda: slab.matvec_K(vs), 10)
    out["layout"] = slab.layout; out["exchange"] = slab.exchange; out["chunks"] = slab.chunks
    out["pcg20_s"] = timed(lambda: slab.solve(vs, do_precond=True, maxiter=MAXITER, tol=TOL), 1, warm=1) / 1e3
    esz = 8
    sent = slab.exch_elems * esz * (world - 1) // world               # bytes that leave this GPU per transpose
    if slab.exchange == "peer":
        # the transfer kernels alone (16-byte stores into the peers' buffers), as the matvec launches them once each way
        p0 = slab.plans[0]
        import ctypes as C
        from hipgp_b200.plan import _stream_ptr

        def push(back):
            L.check(p0.lib, p0.lib.hipgp_slab2_push_only(p0._h, back, _stream_ptr(dev)))
        x_ms = 0.5 * (timed(lambda: push(0), 10) + timed(lambda: push(1), 10))
        out["exchange_how"] = "packing kernels store into the peers' receive buffers (CUDA IPC mappings over NVLink); 2 all-reduce barriers per matvec"
    else:
        buf = torch.empty(slab.exch_elems, dtype=slab.cdtype, device=dev); rcv = torch.empty_like(buf)
        x_ms = timed(lambda: dist.all_to_all_single(torch.view_as_real(rcv), torch.view_as_real(buf)), 10)
        out["exchange_how"] = "NCCL all_to_all_single between the stages"
    # the same bytes through NCCL's all-to-all, for comparison
    buf = torch.empty(slab.exch_elems, dtype=slab.cdtype, device=dev); rcv = torch.empty_like(buf)
    out["nccl_alltoall_ms_same_bytes"] = timed(lambda: dist.all_to_all_single(torch.view_as_real(rcv), torch.view_as_real(buf)), 10)
    del buf, rcv
    out.update({"alltoall_bytes_per_rank": int(sent), "alltoalls_per_matvec": 2, "alltoall_ms": x_ms,
                "nvlink_GBps_achieved": sent / (x_ms / 1e3) / 1e9, "nvlink_frac_of_900": sent / (x_ms / 1e3) / 1e9 / 900.0,
                "alltoall_share_of_matvec": 2 * x_ms / out["matvec_ms"],
                "strong_speedup_vs_1gpu": float(one[0]) / out["matvec_ms"],
                "strong_eff_vs_1gpu": float(one[0]) / out["matvec_ms"] / world,
                "pcg_strong_eff_vs_1gpu": float(one[1]) / out["pcg20_s"] / world})
    return out


# ---------------------------------------------------------------------------------------------------------------------
def run_gpu(args):
    import torch
    import torch.distributed as dist
    from hipgp_b200.plan import Plan
    from hipgp_b200 import _lib as L

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # several ranks on one node: keep this rank's pinned buffers on the GPU's NUMA node (N = 1 keeps every core for the CPU leg)
    numa = None
    if world > 1:
        from hipgp_b200.hostmem import bind_to_gpu_numa_node
        numa = bind_to_gpu_numa_node(local)

    dtype = torch.float32
    B = B_PER_GPU
    M = GRID[0] * GRID[1]
    warmup = max(args.warmup, 3)
    plan = Plan(GRID, dtype, dev)
    plan.set_first_row(first_row(dtype, dev))
    gen = torch.Generator(device=dev); gen.manual_seed(42 + rank)
    b = torch.randn(B, M, dtype=dtype, device=dev, generator=gen)
    b_host = b.cpu().pin_memory()
    x_host = torch.empty_like(b_host).pin_memory()

    def step_dev():
        return plan.pcg(b, maxiter=MAXITER, tol=TOL, precond=True)

    last = [None]

    def step_dev_kept():          # --dump-outputs: the timed steps keep what they return
        last[0] = step_dev()

    def step_e2e():
        return plan.pcg_host(b_host, x_host, maxiter=MAXITER, tol=TOL, precond=True, group=E2E_GROUP)

    def timed(fn, steps):
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
        sampler.wait_running()
    for _ in range(warmup):
        step_dev()
    m0 = sampler.mark() if sampler else 0
    l0 = plan.launch_count()
    ms_total = timed(step_dev_kept if args.dump_outputs else step_dev, args.steps)
    launches = plan.launch_count() - l0
    m1 = sampler.mark() if sampler else 0
    x_timed, last[0] = last[0], None      # what the last timed step returned (None without --dump-outputs)

    # e2e (headline): a stream of `steps` batches through the asynchronous host entry points, two in flight -- every step's
    # right-hand sides are uploaded from pinned memory and its solution downloaded inside the timed region; the upload of step
    # k+1 and the download of step k-1 travel under the solve of step k.  The end event is recorded after the host has waited
    # for the last download.
    x_hosts = [x_host, torch.empty_like(b_host).pin_memory()]

    def stream_e2e(steps):
        plan.pcg_host_submit(b_host, x_hosts[0], 0, maxiter=MAXITER, tol=TOL, precond=True)
        for k in range(1, steps):
            plan.pcg_host_submit(b_host, x_hosts[k % 2], k % 2, maxiter=MAXITER, tol=TOL, precond=True)
            plan.pcg_host_wait((k - 1) % 2)
        plan.pcg_host_wait((steps - 1) % 2)

    stream_e2e(2)
    barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    stream_e2e(args.steps)
    e1.record()
    barrier()
    ms_t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms_t.item())
    xd = step_dev()
    xd_host = xd.cpu()
    e2e_matches = bool(torch.equal(xd_host, x_hosts[0])) and bool(torch.equal(xd_host, x_hosts[1]))
    # one synchronous call per step (hipgp_pcg_host_pipelined: the copies hide inside ONE step, groups of 8 / 48 / 8)
    for _ in range(2):
        step_e2e()
    ms_e2e_sync = timed(step_e2e, max(2, args.steps // 4))
    ms_e2e_sync_step = ms_e2e_sync / max(2, args.steps // 4)
    e2e_matches = e2e_matches and bool(torch.equal(xd_host, x_host))

    # roofline pass: same steps with per-kernel-class events on
    plan.profile(True)
    plan.profile_read(reset=True)
    for _ in range(args.steps):
        step_dev()
    prof = plan.profile_read(reset=True)
    plan.profile(False)
    m2 = sampler.mark() if sampler else 0
    clocks = sampler.finish(m0, m1, m0, m2) if sampler else None
    if x_timed is not None and rank == 0:
        dump_outputs(args.dump_outputs, x_timed)
    del x_timed

    # companions (not the headline; same step definition): one right-hand side, plain matvecs, fp64, cuFFT comparison point
    extra = {}
    if world == 1 and not args.quick:          # single-GPU run only: `timed` synchronises all ranks
        nrep = max(5, min(args.steps, 20))
        b16 = b[:16].contiguous(); b1 = b[:1].contiguous()
        for _ in range(3):
            plan.pcg(b1, maxiter=MAXITER, tol=TOL)
        extra["pcg_solve_s_B1_f32"] = timed(lambda: plan.pcg(b1, maxiter=MAXITER, tol=TOL), nrep) / nrep / 1e3
        for _ in range(2):
            plan.pcg(b16, maxiter=MAXITER, tol=TOL)
        extra["pcg_solve_s_B16_f32"] = timed(lambda: plan.pcg(b16, maxiter=MAXITER, tol=TOL), nrep) / nrep / 1e3
        for mode, nm in ((L.MV_K, "K"), (L.MV_CINV, "Cinv"), (L.MV_RT, "RT")):
            for _ in range(3):
                plan.matvec(mode, b16)
            extra["matvec_ms_B16_f32_" + nm] = timed(lambda: plan.matvec(mode, b16), nrep) / nrep
        extra["matvec_GBps_B16_f32_K"] = alg_bytes_matvec(16) / extra["matvec_ms_B16_f32_K"] / 1e6
        t0 = time.perf_counter(); plan.set_first_row(first_row(dtype, dev)); torch.cuda.synchronize()
        extra["spectrum_setup_ms_f32"] = (time.perf_counter() - t0) * 1e3
        # cuFFT comparison point (library FFTs through torch.fft: rfft2 -> spectrum multiply -> irfft2 -> crop; same embedding)
        Lf = plan.embedding()[0]
        S = torch.rand(Lf[0], Lf[1] // 2 + 1, dtype=dtype, device=dev)
        def cufft_mv():
            F = torch.fft.rfft2(b16.view(16, GRID[0], GRID[1]), s=(Lf[0], Lf[1]))
            return torch.fft.irfft2(F * S, s=(Lf[0], Lf[1]))[:, :GRID[0], :GRID[1]]
        for _ in range(3):
            cufft_mv()
        extra["cufft_comparison_matvec_ms_B16_f32"] = timed(cufft_mv, nrep) / nrep
        del S
        # fp64 (BASELINE config 2 names both precisions)
        plan64 = Plan(GRID, torch.float64, dev).set_first_row(first_row(torch.float64, dev))
        b64 = b16.double()
        for _ in range(3):
            plan64.matvec(L.MV_K, b64)
        extra["matvec_ms_B16_f64_K"] = timed(lambda: plan64.matvec(L.MV_K, b64), nrep) / nrep
        extra["matvec_GBps_B16_f64_K"] = alg_bytes_matvec(16, 8) / extra["matvec_ms_B16_f64_K"] / 1e6
        plan64.pcg(b64, maxiter=MAXITER, tol=TOL)
        extra["pcg_solve_s_B16_f64"] = timed(lambda: plan64.pcg(b64, maxiter=MAXITER, tol=TOL), 5) / 5 / 1e3
        extra["toeplitz_matvec_GBps_in_pcg_f64"] = N_MATVEC * alg_bytes_matvec(16, 8) / extra["pcg_solve_s_B16_f64"] / 1e9
        del plan64, b64
        torch.cuda.empty_cache()
    if world > 1:
        dist.barrier()

    line = None
    if rank == 0:
        t_step = ms_total / args.steps / 1e3
        alg_step = N_MATVEC * alg_bytes_matvec(B) * world
        value = alg_step / t_step / 1e9
        e2e_val = alg_step / (ms_e2e / args.steps / 1e3) / 1e9
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        per = {k: (v[0] / v[1] if v[1] else 0.0) for k, v in prof.items()}
        mv_ms = per["rows_fwd"] + per["cols_pass"] + per["rows_inv"]
        dom = max(("rows_fwd", "cols_pass", "rows_inv"), key=lambda k: per[k])
        achieved = alg_bytes_matvec(B) / (mv_ms / 1e3) / 1e9 if mv_ms > 0 else 0.0
        traffic, traffic_source = None, None
        tpath = os.path.join(ROOT, "profiles", "traffic_r2.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                traffic = tj.get("dram_bytes_per_matvec_B16_f32") * (B / 16.0)      # measured at B = 16; bytes scale with the batch
                traffic_source = tj.get("source")
            except Exception:
                traffic = None
        # bounded CPU sample on this box's host cores (rank 0, N = 1 only): the reference arm of this script, one warm-up + one step
        cpu = None
        if world == 1 and not args.no_cpu:
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                                   capture_output=True, text=True, timeout=900)
                cpu = json.loads(r.stdout.strip().splitlines()[-1])["cpu_baseline"]
            except Exception as e:
                cpu = {"error": repr(e)[:200]}
        # the other configurations: reference on the host cores (bounded samples) next to the CUDA path at the full batch
        others = None
        if world == 1 and not args.no_cpu and not args.quick:
            try:
                g_o = other_configs_gpu(dev)
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--impl", "reference", "--other-configs"],
                                   capture_output=True, text=True, timeout=600)
                others = json.loads(r.stdout.strip().splitlines()[-1])
                for o in others:
                    g = g_o[(o["config"], o["dtype"])]
                    o["cpu"] = {k: o.pop(k) for k in ("sample_rhs", "s", "s_per_rhs", "setup_s", "cores", "kind")}
                    o["gpu"] = g
                    o["speedup_per_rhs"] = o["cpu"]["s_per_rhs"] / g["s_per_rhs"]
            except Exception as e:
                others = {"error": repr(e)[:200]}
        # per-pass streaming bytes (DESIGN.md section 4: what each pass moves when its input / output do not stay on chip),
        # averaged over the launches of one PCG iteration, against the same HBM peak
        Mv = 4 * GRID[0] * GRID[1] * B                                   # one vector, all right-hand sides
        Wb = 8 * GRID[0] * ((2 * GRID[1] - 2) // 2 + 1) * B              # half-spectrum workspace of the pruned rows
        spec_b = 4 * plan.embedding()[0][0] * ((2 * GRID[1] - 2) // 2 + 1)
        stream = {"rows_fwd": (3 * Mv + Wb + 6 * Mv + Wb) / 2.0,         # p = z + beta p | x += a p, r -= a Ap, r.r
                  "cols_pass": 2 * Wb + spec_b,
                  "rows_inv": Wb + 2 * Mv}                               # write result, read the dot operand
        per_kernel = {k: {"streaming_bytes": stream[k], "ms": per[k],
                          "achieved_GBps": stream[k] / (per[k] / 1e3) / 1e9 if per[k] > 0 else None,
                          "frac_of_hbm_peak": stream[k] / (per[k] / 1e3) / 1e9 / peak if per[k] > 0 else None} for k in stream}
        it_frac = MAXITER * alg_bytes_pcg_iteration(B) / t_step / 1e9 / peak
        cfg = workload_config()
        line = {
            "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world,
            "steps": args.steps, "warmup": warmup, "ms_per_step": ms_total / args.steps,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "pcg_solve_s": t_step, "pcg_solve_s_per_rhs": t_step / B,
            "config": cfg,
            "parallelism": "rhs-sharded x%d, no data-path collective (the collective-bearing paths are the svi_cfg3 / slab_cfg5 keys)" % world,
            "embedding": list(plan.embedding()[0]),
            "e2e": {"value": e2e_val, "unit": "GB/s", "h2d_bytes_per_step": int(b_host.numel() * 4) * world,
                    "d2h_bytes_per_step": int(x_host.numel() * 4) * world, "ms_per_step": ms_e2e / args.steps,
                    "how": "hipgp_pcg_host_submit / _wait, two batches in flight: every step uploads its right-hand sides from pinned host memory "
                           "and downloads its solution; the copies of neighbouring steps run on two copy streams under the current solve",
                    "matches_device_path_bitwise": e2e_matches, "frac_of_value": e2e_val / value if value else None,
                    "one_synchronous_call_per_step": {"ms_per_step": ms_e2e_sync_step, "value": alg_step / (ms_e2e_sync_step / 1e3) / 1e9,
                                                      "how": "hipgp_pcg_host_pipelined: groups of %d / %d / %d right-hand sides inside one call" % (E2E_GROUP, B_PER_GPU - 2 * E2E_GROUP, E2E_GROUP)},
                    "host_numa": numa},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak if peak else None, "traffic": traffic, "traffic_source": traffic_source,
                         "peak_source": "MEASURED_PEAKS.json hbm_gbs" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                         "kernel": dom, "kernel_share_of_matvec": per[dom] / mv_ms if mv_ms else None,
                         "per_launch_ms": per, "algorithmic_bytes_per_matvec": alg_bytes_matvec(B), "per_kernel_streaming": per_kernel,
                         "pcg_iteration_contract_frac": it_frac,
                         "note": "achieved = contract bytes w(2MB+E_h) of one matvec / (rows_fwd + cols_pass + rows_inv average launch durations), CUDA events around every launch in a second pass of the same steps; the contract figure assumes the half-spectrum never leaves the chip -- per_kernel_streaming gives each pass against the bytes it actually has to stream; pcg_iteration_contract_frac = 20 x w(13MB+2E_h) / step time / peak; the passes are bound by FP32 issue (2 cycles per packed op) + shared-memory exchange, not by HBM (DESIGN.md 4a, profiles/README.md r2)"},
            "cpu_baseline": cpu,
            "cpu_baselines_other_configs": others,
        }
        line.update(extra)

    # the collective-bearing multi-GPU paths (and their one-GPU reference points).  A watchdog guarantees the headline
    # line: if a section hangs (a rank lost in a collective) rank 0 prints what it has and every rank leaves.
    if not args.quick and not args.no_multi:
        def bail():
            if rank == 0:
                line["sections_error"] = "a multi-GPU section exceeded %d s; headline printed without it" % args.section_timeout
                print(json.dumps(line), flush=True)
            os._exit(0)
        wd = threading.Timer(args.section_timeout, bail)
        wd.daemon = True
        wd.start()
        del b
        torch.cuda.empty_cache()
        for name, fn in (("svi_cfg3", lambda: svi_cfg3_section(dev, world, rank)), ("slab_cfg5", lambda: slab_cfg5_section(dev, world, rank))):
            try:
                res = fn()
            except Exception as e:   # the headline must survive a failure of a companion section
                res = {"error": repr(e)[:300]}
                if world > 1:        # the other ranks may be inside a collective: leave through the watchdog path
                    if rank == 0:
                        line[name] = res
                    bail()
            if rank == 0:
                line[name] = res
            torch.cuda.empty_cache()
        wd.cancel()
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--quick", action="store_true", help="skip the companion measurements and the multi-GPU sections")
    ap.add_argument("--no-cpu", action="store_true", help="skip the CPU baseline sample")
    ap.add_argument("--no-multi", action="store_true", help="skip the svi_cfg3 / slab_cfg5 sections")
    ap.add_argument("--other-configs", action="store_true", help="with --impl reference: time the other BASELINE configurations instead")
    ap.add_argument("--section-timeout", type=int, default=420, help="watchdog for the multi-GPU sections (seconds)")
    ap.add_argument("--cpu-sample-b", type=int, default=CPU_SAMPLE_B, help="right-hand sides per CPU step (bounded sample)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's solution to DIR/*.npy (rank 0's right-hand sides)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's outputs; it does not apply to --impl reference")
    if args.impl == "reference":
        if args.other_configs:
            run_reference_other(args)
        else:
            run_reference(args)
        return
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback); use --impl reference for the CPU arm")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: re-launch under torchrun
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(args.gpus),
               "--master-addr", "127.0.0.1", "--master-port", "29511", os.path.abspath(__file__)] + sys.argv[1:]
        raise SystemExit(subprocess.call(cmd))
    run_gpu(args)


if __name__ == "__main__":
    main()
