"""Slab-decomposed structured K_uu for grids sharded over several GPUs (SURVEY.md 8e, BASELINE config 5).

Axis 0 of a 3-D grid is split contiguously over the ranks.  A matvec is three local stages with two all-to-all
transposes between them.  What travels is the UN-PADDED output of the row pass, split along the bins of the last axis; after
the exchange a rank owns every (i0, i1) for its bins and runs the three ordinary column passes locally.
  exchange="peer" (default): no collective library on the data path -- the packing kernels store the blocks straight into
      the peers' receive buffers over NVLink; exchange="nccl": all_to_all_single (torch.distributed), cut into `chunks`
      overlapped pieces (default 2).

PCG on slab vectors is the reference's conj_grad2 with the dot products summed over ranks (one small all-reduce per dot).

`SlabToeplitz.matvec_K/_Cinv(v_slab)`: v_slab is this rank's (n0/P, m1, m2) block, flattened or not.
`emulate=True` runs all ranks inside one process on one GPU (lists of slabs in, lists out) -- used by the tests.
"""
import ctypes as C

import torch
import torch.distributed as dist

from . import _lib as L
from .plan import Plan, _stream_ptr
from .cg import conj_grad2


class SlabToeplitz:
    def __init__(self, dims, column, dtype, device, rank=None, nranks=None, emulate_ranks=None, chunks=None, exchange=None):
        assert len(dims) == 3, "slab decomposition is implemented for 3-D grids"
        # how the blocks travel: "peer" = the packing kernels store straight into the peers' receive buffers over NVLink (CUDA
        # inter-process handles, two small all-reduces per matvec as barriers); "nccl" = all_to_all_single between the stages
        exchange = exchange or "peer"
        assert exchange in ("peer", "nccl")
        self.exchange = exchange
        # cut the exchange into `chunks` independent all-to-alls so that the column passes of one chunk run while its
        # neighbours are on the wire (NCCL's stream next to the compute stream)
        self.chunks = int(chunks or (1 if exchange == "peer" else 2))
        self.dims = tuple(int(d) for d in dims)
        self.emulated = emulate_ranks is not None
        if self.emulated:
            self.nranks = int(emulate_ranks); ranks = range(self.nranks)
        else:
            self.nranks = nranks if nranks is not None else (dist.get_world_size() if dist.is_initialized() else 1)
            ranks = [rank if rank is not None else (dist.get_rank() if dist.is_initialized() else 0)]
        self.plans = []
        for r in ranks:
            p = Plan(self.dims, dtype, device)
            L.check(p.lib, p.lib.hipgp_plan_set_slab(p._h, r, self.nranks))
            if self.chunks > 1:
                L.check(p.lib, p.lib.hipgp_plan_set_slab_chunks(p._h, self.chunks))
            p.set_first_row(column)
            self.plans.append(p)
        p0 = self.plans[0]
        a, b = C.c_int64(), C.c_int64()
        L.check(p0.lib, p0.lib.hipgp_slab2_sizes(p0._h, C.byref(a), C.byref(b)))
        self.slab_elems, self.exch_elems = a.value, b.value
        self.dtype, self.device = dtype, p0.device
        self.cdtype = torch.complex64 if dtype == torch.float32 else torch.complex128
        self.slab_shape = (self.dims[0] // self.nranks, self.dims[1], self.dims[2])
        if self.exchange == "peer":
            self._connect_peers()

    @property
    def layout(self):
        """what travels between the stages: the row pass's un-padded output split along the last-axis bins"""
        return "bins"

    def _connect_peers(self):
        """every rank allocates its two receive buffers and maps everybody else's"""
        P = self.nranks
        r1 = [C.c_void_p() for _ in self.plans]; r2 = [C.c_void_p() for _ in self.plans]
        h1 = [(C.c_ubyte * 64)() for _ in self.plans]; h2 = [(C.c_ubyte * 64)() for _ in self.plans]
        for i, p in enumerate(self.plans):
            L.check(p.lib, p.lib.hipgp_slab2_peer_alloc(p._h, C.byref(r1[i]), C.byref(r2[i]), h1[i], h2[i]))
        if self.emulated or P == 1:
            a1 = (C.c_void_p * P)(*[x.value for x in r1]) if self.emulated else (C.c_void_p * 1)(r1[0].value)
            a2 = (C.c_void_p * P)(*[x.value for x in r2]) if self.emulated else (C.c_void_p * 1)(r2[0].value)
            for p in self.plans:
                L.check(p.lib, p.lib.hipgp_slab2_peer_set(p._h, a1, a2))
            self._tok = None
            return
        mine = torch.tensor(list(bytes(h1[0])) + list(bytes(h2[0])), dtype=torch.uint8, device=self.device)
        allh = torch.empty(P * 128, dtype=torch.uint8, device=self.device)
        dist.all_gather_into_tensor(allh, mine)
        allh = allh.cpu().numpy().reshape(P, 2, 64)
        b1 = allh[:, 0, :].tobytes(); b2 = allh[:, 1, :].tobytes()
        p = self.plans[0]
        L.check(p.lib, p.lib.hipgp_slab2_peer_open(p._h, b1, b2))
        self._tok = torch.zeros(1, dtype=torch.float32, device=self.device)
        dist.all_reduce(self._tok)      # nobody pushes before everybody has mapped the buffers
        torch.cuda.synchronize(self.device)

    def _rank_barrier(self):
        """stream-ordered: work queued after it starts only when every rank's earlier work on its stream is complete"""
        if self._tok is not None:
            dist.all_reduce(self._tok)

    def _matvec_peer(self, mode, vs):
        st = _stream_ptr(self.device)
        for p, x in zip(self.plans, vs):
            x = x.reshape(-1).to(self.dtype).contiguous()
            L.check(p.lib, p.lib.hipgp_slab2_push_a(p._h, C.c_void_p(x.data_ptr()), st))
        self._rank_barrier()
        for p in self.plans:
            L.check(p.lib, p.lib.hipgp_slab2_push_b(p._h, mode, -1, st))
        self._rank_barrier()
        outs = []
        for p in self.plans:
            out = torch.empty(self.slab_elems, dtype=self.dtype, device=self.device)
            L.check(p.lib, p.lib.hipgp_slab2_finish(p._h, C.c_void_p(out.data_ptr()), st))
            outs.append(out)
        return outs

    # ---- stages -------------------------------------------------------------------------------------
    def _s1(self, p, v):
        send = torch.empty(self.exch_elems, dtype=self.cdtype, device=self.device)
        v = v.reshape(-1).to(self.dtype).contiguous()
        L.check(p.lib, p.lib.hipgp_slab2_stage_a(p._h, C.c_void_p(v.data_ptr()), C.c_void_p(send.data_ptr()), _stream_ptr(self.device)))
        return send

    def _s2(self, p, mode, buf, chunk=-1):
        L.check(p.lib, p.lib.hipgp_slab2_stage_b_chunk(p._h, mode, C.c_void_p(buf.data_ptr()), chunk, _stream_ptr(self.device)))
        return buf

    def _s3(self, p, buf):
        out = torch.empty(self.slab_elems, dtype=self.dtype, device=self.device)
        L.check(p.lib, p.lib.hipgp_slab2_stage_c(p._h, C.c_void_p(buf.data_ptr()), C.c_void_p(out.data_ptr()), _stream_ptr(self.device)))
        return out

    def _exchange(self, bufs):
        """all-to-all of equal blocks (per chunk); `bufs` is a list with one buffer per local (or emulated) rank"""
        if self.emulated:
            nch = self.chunks; per = self.exch_elems // nch; blk = per // self.nranks
            return [torch.cat([bufs[q][c * per + r * blk:c * per + (r + 1) * blk] for c in range(nch) for q in range(self.nranks)])
                    for r in range(self.nranks)]
        if self.nranks == 1:
            return bufs
        recv = torch.empty_like(bufs[0])
        per = self.exch_elems // self.chunks
        for c in range(self.chunks):
            dist.all_to_all_single(torch.view_as_real(recv[c * per:(c + 1) * per]), torch.view_as_real(bufs[0][c * per:(c + 1) * per]))
        return [recv]

    def _matvec_overlapped(self, mode, v):
        """several chunks, one rank per process: chunk c's column passes run while chunk c+1 arrives and chunk
        c-1 already travels back (the collectives sit on NCCL's stream, ordered among themselves as issued)."""
        p = self.plans[0]
        per = self.exch_elems // self.chunks
        send = self._s1(p, v)
        recv = torch.empty_like(send)
        cut = lambda t, c: torch.view_as_real(t[c * per:(c + 1) * per])
        there = [dist.all_to_all_single(cut(recv, c), cut(send, c), async_op=True) for c in range(self.chunks)]
        back = []
        for c in range(self.chunks):
            there[c].wait()
            self._s2(p, mode, recv, c)
            # chunk c of `send` has left (its all-to-all is complete): it receives the way back
            back.append(dist.all_to_all_single(cut(send, c), cut(recv, c), async_op=True))
        for w in back:
            w.wait()
        return self._s3(p, send)

    def matvec(self, mode, v):
        """v: this rank's slab (emulated: list of slabs, one per rank); returns the result slab(s), flattened."""
        vs = v if self.emulated else [v]
        with torch.cuda.device(self.device):
            if self.exchange == "peer":
                outs = self._matvec_peer(mode, vs)
                return outs if self.emulated else outs[0]
            if not self.emulated and self.nranks > 1 and self.chunks > 1:
                return self._matvec_overlapped(mode, v)
            bufs = self._exchange([self._s1(p, x) for p, x in zip(self.plans, vs)])
            bufs = self._exchange([self._s2(p, mode, b) for p, b in zip(self.plans, bufs)])
            outs = [self._s3(p, b) for p, b in zip(self.plans, bufs)]
        return outs if self.emulated else outs[0]

    def matvec_K(self, v):
        return self.matvec(L.MV_K, v)

    def matvec_Cinv(self, v):
        return self.matvec(L.MV_CINV, v)

    # ---- distributed PCG on slab vectors -----------------------------------------------------------
    def solve(self, b_slab, do_precond=True, maxiter=20, tol=1e-8, callback=None, check_every=5):
        """K^-1 b with b sharded like the grid (one right-hand side); the stopping rule and the iterates are those of
        ziggy/misc/cg.py:44-80 with the dot products summed over ranks.

        The loop never waits for the device inside an iteration: the reference's `break` is a device-side flag that turns every
        later update into a no-op (so x is the reference's iterate at the iteration it would have stopped), and the host
        looks at the flag every `check_every` iterations only to stop launching.  Two small all-reduces per iteration
        (p.Ap, then r.r and z.r together).  `self.last_iters` holds the iteration count afterwards.
        A `callback` needs the iterate on the host each iteration: that case takes the generic synchronous loop."""
        assert not self.emulated, "solve() runs one rank per process"
        A = lambda v: self.matvec_K(v.reshape(-1)).reshape(1, -1)
        Pm = (lambda v: self.matvec_Cinv(v.reshape(-1)).reshape(1, -1)) if do_precond else None
        multi = self.nranks > 1
        red = (lambda t: dist.all_reduce(t)) if multi else (lambda t: t)
        if callback is not None:
            return conj_grad2(A, b_slab.reshape(1, -1).to(self.dtype), precond=Pm, maxiter=maxiter, tol=tol, callback=callback,
                              reduce=red)
        p0 = self.plans[0]; lib = p0.lib
        dt = L.F32 if self.dtype == torch.float32 else L.F64
        dev = self.device
        ptr = lambda t: C.c_void_p(t.data_ptr())
        with torch.cuda.device(dev):
            st = lambda: _stream_ptr(dev)
            b = b_slab.reshape(1, -1).to(self.dtype).contiguous()
            M = b.shape[1]
            x = torch.zeros_like(b)
            r = b.clone()                                   # r = b - K 0
            z = Pm(r) if Pm is not None else r
            p = z.clone()
            f64 = dict(dtype=torch.float64, device=dev)
            rs = torch.empty(1, **f64); pAp = torch.empty(1, **f64); sc = torch.empty(2, **f64)
            zero = torch.zeros(1, **f64); one = torch.ones(1, **f64)
            active = torch.ones(1, dtype=torch.bool, device=dev)
            iters = torch.zeros(1, dtype=torch.int64, device=dev)
            L.check(lib, lib.hipgp_vec_dot(dt, ptr(r), ptr(z), ptr(rs), 1, M, st()))
            red(rs)
            for n in range(maxiter):
                Ap = A(p)
                L.check(lib, lib.hipgp_vec_dot(dt, ptr(p), ptr(Ap), ptr(pAp), 1, M, st()))
                red(pAp)
                num = torch.where(active, rs, zero); den = torch.where(active, pAp, one)      # alpha = 0 once stopped
                L.check(lib, lib.hipgp_vec_xr_update(dt, ptr(x), ptr(r), ptr(p), ptr(Ap), ptr(num), ptr(den), ptr(sc), 1, M, st()))
                z = Pm(r) if Pm is not None else r
                L.check(lib, lib.hipgp_vec_dot(dt, ptr(z), ptr(r), C.c_void_p(sc.data_ptr() + 8), 1, M, st()))
                red(sc)
                iters += active
                active = active & (torch.sqrt(sc[0:1]) >= tol)
                num = torch.where(active, sc[1:2], zero); den = torch.where(active, rs, one)
                L.check(lib, lib.hipgp_vec_p_update(dt, ptr(p), ptr(z), ptr(num), ptr(den), 1, M, st()))
                rs = sc[1:2].clone()
                if (n + 1) % check_every == 0 and n + 1 < maxiter and not bool(active):
                    break
            self._iters_dev = iters
        return x

    @property
    def last_iters(self):
        return int(self._iters_dev.item())
