"""`Plan`: torch-tensor front end of the C-ABI plan object (include/hipgp_b200.h).

PyTorch is used for device memory and streams only; all arithmetic happens inside libhipgp_b200.so.
Tensors must live on a CUDA device -- there is no CPU path.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L

_DT = {torch.float32: L.F32, torch.float64: L.F64}


def _stream_ptr(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _require_cuda(t, what):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise RuntimeError("hipgp_b200: %s must be a CUDA tensor (the structured path has no CPU fallback)" % what)


class Plan:
    """One structured K_uu on a D-dimensional inducing grid (replaces the state of the reference's
    ToeplitzTensor / ToeplitzMatmul, ziggy/misc/toeplitz_tensor.py:9-45)."""

    def __init__(self, dims, dtype, device):
        self.lib = L.load()
        device = torch.device(device)
        if device.type != "cuda":
            raise RuntimeError("hipgp_b200: plans live on CUDA devices only (got %s); there is no CPU fallback" % device)
        if dtype not in _DT:
            raise TypeError("dtype must be torch.float32 or torch.float64")
        self.device = device if device.index is not None else torch.device("cuda", torch.cuda.current_device())
        self.dtype = dtype
        self.dims = tuple(int(d) for d in dims)
        m = (C.c_int64 * len(self.dims))(*self.dims)
        h = C.c_void_p()
        L.check(self.lib, self.lib.hipgp_plan_create(len(self.dims), m, _DT[dtype], self.device.index, C.byref(h)))
        self._h = h
        M, E = C.c_int64(), C.c_int64()
        L.check(self.lib, self.lib.hipgp_plan_sizes(h, C.byref(M), C.byref(E)))
        self.M, self.Mprime = M.value, E.value
        self.embedded_dims = tuple(2 * d - 2 if d > 1 else 1 for d in self.dims)
        self.num_clamped = None

    def __del__(self):
        h = getattr(self, "_h", None)
        if h is not None and h.value:
            try:
                self.lib.hipgp_plan_destroy(h)
            except Exception:
                pass
            self._h = None

    # ------------------------------------------------------------------
    def _vec(self, t, ncols, what):
        _require_cuda(t, what)
        if t.dim() != 2 or t.shape[1] != ncols:
            raise ValueError("%s must have shape (bsz, %d), got %s" % (what, ncols, tuple(t.shape)))
        if t.device != self.device:
            raise RuntimeError("%s is on %s but the plan is on %s" % (what, t.device, self.device))
        return t.to(self.dtype).contiguous()

    def embedding(self):
        n = len(self.dims)
        a, b = (C.c_int64 * n)(), (C.c_int64 * n)()
        L.check(self.lib, self.lib.hipgp_plan_embedding(self._h, a, b))
        return tuple(a), tuple(b)

    def set_first_row(self, column, clamp=1e-6):
        _require_cuda(column, "column")
        col = column.detach().reshape(-1).to(self.dtype).contiguous()
        if col.numel() != self.M:
            raise ValueError("column must have %d entries" % self.M)
        n = C.c_int64()
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_plan_set_first_row(self._h, C.c_void_p(col.data_ptr()), float(clamp),
                                                                 C.byref(n), _stream_ptr(self.device)))
        self.num_clamped = n.value
        return self

    def spectrum(self, which=L.SPEC_D):
        out = torch.empty(self.embedded_dims, dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_plan_spectrum(self._h, which, C.c_void_p(out.data_ptr()), _stream_ptr(self.device)))
        return out

    def matvec(self, mode, vec):
        nin = self.Mprime if mode == L.MV_R else self.M
        nout = self.Mprime if mode == L.MV_RT else self.M
        v = self._vec(vec, nin, "vec")
        out = torch.empty((v.shape[0], nout), dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_matvec(self._h, mode, C.c_void_p(v.data_ptr()), C.c_void_p(out.data_ptr()),
                                                     v.shape[0], _stream_ptr(self.device)))
        return out

    def pcg(self, b, maxiter=20, tol=1e-10, precond=True, callback=None, return_info=False):
        """Fused device-resident PCG (replaces conj_grad/conj_grad2, ziggy/misc/cg.py).  `callback(n, x)` fires
        after every iteration that did not satisfy the stopping test, as in the reference (cg.py:70-78)."""
        v = self._vec(b, self.M, "b")
        x = torch.empty_like(v)
        iters, ncb = C.c_int(), C.c_int()
        resid = (C.c_double * v.shape[0])()
        if callback is not None:
            def _cb(n, xptr, user):
                callback(n, x.clone())
            cfn = L.ITER_CB(_cb)
        else:
            cfn = L.ITER_CB(0)
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_pcg(self._h, C.c_void_p(v.data_ptr()), C.c_void_p(x.data_ptr()), v.shape[0],
                                                  int(maxiter), float(tol), 1 if precond else 0, C.byref(iters), C.byref(ncb),
                                                  resid, cfn, None, _stream_ptr(self.device)))
        if return_info:
            return x, {"iters": iters.value, "callbacks": ncb.value, "resid": np.array(resid[:])}
        return x

    def compute_kn(self, Knm, maxiter=10, tol=1e-8):
        """k_n = R^T K_uu^-1 K_un  (ziggy/hipgp.py:139-146)"""
        v = self._vec(Knm, self.M, "Knm")
        out = torch.empty((v.shape[0], self.Mprime), dtype=self.dtype, device=self.device)
        iters = C.c_int()
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_compute_kn(self._h, C.c_void_p(v.data_ptr()), C.c_void_p(out.data_ptr()),
                                                         v.shape[0], int(maxiter), float(tol), C.byref(iters),
                                                         _stream_ptr(self.device)))
        return out

    def rt_column_grad(self, vec, grad_out, scale=1.0):
        """d/d column of sum_b grad_out_b . (R^T vec_b)  (autograd through toeplitz_tensor.py:21-33,85-97 in the reference).
        vec (B, M), grad_out (B, M').  Returns (M,)."""
        v = self._vec(vec, self.M, "vec"); g = self._vec(grad_out, self.Mprime, "grad_out")
        if v.shape[0] != g.shape[0]:
            raise ValueError("vec and grad_out must have the same number of rows")
        out = torch.empty(self.M, dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_rt_column_grad(self._h, C.c_void_p(v.data_ptr()), C.c_void_p(g.data_ptr()), v.shape[0],
                                                             float(scale), C.c_void_p(out.data_ptr()), _stream_ptr(self.device)))
        return out

    def toeplitz_quadform(self, left, right, scale=1.0):
        """sum_j u_j^T (dT/dc_i) v_j over the FLATTENED M-vectors (gpt_toeplitz.py:169-209
        `sym_toeplitz_derivative_quadratic_form`); left / right are (S, M).  Returns (M,)."""
        u = self._vec(left, self.M, "left")
        v = self._vec(right, self.M, "right")
        if u.shape != v.shape:
            raise ValueError("left and right must have the same shape")
        out = torch.empty(self.M, dtype=self.dtype, device=self.device)
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_toeplitz_quadform(self._h, C.c_void_p(u.data_ptr()), C.c_void_p(v.data_ptr()),
                                                                u.shape[0], float(scale), C.c_void_p(out.data_ptr()),
                                                                _stream_ptr(self.device)))
        return out

    # host-buffer entry points (H2D / D2H inside the call) -- used for the end-to-end benchmark figure
    def matvec_host(self, mode, vec_host, out_host):
        assert not vec_host.is_cuda and not out_host.is_cuda and vec_host.is_contiguous() and out_host.is_contiguous()
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_matvec_host(self._h, mode, C.c_void_p(vec_host.data_ptr()),
                                                          C.c_void_p(out_host.data_ptr()), vec_host.shape[0],
                                                          _stream_ptr(self.device)))
        return out_host

    def pcg_host(self, b_host, x_host, maxiter=20, tol=1e-10, precond=True, group=None):
        """Host buffers in / out (H2D + solve + D2H).  `group`: process the right-hand sides in independent groups of that
        many and hide the copies of neighbouring groups behind the solve (hipgp_pcg_host_pipelined)."""
        assert not b_host.is_cuda and not x_host.is_cuda and b_host.is_contiguous() and x_host.is_contiguous()
        iters, ncb = C.c_int(), C.c_int()
        if group:
            with torch.cuda.device(self.device):
                L.check(self.lib, self.lib.hipgp_pcg_host_pipelined(self._h, C.c_void_p(b_host.data_ptr()), C.c_void_p(x_host.data_ptr()),
                                                                     b_host.shape[0], int(maxiter), float(tol), 1 if precond else 0,
                                                                     int(group), C.byref(iters), _stream_ptr(self.device)))
            return x_host, iters.value
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_pcg_host(self._h, C.c_void_p(b_host.data_ptr()), C.c_void_p(x_host.data_ptr()),
                                                       b_host.shape[0], int(maxiter), float(tol), 1 if precond else 0,
                                                       C.byref(iters), C.byref(ncb), None, _stream_ptr(self.device)))
        return x_host, iters.value

    def pcg_host_submit(self, b_host, x_host, slot, maxiter=20, tol=1e-10, precond=True):
        """Queue one host-buffer solve on `slot` (0 or 1) and return at once (hipgp_pcg_host_submit): with two slots in flight the
        copies of neighbouring batches hide under the current solve.  Both buffers must be pinned and stay untouched until
        `pcg_host_wait(slot)`."""
        assert not b_host.is_cuda and not x_host.is_cuda and b_host.is_contiguous() and x_host.is_contiguous()
        assert b_host.is_pinned() and x_host.is_pinned(), "asynchronous host solves need pinned buffers"
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_pcg_host_submit(self._h, C.c_void_p(b_host.data_ptr()), C.c_void_p(x_host.data_ptr()),
                                                              b_host.shape[0], int(maxiter), float(tol), 1 if precond else 0, int(slot),
                                                              _stream_ptr(self.device)))

    def pcg_host_wait(self, slot):
        """Block until the solve submitted on `slot` has delivered x_host; returns its iteration count."""
        iters = C.c_int()
        L.check(self.lib, self.lib.hipgp_pcg_host_wait(self._h, int(slot), C.byref(iters)))
        return iters.value

    def device_bytes(self):
        n = C.c_size_t()
        L.check(self.lib, self.lib.hipgp_plan_device_bytes(self._h, C.byref(n)))
        return n.value

    def launch_count(self):
        n = C.c_int64()
        L.check(self.lib, self.lib.hipgp_plan_launch_count(self._h, C.byref(n)))
        return n.value

    def profile(self, enable):
        L.check(self.lib, self.lib.hipgp_plan_profile(self._h, 1 if enable else 0))

    def profile_read(self, reset=True):
        """{class: (total_ms, launches)} for rows_fwd / cols_pass / rows_inv / vec kernels."""
        out = {}
        names = ("rows_fwd", "cols_pass", "rows_inv", "vec")
        for i, nm in enumerate(names):
            ms, n = C.c_double(), C.c_int64()
            L.check(self.lib, self.lib.hipgp_plan_profile_read(self._h, i, C.byref(ms), C.byref(n),
                                                                1 if (reset and i == len(names) - 1) else 0))
            out[nm] = (ms.value, n.value)
        return out

    # ---- PCG split in two for callers that own the stopping rule (multi-GPU sharded minibatches) ----
    def pcg_begin(self, b, tol=-1.0, precond=True):
        v = self._vec(b, self.M, "b")
        x = torch.empty_like(v)
        self._run = (v, x)                      # keep both alive while the solve is in flight
        with torch.cuda.device(self.device):
            L.check(self.lib, self.lib.hipgp_pcg_begin(self._h, C.c_void_p(v.data_ptr()), C.c_void_p(x.data_ptr()), v.shape[0],
                                                        float(tol), 1 if precond else 0, _stream_ptr(self.device)))
        return x

    def pcg_step(self, niter=1, poll=True):
        """`niter` more iterations; returns (done, iters, max_b sqrt(r.r)) of this rank when `poll`."""
        done, iters, mx = C.c_int(), C.c_int(), C.c_double()
        with torch.cuda.device(self.device):
            if poll:
                L.check(self.lib, self.lib.hipgp_pcg_step(self._h, int(niter), C.byref(done), C.byref(iters), C.byref(mx),
                                                           _stream_ptr(self.device)))
                return bool(done.value), iters.value, mx.value
            L.check(self.lib, self.lib.hipgp_pcg_step(self._h, int(niter), None, None, None, _stream_ptr(self.device)))
        return None


def meanfield_rowstats(kn, qm, qS):
    """(kn.qm, kn.kn, kn^2.qS) per row of kn (B, M'): hipgp.py:395-397,524.  Returns a (3, B) tensor."""
    _require_cuda(kn, "kn")
    lib = L.load()
    kn = kn.contiguous(); qm = qm.reshape(-1).to(kn.dtype).contiguous(); qS = qS.reshape(-1).to(kn.dtype).contiguous()
    B, E = kn.shape
    out = torch.empty((3, B), dtype=kn.dtype, device=kn.device)
    with torch.cuda.device(kn.device):
        L.check(lib, lib.hipgp_meanfield_rowstats(_DT[kn.dtype], C.c_void_p(kn.data_ptr()), C.c_void_p(qm.data_ptr()),
                                                  C.c_void_p(qS.data_ptr()), B, E, C.c_void_p(out.data_ptr()),
                                                  _stream_ptr(kn.device)))
    return out


def meanfield_colstats(kn, w1, w2):
    """(sum_b w1_b kn[b,:], sum_b w2_b kn[b,:]^2): hipgp.py:241-250.  Returns two (M',) tensors."""
    _require_cuda(kn, "kn")
    lib = L.load()
    kn = kn.contiguous(); w1 = w1.reshape(-1).to(kn.dtype).contiguous(); w2 = w2.reshape(-1).to(kn.dtype).contiguous()
    B, E = kn.shape
    dm = torch.empty(E, dtype=kn.dtype, device=kn.device); lam = torch.empty_like(dm)
    with torch.cuda.device(kn.device):
        L.check(lib, lib.hipgp_meanfield_colstats(_DT[kn.dtype], C.c_void_p(kn.data_ptr()), C.c_void_p(w1.data_ptr()),
                                                  C.c_void_p(w2.data_ptr()), B, E, C.c_void_p(dm.data_ptr()),
                                                  C.c_void_p(lam.data_ptr()), _stream_ptr(kn.device)))
    return dm, lam


def _blk_idx(blk_idx, device):
    idx = blk_idx.to(device=device, dtype=torch.int64).contiguous()
    if idx.dim() != 2:
        raise ValueError("block index must be (num_blocks, block_size)")
    return idx


def block_lam(kn, w, blk_idx, scale=1.0, diag=1.0):
    """lam[k] = scale * sum_n w_n kn_blk[n,k] kn_blk[n,k]^T + diag * I  (get_lam, hipgp.py:666-685) without the permuted
    copy of kn or the (B, num_blocks, bs, bs) outer products of hipgp.py:252-255.  Returns (num_blocks, bs, bs)."""
    _require_cuda(kn, "kn")
    lib = L.load()
    kn = kn.contiguous(); w = w.reshape(-1).to(kn.dtype).contiguous()
    idx = _blk_idx(blk_idx, kn.device)
    B, E = kn.shape
    nblk, bs = idx.shape
    out = torch.empty((nblk, bs, bs), dtype=kn.dtype, device=kn.device)
    with torch.cuda.device(kn.device):
        L.check(lib, lib.hipgp_block_lam(_DT[kn.dtype], C.c_void_p(kn.data_ptr()), C.c_void_p(w.data_ptr()),
                                         C.c_void_p(idx.data_ptr()), B, E, nblk, bs, float(scale), float(diag),
                                         C.c_void_p(out.data_ptr()), _stream_ptr(kn.device)))
    return out


def block_diag_multiply(S_block, v, blk_idx):
    """from_blocks(S_block @ to_blocks(v)) for v (B, M')  (hipgp.py:640-652).  Returns (B, M')."""
    _require_cuda(v, "v")
    lib = L.load()
    v = v.contiguous(); S = S_block.to(v.dtype).contiguous()
    idx = _blk_idx(blk_idx, v.device)
    B, E = v.shape
    nblk, bs = idx.shape
    if tuple(S.shape) != (nblk, bs, bs):
        raise ValueError("S_block must be (num_blocks, block_size, block_size)")
    out = torch.empty_like(v)
    with torch.cuda.device(v.device):
        L.check(lib, lib.hipgp_block_diag_multiply(_DT[v.dtype], C.c_void_p(S.data_ptr()), C.c_void_p(v.data_ptr()),
                                                   C.c_void_p(idx.data_ptr()), B, E, nblk, bs, C.c_void_p(out.data_ptr()),
                                                   _stream_ptr(v.device)))
    return out


def block_quadform_grad(S_block, kn, g, blk_idx):
    """g[:, None] * from_blocks((S_block + S_block^T) @ to_blocks(kn)): the gradient of knSkn_b = kn_b^T blockdiag(S) kn_b
    with upstream g (B,), in one pass over kn and S.  Returns (B, M')."""
    _require_cuda(kn, "kn")
    lib = L.load()
    kn = kn.contiguous(); S = S_block.to(kn.dtype).contiguous(); g = g.reshape(-1).to(kn.dtype).contiguous()
    idx = _blk_idx(blk_idx, kn.device)
    B, E = kn.shape
    nblk, bs = idx.shape
    if tuple(S.shape) != (nblk, bs, bs):
        raise ValueError("S_block must be (num_blocks, block_size, block_size)")
    if g.numel() != B:
        raise ValueError("g must have one entry per row of kn")
    out = torch.empty_like(kn)
    with torch.cuda.device(kn.device):
        L.check(lib, lib.hipgp_block_quadform_grad(_DT[kn.dtype], C.c_void_p(S.data_ptr()), C.c_void_p(kn.data_ptr()),
                                                   C.c_void_p(g.data_ptr()), C.c_void_p(idx.data_ptr()), B, E, nblk, bs,
                                                   C.c_void_p(out.data_ptr()), _stream_ptr(kn.device)))
    return out


def row_dot(a, b):
    """per-row dot products of two (B, M) tensors, deterministic fixed-order reduction (hipgp_vec_dot).  Returns (B,)."""
    _require_cuda(a, "a")
    lib = L.load()
    a = a.contiguous(); b = b.to(a.dtype).contiguous()
    B, M = a.shape
    out = torch.empty(B, dtype=torch.float64, device=a.device)
    with torch.cuda.device(a.device):
        L.check(lib, lib.hipgp_vec_dot(_DT[a.dtype], C.c_void_p(a.data_ptr()), C.c_void_p(b.data_ptr()),
                                       C.c_void_p(out.data_ptr()), B, M, _stream_ptr(a.device)))
    return out.to(a.dtype)


class _ToeplitzMatvec(torch.autograd.Function):
    """The four structured matvecs as differentiable maps, like the torch ops of the reference (toeplitz_tensor.py:70-125).
    In the vector argument they are linear: K and the C^-1 block are symmetric, R^T and R are each other's transpose.
    In the Toeplitz column (kernel hyper-parameters through the spectrum): built for R^T -- the one matvec the model
    differentiates (k_n = R^T K^-1 K_un, hipgp.py:139-146; the solve's column gradient is InvMatmul.backward) -- through
    `hipgp_rt_column_grad`; the other three fail loudly instead of returning a gradient with that term missing."""
    _ADJOINT = {L.MV_K: L.MV_K, L.MV_CINV: L.MV_CINV, L.MV_RT: L.MV_R, L.MV_R: L.MV_RT}

    @staticmethod
    def forward(ctx, plan, column, vec, mode):
        ctx.plan, ctx.mode = plan, mode
        ctx.save_for_backward(vec)
        return plan.matvec(mode, vec)

    @staticmethod
    def backward(ctx, grad_output):
        (vec,) = ctx.saved_tensors
        g = grad_output.contiguous()
        gc = None
        if ctx.needs_input_grad[1]:
            if ctx.mode != L.MV_RT:
                raise NotImplementedError("hipgp_b200: gradient of this structured matvec with respect to the Toeplitz column "
                                          "(toeplitz_tensor.py:70-125) is not built; R^T (hipgp_rt_column_grad) and the solve "
                                          "(InvMatmul.backward) are")
            gc = ctx.plan.rt_column_grad(vec.detach(), g)
        gv = ctx.plan.matvec(_ToeplitzMatvec._ADJOINT[ctx.mode], g) if ctx.needs_input_grad[2] else None
        return None, gc, gv, None


def matvec_autograd(plan, mode, vec, column=None):
    """plan.matvec that takes part in autograd when the vector (or the column) requires a gradient"""
    if torch.is_grad_enabled() and (vec.requires_grad or (column is not None and column.requires_grad)):
        return _ToeplitzMatvec.apply(plan, column, vec, mode)
    return plan.matvec(mode, vec)
