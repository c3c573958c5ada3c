"""Drop-in for `ziggy/kernels.py` (and the hot functions of `ziggy/exact_gp_1d_derivatives.py:9-38`).

Same class names, constructor arguments, method names and argument meaning as the reference; the arithmetic
runs in libhipgp_b200.so (hand-written CUDA).  Two call shapes exist:

  * generic      `kernel(x, y, params)` with arbitrary point sets -> hipgp_kernel_pairwise
  * grid-aware   `kernel.forward_grid(x, xgrids, params)` etc.    -> hipgp_kxu, which derives the inducing point of
                 every column from the 1-D grids instead of reading an (M, D) meshgrid; used by our `_make_grams`.

Out of the hot path, kept on the host exactly as in the reference: the 50-entry doubly-integrated-diagonal table is
built once by scipy `dblquad` (kernels.py:183-197,266-287) -- it is an INPUT of the CUDA interpolation kernel.
"""
import ctypes as C

import numpy as np
import torch
from torch import nn

from . import _lib as L

_DT = {torch.float32: L.F32, torch.float64: L.F64}


def _stream(device):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def _ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else None


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("hipgp_b200.kernels: inputs must be CUDA tensors (no CPU fallback)")


def _ell_array(ell, ndim):
    """ell is a python/torch scalar or a (D,) tensor (kernels.py:9)."""
    if isinstance(ell, torch.Tensor):
        vals = ell.detach().double().reshape(-1).cpu().tolist()
    elif isinstance(ell, (list, tuple, np.ndarray)):
        vals = [float(v) for v in np.asarray(ell, dtype=np.float64).reshape(-1)]
    else:
        vals = [float(ell)]
    if len(vals) not in (1, ndim):
        raise ValueError("ell must be a scalar or have one entry per input dimension")
    return (C.c_double * len(vals))(*vals), len(vals)


def _f(v):
    return float(v.detach()) if isinstance(v, torch.Tensor) else float(v)


def _wants_grad(*vals):
    return torch.is_grad_enabled() and any(isinstance(v, torch.Tensor) and v.requires_grad for v in vals)


class _KxuParamGrad(torch.autograd.Function):
    """K_xu (or a pairwise kernel matrix) as a differentiable function of (sig2, ell): the forward is the same CUDA call
    as the no-grad path, the backward reduces G * dk/d(sig2, ell_d) on the fly (hipgp_kxu_param_grad) -- the (B, M)
    derivative matrices are never formed.  learn_kernel=True in the reference differentiates kernels.py:73-79,145-158
    with autograd."""

    @staticmethod
    def forward(ctx, sig2_t, ell_t, call, meta):
        ctx.meta = meta
        ctx.ell_numel = ell_t.numel()
        ctx.sig2_dtype, ctx.ell_dtype, ctx.ell_shape = sig2_t.dtype, ell_t.dtype, ell_t.shape
        return call((sig2_t.detach(), ell_t.detach()))

    @staticmethod
    def backward(ctx, G):
        m = ctx.meta
        lib = L.load()
        G = G.to(m["dtype"]).contiguous()
        B, Mcols = G.shape
        nbx = (Mcols + 1023) // 1024
        partial = torch.empty((B, nbx, 4), dtype=torch.float64, device=G.device)
        with torch.cuda.device(G.device):
            L.check(lib, lib.hipgp_kxu_param_grad(_DT[m["dtype"]], m["kernel_id"], m["mode"], m["sig2"], m["ellv"], m["n_ell"], _ptr(m["x"]), B,
                                                  m["D"], m["marr"], _ptr(m["grids"]), _ptr(m["ypts"]), Mcols, _ptr(m["mc_alphas"]), m["npts"],
                                                  _ptr(G), C.cast(C.c_void_p(partial.data_ptr()), L._pd), _stream(G.device)))
        tot = partial.sum(dim=(0, 1))
        g_sig2 = tot[0].to(ctx.sig2_dtype).reshape(()) if ctx.needs_input_grad[0] else None
        g_ell = None
        if ctx.needs_input_grad[1]:
            g_ell = (tot[1:4].sum() if ctx.ell_numel == 1 else tot[1:1 + ctx.ell_numel]).to(ctx.ell_dtype).reshape(ctx.ell_shape)
        return g_sig2, g_ell, None, None


def _with_param_grad(call, params, meta):
    """run `call(params)`; route it through _KxuParamGrad when a hyper-parameter tensor requires a gradient"""
    sig2, ell = params
    if not _wants_grad(sig2, ell):
        return call(params)
    if meta["kernel_id"] == L.K_GNEITING or meta["mode"] not in (L.KXU_POINT, L.KXU_SEMI_ANALYTIC, L.KXU_SEMI_MC):
        raise NotImplementedError("hipgp_b200: hyper-parameter gradients (learn_kernel=True) are built for the SqExp / Matern point "
                                  "kernels, their Monte-Carlo line integrals and the analytic SqExp line integral; not for this "
                                  "kernel / estimator")
    dev = meta["x"].device
    s_t = sig2 if isinstance(sig2, torch.Tensor) else torch.tensor(float(sig2), dtype=torch.float64, device=dev)
    e_t = ell if isinstance(ell, torch.Tensor) else torch.tensor(np.asarray(ell, dtype=np.float64), device=dev)
    meta["sig2"] = _f(sig2)
    return _KxuParamGrad.apply(s_t, e_t, call, meta)


def _pairwise(kernel_id, mode, x, y, params, dtype, alpha=1.0, mc_alphas=None):
    """out (n, m) = k(x_i, y_j);   x: (n, D), y: (m, D)"""
    _need_cuda(x, y, mc_alphas)
    assert x.shape[-1] == y.shape[-1], \
        "last dimension should match, but got x.shape = {}, y.shape = {}".format(x.shape, y.shape)
    assert x.ndimension() == 2 and y.ndimension() == 2, "x shape = {}, y shape = {}".format(x.shape, y.shape)
    sig2, ell = params
    lib = L.load()
    x = x.detach().to(dtype).contiguous(); y = y.detach().to(dtype).contiguous()
    n, D = x.shape
    m = y.shape[0]
    ellv, n_ell = _ell_array(ell, D)
    npts = 0
    if mc_alphas is not None:
        mc_alphas = mc_alphas.detach().to(dtype).contiguous(); npts = mc_alphas.numel()

    def call(p):
        out = torch.empty((n, m), dtype=dtype, device=x.device)
        with torch.cuda.device(x.device):
            L.check(lib, lib.hipgp_kernel_pairwise(_DT[dtype], kernel_id, mode, _f(p[0]), ellv, n_ell, float(alpha), _ptr(x), n,
                                                   _ptr(y), m, D, _ptr(mc_alphas), npts, _ptr(out), _stream(x.device)))
        return out
    meta = dict(kernel_id=kernel_id, mode=mode, dtype=dtype, ellv=ellv, n_ell=n_ell, x=x, D=D, marr=None, grids=None, ypts=y,
                mc_alphas=mc_alphas, npts=npts)
    return _with_param_grad(call, params, meta)


def _on_grid(kernel_id, mode, x, xgrids, params, dtype, alpha=1.0, mc_alphas=None):
    """out (n, M) = k(x_i, u_j) with u the C-order meshgrid of xgrids (never materialised)."""
    _need_cuda(x, mc_alphas, *xgrids)
    sig2, ell = params
    lib = L.load()
    x = x.detach().to(dtype).contiguous()
    if x.dim() == 1:
        x = x[:, None]
    n, D = x.shape
    assert D == len(xgrids), "x has %d columns but there are %d grids" % (D, len(xgrids))
    dims = [int(len(g)) for g in xgrids]
    grids = torch.cat([g.detach().to(dtype).reshape(-1) for g in xgrids]).contiguous()
    ellv, n_ell = _ell_array(ell, D)
    M = int(np.prod(dims))
    npts = 0
    if mc_alphas is not None:
        mc_alphas = mc_alphas.detach().to(dtype).contiguous(); npts = mc_alphas.numel()
    marr = (C.c_int64 * D)(*dims)

    def call(p):
        out = torch.empty((n, M), dtype=dtype, device=x.device)
        with torch.cuda.device(x.device):
            L.check(lib, lib.hipgp_kxu(_DT[dtype], kernel_id, mode, _f(p[0]), ellv, n_ell, float(alpha), _ptr(x), n, D, marr,
                                       _ptr(grids), _ptr(mc_alphas), npts, _ptr(out), _stream(x.device)))
        return out
    meta = dict(kernel_id=kernel_id, mode=mode, dtype=dtype, ellv=ellv, n_ell=n_ell, x=x, D=D, marr=marr, grids=grids, ypts=None,
                mc_alphas=mc_alphas, npts=npts)
    return _with_param_grad(call, params, meta)


def mc_alphas(npts, dtype, device):
    """Stratified offsets of `Kernel.k_semi_mc` (kernels.py:24-27): one torch.rand(1) from the global generator of
    `device`, so RNG streams stay identical to the reference's."""
    delta = 1. / npts
    return torch.arange(npts, dtype=dtype, device=device) / npts + torch.rand(1, dtype=dtype, device=device) * delta


class Kernel(nn.Module):
    """base kernel class (kernels.py:11-61)"""
    kernel_id = None
    gneiting_alpha = 1.0

    def __init__(self):
        super(Kernel, self).__init__()
        self._diag_interp = None
        self._Ndiag, self._dmax = 50, 5

    # -- generic point sets ---------------------------------------------------------------------
    def forward(self, x, y, params):
        return _pairwise(self.kernel_id, L.KXU_POINT, x, y, params, self.dtype, self.gneiting_alpha)

    def k_semi(self, xpoint, xintegrated, params):
        raise NotImplementedError

    def k_semi_mc(self, xpoint, xintegrated, params, npts=5, alphas=None):
        """monte carlo approximation of the semi integrated kernel -> (Npoint, Nintegrated) (kernels.py:19-39)"""
        if alphas is None:
            alphas = mc_alphas(npts, self.dtype, xpoint.device)
        return _pairwise(self.kernel_id, L.KXU_SEMI_MC, xintegrated, xpoint, params, self.dtype, self.gneiting_alpha,
                         alphas).transpose(0, 1)

    # -- inducing grid given by its 1-D axes (the SVI hot path) -------------------------------
    def forward_grid(self, x, xgrids, params):
        return _on_grid(self.kernel_id, L.KXU_POINT, x, xgrids, params, self.dtype, self.gneiting_alpha)

    def k_semi_mc_grid(self, xgrids, xintegrated, params, npts=5, alphas=None):
        """(Nintegrated, M) -- already transposed the way `_make_grams` wants it (svi_gp.py:62-64)"""
        if alphas is None:
            alphas = mc_alphas(npts, self.dtype, xintegrated.device)
        return _on_grid(self.kernel_id, L.KXU_SEMI_MC, xintegrated, xgrids, params, self.dtype, self.gneiting_alpha, alphas)

    # -- doubly integrated diagonal -----------------------------------------------------------
    @property
    def diag_interp(self):
        if self._diag_interp is None:
            self._diag_interp = KernelDoublyDiagInterpolator(self, N=self._Ndiag, dmax=self._dmax)
        return self._diag_interp

    def k_doubly_diag(self, x, params):
        return self.diag_interp(x, params)

    def _host_eval(self, r):
        """k at distance r for (sig2, ell) = (1, 1) on the host, for the ctor-time quadrature only."""
        raise NotImplementedError


class SqExp(Kernel):
    """squared exponential kernel (kernels.py:64-93)"""
    kernel_id = L.K_SQEXP

    def __init__(self, dtype=torch.double, Ndiag=50, dmax=5):
        super(SqExp, self).__init__()
        self.dtype = dtype
        self._Ndiag, self._dmax = Ndiag, dmax
        self.has_k_semi = True

    def diag(self, x, params):
        sig2, ell = params
        return sig2 * torch.ones(x.shape[0], dtype=self.dtype, device=x.device)

    def k_semi(self, xpoint, xintegrated, params):
        """analytic line integral from the origin -> (Npoint, Nintegrated) (kernels.py:85-90,223-237)"""
        return _pairwise(self.kernel_id, L.KXU_SEMI_ANALYTIC, xintegrated, xpoint, params, self.dtype).transpose(0, 1)

    def k_semi_grid(self, xgrids, xintegrated, params):
        """(Nintegrated, M)"""
        return _on_grid(self.kernel_id, L.KXU_SEMI_ANALYTIC, xintegrated, xgrids, params, self.dtype)

    def _host_eval(self, r):
        return np.exp(-0.5 * r * r)


class Gneiting(Kernel):
    """kernels.py:96-128"""
    kernel_id = L.K_GNEITING

    def __init__(self, alpha=1., length_scale=1., dtype=torch.double, Ndiag=50, dmax=5.):
        super(Gneiting, self).__init__()
        self.dtype = dtype
        self.alpha = alpha
        self.gneiting_alpha = alpha
        self.length_scale = length_scale
        self.anisotropic = False
        self._Ndiag, self._dmax = Ndiag, dmax
        self.has_k_semi = False

    def diag(self, x, params):
        sig2, ell = params
        return sig2 * torch.ones(x.shape[0], dtype=self.dtype, device=x.device)

    def _host_eval(self, r):
        t = r
        c = (1 - t) * np.cos(np.pi * t) + (1 / np.pi) * np.sin(np.pi * t)
        return np.where(t > 1., 0., (1 + t ** self.alpha) ** (-3) * c)


class Matern(Kernel):
    """kernels.py:131-165"""

    def __init__(self, nu=0.5, length_scale=1., dtype=torch.double, Ndiag=50, dmax=5.):
        super(Matern, self).__init__()
        if nu not in {0.5, 1.5, 2.5}:
            raise RuntimeError("nu expected to be 0.5, 1.5, or 2.5")
        self.nu = nu
        self.kernel_id = {0.5: L.K_MATERN12, 1.5: L.K_MATERN32, 2.5: L.K_MATERN52}[nu]
        self.dtype = dtype
        self.length_scale = length_scale
        self.anisotropic = False
        self._Ndiag, self._dmax = Ndiag, dmax
        self.has_k_semi = False

    def diag(self, x, params):
        sig2, ell = params
        return sig2 * x.new_ones(x.shape[0])

    def _host_eval(self, r):
        if self.nu == .5:
            return np.exp(-r)
        if self.nu == 1.5:
            dp = np.sqrt(3) * r
            return (1 + dp) * np.exp(-dp)
        dp = np.sqrt(5) * r
        return (1 + dp + (5. / 3.) * r * r) * np.exp(-dp)


def doubly_integrated_diag(x, kern_r, return_errors=False):
    """|x|^2 int_0^1 int_0^1 k(|a - a'| |x|) da da'  -- the prior variance of a line integral from the origin to x
    (what kernels.py:266-287 evaluates with a 2-D adaptive quadrature).  For a stationary kernel the integrand depends on
    t = |a - a'| only and the square [0,1]^2 holds a strip of length 2 (1 - t) at offset t, so the double integral equals
    2 int_0^1 (1 - t) k(t |x|) dt: ONE 1-D adaptive quadrature per point, to a tighter tolerance than the reference's
    (whose table it reproduces to that table's own accuracy, 1.49e-5 relative)."""
    from scipy import integrate
    dist = np.sqrt(np.sum(np.asarray(x, dtype=np.float64) ** 2, axis=1))
    knn = np.zeros(len(dist)); errs = np.zeros(len(dist))
    for n, d in enumerate(dist):
        val, err = integrate.quad(lambda t: (1.0 - t) * float(kern_r(t * d)), 0.0, 1.0, epsrel=1e-10, epsabs=0.0, limit=200)
        knn[n] = 2.0 * val * d * d
        errs[n] = 2.0 * err * d * d
    if return_errors:
        return knn, errs
    return knn


class KernelDoublyDiagInterpolator(nn.Module):
    """linear interpolation of the doubly integrated diagonal (kernels.py:168-218).  The table may be passed in
    (`table=(distance_grid, slopes, knn)`), e.g. read from a reference object; otherwise it is built on the host."""

    def __init__(self, kernel, N=50, dmax=5, dtype=None, table=None):
        super(KernelDoublyDiagInterpolator, self).__init__()
        if dtype is None:
            dtype = kernel.dtype
        self.dtype = dtype
        if table is None:
            dgrid = np.linspace(0, dmax, N)
            xs = np.column_stack([dgrid, np.zeros(N)])
            knn = doubly_integrated_diag(xs, kernel._host_eval)
            slopes = (knn[1:] - knn[:-1]) / (dgrid[1:] - dgrid[:-1])
            slopes = np.concatenate([slopes, [slopes[-1]]])
            table = (dgrid, slopes, knn)
        self.distance_grid = torch.as_tensor(np.asarray(table[0], dtype=np.float32)).to(dtype)
        self.slopes = torch.as_tensor(np.asarray(table[1], dtype=np.float32)).to(dtype)
        self.knn = torch.as_tensor(np.asarray(table[2], dtype=np.float32)).to(dtype)

    def forward(self, x, params):
        _need_cuda(x)
        sig2, ell = params
        lib = L.load()
        x = x.detach().to(self.dtype).contiguous()
        n, D = x.shape
        dg = self.distance_grid.to(x.device).contiguous()
        sl = self.slopes.to(x.device).contiguous()
        kn = self.knn.to(x.device).contiguous()
        ellv, n_ell = _ell_array(ell, D)
        dt = _DT[self.dtype]

        def call():
            out = torch.empty(n, dtype=self.dtype, device=x.device)
            with torch.cuda.device(x.device):
                L.check(lib, lib.hipgp_doubly_diag(dt, _ptr(x), n, D, _f(sig2), ellv, n_ell, _ptr(dg), _ptr(sl), _ptr(kn), dg.numel(),
                                                   _ptr(out), _stream(x.device)))
            return out
        if not _wants_grad(sig2, ell):
            return call()
        if n_ell != 1:
            raise NotImplementedError("hipgp_b200: hyper-parameter gradients of the doubly integrated diagonal need a scalar ell "
                                      "(the prefactor ell^2 is not defined for a per-axis ell)")

        def grad_call(g):
            g = g.to(self.dtype).contiguous()
            partial = torch.empty(((n + 255) // 256, 2), dtype=torch.float64, device=x.device)
            with torch.cuda.device(x.device):
                L.check(lib, lib.hipgp_doubly_diag_param_grad(dt, _ptr(x), n, D, _f(sig2), ellv, n_ell, _ptr(dg), _ptr(sl), _ptr(kn),
                                                              dg.numel(), _ptr(g), _ptr(partial), _stream(x.device)))
            return partial.sum(dim=0)
        s_t = sig2 if isinstance(sig2, torch.Tensor) else torch.tensor(float(sig2), dtype=torch.float64, device=x.device)
        e_t = ell if isinstance(ell, torch.Tensor) else torch.tensor(float(ell), dtype=torch.float64, device=x.device)
        return _DoublyDiagParamGrad.apply(s_t, e_t, call, grad_call)


class _DoublyDiagParamGrad(torch.autograd.Function):
    """The doubly integrated diagonal as a differentiable function of (sig2, ell) for a scalar ell: the forward is the
    hipgp_doubly_diag call of the no-grad path, the backward reduces g * d/d(sig2, ell) in hipgp_doubly_diag_param_grad.
    learn_kernel=True in the reference differentiates kernels.py:199-218 with autograd."""

    @staticmethod
    def forward(ctx, sig2_t, ell_t, call, grad_call):
        ctx.grad_call = grad_call
        ctx.sig2_dtype, ctx.ell_dtype, ctx.ell_shape = sig2_t.dtype, ell_t.dtype, ell_t.shape
        return call()

    @staticmethod
    def backward(ctx, g):
        tot = ctx.grad_call(g)
        g_sig2 = tot[0].to(ctx.sig2_dtype).reshape(()) if ctx.needs_input_grad[0] else None
        g_ell = tot[1].to(ctx.ell_dtype).reshape(ctx.ell_shape) if ctx.needs_input_grad[1] else None
        return g_sig2, g_ell, None, None


# --------------------------------------------------------------------------------------------------
# 1-D derivative inter-domain kernels (exact_gp_1d_derivatives.py:9-38)
def _deriv(mode, x, y, sig2, ell):
    dtype = x.dtype if x.dtype in _DT else torch.float64
    return _pairwise(L.K_SQEXP, mode, x.reshape(-1, 1), y.reshape(-1, 1), (sig2, ell), dtype)


def k(x, y, sig2, ell):
    return _deriv(L.KXU_POINT, x, y, sig2, ell)


def k_1d(x, sig2, ell):
    return sig2


def kprime(x, y, sig2, ell):
    return _deriv(L.KXU_DERIV, x, y, sig2, ell)


def kprime_double_1d(x, sig2, ell):
    return sig2 / (ell ** 2)


def kprime_double_full(x, y, sig2, ell):
    return _deriv(L.KXU_DERIV2, x, y, sig2, ell)


# --------------------------------------------------------------------------------------------------
def first_row(xgrids, kernel, params, jitter=None):
    """k(u_0, u_.) on the grid (toeplitz_tensor.py:127-133) without building the meshgrid."""
    x0 = torch.stack([g[0] for g in xgrids]).reshape(1, -1)
    row = kernel.forward_grid(x0, xgrids, params).reshape(-1)
    if jitter is not None:
        row = torch.cat([row[:1] + jitter, row[1:]])        # (out of place: the row may carry the hyper-parameter graph)
    return row
