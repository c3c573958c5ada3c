"""Host-side mirror of the two callers on the hot path:

  * `ToeplitzInducingGP.compute_kn`  (ziggy/hipgp.py:117-146, ziggy branch)  k_n = R^T K_uu^-1 K_un
  * `SviGP._make_grams`              (ziggy/svi_gp.py:48-76)                  K_xu and the prior diagonal

with the reference's names, arguments and error behaviour, so the unmodified variational families of the reference
(`MeanFieldToeplitzGP` ...) can sit on top of it.  The dense Cholesky branch (hipgp.py:132-137) is the reference's
O(M^3) baseline and is not part of this library.
"""
import numpy as np
import torch
from torch import nn

from .toeplitz_tensor import ToeplitzTensor
from . import kernels as hk
from . import dist as hdist
from .plan import meanfield_rowstats, meanfield_colstats, block_lam, block_diag_multiply, block_quadform_grad, row_dot
from . import util as hutil


class _GridKernelFn:
    """`kfun = lambda x, y: kernel(x, y, params=cov_params)` (hipgp.py:139) that also knows how to produce the first
    row of K_uu straight from the 1-D grids."""

    def __init__(self, kernel, params):
        self.kernel, self.params = kernel, params

    def __call__(self, x, y):
        return self.kernel(x, y, params=self.params)

    def grid_row(self, xgrids):
        return hk.first_row(xgrids, self.kernel, self.params)


class ToeplitzInducingGP(nn.Module):
    def __init__(self, kernel, xgrids, num_obs, sig2_init=1., ell_init=.05, noise2_init=1., learn_kernel=True,
                 learn_noise=True, dtype=torch.float, whitened_type='ziggy', parameterization='expectation-family',
                 jitter_val=1e-3):
        super(ToeplitzInducingGP, self).__init__()
        self.learn_kernel = learn_kernel
        self.learn_noise = learn_noise
        self.jitter_val = jitter_val
        self.ell = torch.tensor(ell_init, dtype=dtype)
        self.log_ell = nn.Parameter(torch.log(torch.tensor(ell_init, dtype=dtype)), requires_grad=self.learn_kernel)
        self.sig2 = torch.tensor(sig2_init, dtype=dtype)
        self.log_sig2 = nn.Parameter(torch.log(torch.tensor(sig2_init, dtype=dtype)), requires_grad=self.learn_kernel)
        self.noise2 = torch.tensor(noise2_init, dtype=dtype)
        self.log_noise2 = nn.Parameter(torch.log(torch.tensor(noise2_init, dtype=dtype)), requires_grad=self.learn_noise)
        self.kernel = kernel
        self.dtype = dtype
        self.N = num_obs
        assert len(xgrids) > 1, len(xgrids)
        self.xgrids = xgrids
        self.M = int(np.prod([len(xg) for xg in xgrids]))
        if whitened_type != 'ziggy':
            raise NotImplementedError("hipgp_b200 implements whitened_type='ziggy' (the structured path) only")
        self.whitened_type = whitened_type
        self.Mprime = int(np.prod([2 * len(xg) - 2 if len(xg) > 1 else len(xg) for xg in self.xgrids]))
        self.parameterization = parameterization
        self._Kmm_cache = None

    @property
    def xinduce(self):
        """(M, D) meshgrid of the inducing points (hipgp.py:63-65) -- built on demand; the hot path never reads it."""
        xxs = torch.meshgrid(*self.xgrids, indexing="ij")
        return torch.stack([x.reshape(-1) for x in xxs], dim=-1)

    def cuda_params(self, cuda_num=0):
        device = torch.device('cuda:{}'.format(cuda_num))
        self.to(device)
        self.kernel = self.kernel.to(device)
        self.xgrids = [x.to(device) for x in self.xgrids]
        return self

    def get_kernel_params(self):
        if not self.learn_kernel:
            return self.sig2, self.ell
        return torch.exp(self.log_sig2), torch.exp(self.log_ell)

    def make_Kmm(self):
        """the structured K_uu for the current kernel parameters; cached while (sig2, ell, jitter) stay unchanged
        (the reference rebuilds it every minibatch, hipgp.py:143)."""
        sig2, ell = self.get_kernel_params()
        if torch.is_grad_enabled() and any(isinstance(p, torch.Tensor) and p.requires_grad for p in (sig2, ell)):
            # learn_kernel=True: the first row has to carry this step's autograd graph (hipgp.py:139-146 rebuilds it every call)
            kfun = _GridKernelFn(self.kernel, (sig2, ell))
            return ToeplitzTensor(xgrids=self.xgrids, kernel=kfun, batch_shape=None, jitter_val=self.jitter_val)
        key = (float(sig2), tuple(np.atleast_1d(ell.detach().cpu().numpy()).tolist()) if isinstance(ell, torch.Tensor)
               else float(ell), float(self.jitter_val), str(self.xgrids[0].device))
        if self._Kmm_cache is None or self._Kmm_cache[0] != key:
            kfun = _GridKernelFn(self.kernel, (sig2, ell))
            Kmm = ToeplitzTensor(xgrids=self.xgrids, kernel=kfun, batch_shape=None, jitter_val=self.jitter_val)
            self._Kmm_cache = (key, Kmm)
        return self._Kmm_cache[1]

    def compute_kn(self, Knm, maxiter_cg=10, tol=1e-8, Kmm=None):
        """kn = R^T Kmm^{-1} Kmn : (bsz, M) -> (bsz, M')  (hipgp.py:117-146)"""
        if Kmm is None:
            Kmm = self.make_Kmm()
        if torch.is_grad_enabled() and (Knm.requires_grad or Kmm.column.requires_grad):
            # differentiable route (learn_kernel=True): InvMatmul (second PCG + Toeplitz-column quadratic form in backward) and the
            # R^T matvec with its column gradient
            d0 = Kmm.inv_matmul(Knm, do_precond=True, maxiter=maxiter_cg, tol=tol)
            return Kmm._matmul_by_RT(d0)
        return Kmm._plan.compute_kn(Knm, maxiter=maxiter_cg, tol=tol)

    @staticmethod
    def batch_slices(n, batch_size):
        """The batches of `batch_predict` (svi_gp.py:81-85): ceil(n / batch_size) slices, the last one ragged."""
        num_batches = int(np.ceil(n / batch_size))
        return [slice((it % num_batches) * batch_size, min(((it % num_batches) + 1) * batch_size, n)) for it in range(num_batches)]

    def batch_predict(self, x, batch_size, verbose=True, **kwargs):
        """Wraps predict(...) into smaller batch predictions (svi_gp.py:78-97).  The batches stream through the device:
        results stay in HBM and come back with ONE device-to-host copy at the end."""
        batches = self.batch_slices(len(x), batch_size)
        mus, sigs = [], []
        for bi, b in enumerate(batches):
            fmu, fsig = self.predict(x[b], _on_device=True, **kwargs)
            mus.append(fmu); sigs.append(fsig)
            if bi % 100 == 0 and verbose:
                print(" ... batch_predict %d / %d batches" % (bi, len(batches)))
        return torch.cat(mus, dim=0).cpu(), torch.cat(sigs, dim=0).cpu()

    def _make_grams(self, xbatch, integrated_obs=False, semi_integrated_estimator="analytic", semi_integrated_samps=10):
        """gram matrices needed for elbo, predict, etc (svi_gp.py:48-76), evaluated on the fly from the grid."""
        kern_params = self.get_kernel_params()
        if integrated_obs:
            if semi_integrated_estimator == "analytic":
                Knm = self.kernel.k_semi_grid(self.xgrids, xbatch, kern_params)
            elif semi_integrated_estimator == "mc-biased":
                Knm = self.kernel.k_semi_mc_grid(self.xgrids, xbatch, kern_params, npts=semi_integrated_samps)
            else:
                raise NotImplementedError
            Knn_diag = self.kernel.k_doubly_diag(xbatch, kern_params)
        else:
            Knm = self.kernel.forward_grid(xbatch, self.xgrids, kern_params)
            Knn_diag = self.kernel.diag(xbatch, kern_params)
        return Knm, Knn_diag


class MeanFieldToeplitzGP(ToeplitzInducingGP):
    """Mean-field variational family (ziggy/hipgp.py:449-524) with the natural-gradient step of
    `elbo_and_grad` (hipgp.py:194-276).  When torch.distributed is initialised the minibatch is sharded over the ranks
    and the statistics are combined with one packed all-reduce, so every rank ends the step with identical gradients."""

    def __init__(self, kernel, xgrids, num_obs, sig2_init=1., ell_init=.05, noise2_init=1., init_Svar=.1, learn_kernel=False,
                 learn_noise=False, dtype=torch.float, whitened_type='ziggy', parameterization='expectation-family',
                 jitter_val=1e-3):
        super(MeanFieldToeplitzGP, self).__init__(kernel, xgrids, num_obs, sig2_init=sig2_init, ell_init=ell_init,
                                                  noise2_init=noise2_init, learn_kernel=learn_kernel, learn_noise=learn_noise,
                                                  dtype=dtype, whitened_type=whitened_type, parameterization=parameterization,
                                                  jitter_val=jitter_val)
        if self.parameterization == 'standard':
            self.global_m = nn.Parameter(torch.nn.init.xavier_normal_(torch.zeros(self.Mprime, 1, dtype=self.dtype)))
            self.global_S = nn.Parameter(init_Svar * torch.ones(self.Mprime, 1, dtype=self.dtype))
        else:
            self.global_theta1 = nn.Parameter(torch.nn.init.xavier_normal_(torch.zeros(self.Mprime, 1, dtype=self.dtype)))
            self.global_theta2 = nn.Parameter((-.5 / init_Svar) * torch.ones(self.Mprime, 1, dtype=self.dtype))

    @property
    def name(self):
        return 'mean-field'

    def standard_variational_params(self):
        if self.parameterization == 'standard':
            return self.global_m, self.global_S
        S = -0.5 * 1 / self.global_theta2
        m = S * self.global_theta1
        return m, S

    def get_kl_to_prior(self, qm=None, qS=None):
        if qm is None or qS is None:
            qm, qS = self.standard_variational_params()
        return .5 * (torch.sum(qS) + torch.sum(qm * qm) - torch.sum(torch.log(qS)) - len(qm))   # stats.py:4-8

    def compute_knSkn(self, kn, qS):
        return meanfield_rowstats(kn, torch.zeros_like(qS), qS)[2]

    def _row_stats(self, kn, qm, qS):
        return meanfield_rowstats(kn, qm, qS)      # knt_m, knt_kn, knSkn

    def _batch_stats(self, kn, bdiff, ivar_noise):
        """sums over the (local) minibatch that the natural gradient needs: sum_n bdiff_n k_n and sum_n w_n k_n^2"""
        return meanfield_colstats(kn, bdiff, ivar_noise)

    def _natural_gradient(self, dm, lam_sum, qm, bscale):
        """hipgp.py:247-250"""
        lam_diag = bscale * lam_sum + 1
        dS = -.5 * lam_diag[:, None] - self.global_theta2.data
        return dm + dS * (-2 * qm), dS

    def elbo_and_grad(self, xbatch, ybatch, noise_std_batch=None, maxiter_cg=10, integrated_obs=False,
                      semi_integrated_estimator="analytic", semi_integrated_samps=10, print_debug_info=False, Kmm=None,
                      shard=True):
        """ELBO estimate and natural gradient for the global parameters (hipgp.py:194-276, mean-field branch).
        xbatch (bsz, D), ybatch (bsz, 1), noise_std_batch None or (bsz, 1): the GLOBAL minibatch on every rank; with
        `shard` and an initialised process group each rank works on its contiguous slice."""
        assert self.parameterization == 'expectation-family', \
            "need parameterization=expectation-family when performing natural gradient descent"
        bsz = xbatch.shape[0]
        sharded = bool(shard and hdist.is_dist())
        sl = hdist.shard_slice(bsz) if sharded else slice(0, bsz)
        xb, yb = xbatch[sl], ybatch[sl]
        nb = noise_std_batch[sl] if noise_std_batch is not None else None
        learn_hyper = torch.is_grad_enabled() and (self.learn_kernel or (self.learn_noise and nb is None))
        if learn_hyper:
            return self._elbo_and_grad_traced(xb, yb, nb, bsz, sharded, maxiter_cg, integrated_obs, semi_integrated_estimator,
                                              semi_integrated_samps, Kmm)
        with torch.no_grad():
            Knm, Knn_diag = self._make_grams(xb, integrated_obs=integrated_obs,
                                             semi_integrated_estimator=semi_integrated_estimator,
                                             semi_integrated_samps=semi_integrated_samps)
            kn = self.compute_kn(Knm, maxiter_cg=maxiter_cg, Kmm=Kmm)
            qm, qS = self.standard_variational_params()
            knt_m, knt_kn, knSkn = self._row_stats(kn, qm, qS)
            y = yb.reshape(-1)
            if nb is not None:
                ivar_noise = (1 / (nb ** 2)).reshape(-1)
                log_noise_std = torch.log(nb).reshape(-1)
            else:
                ivar_noise = torch.exp(-self.log_noise2) * torch.ones_like(y)
                log_noise_std = 0.5 * self.log_noise2
            # compute_batch_an, hipgp.py:370-414
            mse = (knt_m - y) ** 2
            variance = Knn_diag.reshape(-1) - knt_kn + knSkn
            batch_an = -0.5 * ivar_noise * (mse + variance) - log_noise_std - 0.5 * np.log(2 * np.pi)
            an_sum = batch_an.sum().reshape(1)
            elbo_estimate = self._natural_gradient_step(kn, knt_m, y, ivar_noise, an_sum, qm, qS, bsz, sharded)
        return elbo_estimate

    def _natural_gradient_step(self, kn, knt_m, y, ivar_noise, an_sum, qm, qS, bsz, sharded):
        """natural-gradient statistics (hipgp.py:241-250), their all-reduce over the shards of the minibatch, the two
        `.grad` fields; returns the (detached) ELBO estimate"""
        bdiff = ivar_noise * (knt_m - y)
        dm_sum, lam_sum = self._batch_stats(kn, bdiff, ivar_noise)
        if sharded:
            hdist.allreduce_packed([dm_sum, lam_sum, an_sum])      # the one data-path collective of the step
        bscale = self.N / bsz
        data_dm = -dm_sum[:, None]
        dm = bscale * data_dm - qm
        deta1, deta2 = self._natural_gradient(dm, lam_sum, qm, bscale)
        self.global_theta1.grad = -deta1
        self.global_theta2.grad = -deta2
        kl_to_prior = self.get_kl_to_prior(qm, qS)
        return an_sum[0] / bsz - (kl_to_prior / self.N)

    def compute_batch_an(self, xbatch, ybatch, noise_std_batch=None, qm=None, qS=None, Knm=None, Knn_diag=None, kn=None,
                         maxiter_cg=10, integrated_obs=False, semi_integrated_estimator="analytic", semi_integrated_samps=10,
                         Kmm=None, **_ignored):
        """a_n = -1/2 ln 2 pi sigma_n^2 - 1/(2 sigma_n^2) [K_nn - k_n^T k_n + k_n^T S k_n + (k_n^T m - y)^2]  (hipgp.py:370-414),
        in differentiable torch ops on k_n: this is the route the hyper-parameter gradients take"""
        if qm is None or qS is None:
            qm, qS = self.standard_variational_params()
        if Knm is None or Knn_diag is None:
            Knm, Knn_diag = self._make_grams(xbatch, integrated_obs=integrated_obs, semi_integrated_estimator=semi_integrated_estimator,
                                             semi_integrated_samps=semi_integrated_samps)
        if kn is None:
            kn = self.compute_kn(Knm, maxiter_cg=maxiter_cg, Kmm=Kmm)
        y = ybatch.reshape(-1)
        knt_kn = torch.sum(kn * kn, dim=-1)
        knt_m = kn.matmul(qm).reshape(-1)
        knSkn = self._knSkn_traced(kn, qS)
        if noise_std_batch is not None:
            ivar_noise = (1 / (noise_std_batch ** 2)).reshape(-1)
            log_noise_std = torch.log(noise_std_batch).reshape(-1)
        else:
            ivar_noise = torch.exp(-self.log_noise2)
            log_noise_std = 0.5 * self.log_noise2
        mse = (knt_m - y) ** 2
        variance = Knn_diag.reshape(-1) - knt_kn + knSkn
        return -0.5 * ivar_noise * (mse + variance) - log_noise_std - 0.5 * np.log(2 * np.pi)

    def _knSkn_traced(self, kn, qS):
        return torch.sum((kn * qS.t()) * kn, dim=-1)          # hipgp.py:523-524

    def elbo(self, xbatch, ybatch, noise_std_batch=None, maxiter_cg=10, integrated_obs=False, semi_integrated_estimator="analytic",
             semi_integrated_samps=10, Kmm=None, print_debug_info=False):
        """the ELBO estimate with every gradient on the tape (hipgp.py:160-192)"""
        Knm, Knn_diag = self._make_grams(xbatch, integrated_obs=integrated_obs, semi_integrated_estimator=semi_integrated_estimator,
                                         semi_integrated_samps=semi_integrated_samps)
        kn = self.compute_kn(Knm, maxiter_cg=maxiter_cg, Kmm=Kmm)
        qm, qS = self.standard_variational_params()
        batch_an = self.compute_batch_an(xbatch, ybatch, noise_std_batch, qm=qm, qS=qS, Knm=Knm, Knn_diag=Knn_diag, kn=kn)
        return torch.mean(batch_an) - (self.get_kl_to_prior(qm, qS) / self.N)

    def _elbo_and_grad_traced(self, xb, yb, nb, bsz, sharded, maxiter_cg, integrated_obs, estimator, samps, Kmm):
        """learn_kernel / learn_noise: the reference keeps the ELBO on the autograd tape through k_n = R^T K^-1 K_un down to
        log_sig2 / log_ell / log_noise2 ("we still trace kernel grads", hipgp.py:214-218) while the natural gradients of the
        variational parameters are set by hand.  Here K_xu, the first row, the solve and R^T are custom autograd nodes around
        the CUDA kernels; the statistics downstream of k_n are torch ops.  Sharded minibatches: every rank backpropagates its
        own part of the ELBO; the caller all-reduces the hyper-parameter gradients (as DistributedDataParallel would)."""
        Knm, Knn_diag = self._make_grams(xb, integrated_obs=integrated_obs, semi_integrated_estimator=estimator, semi_integrated_samps=samps)
        kn = self.compute_kn(Knm, maxiter_cg=maxiter_cg, Kmm=Kmm)
        with torch.no_grad():
            qm, qS = self.standard_variational_params()
        batch_an = self.compute_batch_an(xb, yb, nb, qm=qm, qS=qS, Knm=Knm, Knn_diag=Knn_diag, kn=kn)
        with torch.no_grad():
            knd = kn.detach()
            y = yb.reshape(-1)
            ivar_noise = (1 / (nb ** 2)).reshape(-1) if nb is not None else torch.exp(-self.log_noise2) * torch.ones_like(y)
            knt_m = self._row_stats(knd, qm, qS)[0]
            an_sum = batch_an.detach().sum().reshape(1)
            self._natural_gradient_step(knd, knt_m, y, ivar_noise, an_sum, qm, qS, bsz, sharded)
        # traced estimate: this rank's observations over the GLOBAL minibatch size (= torch.mean when not sharded)
        return batch_an.sum() / bsz - (self.get_kl_to_prior(qm, qS) / self.N)

    def predict(self, x, integrated_obs=False, semi_integrated_estimator="analytic", semi_integrated_samps=10,
                maxiter_cg=50, Kmm=None, _on_device=False):
        """E[f(x)] and sd[f(x)] (hipgp.py:416-446)"""
        x = x.to(self.xgrids[0].device)
        with torch.no_grad():
            Knm, Knn_diag = self._make_grams(x, integrated_obs=integrated_obs,
                                             semi_integrated_estimator=semi_integrated_estimator,
                                             semi_integrated_samps=semi_integrated_samps)
            kn = self.compute_kn(Knm, maxiter_cg=maxiter_cg, Kmm=Kmm)
            qm, qS = self.standard_variational_params()
            knt_m, knt_kn, knSkn = self._row_stats(kn, qm, qS)
            ktilde_star = (Knn_diag.reshape(-1) - knt_kn).clamp_min(1e-5)
            sig_star = torch.sqrt(ktilde_star + knSkn)[:, None]
        if _on_device:
            return knt_m[:, None].detach(), sig_star.detach()
        return knt_m[:, None].cpu().detach(), sig_star.cpu().detach()


class _BlockKnSkn(torch.autograd.Function):
    """knSkn_b = kn_b^T blockdiag(S) kn_b for kn (B, M'), S (num_blocks, bs, bs) read through the block index map, as a
    differentiable map (the reference gets its gradient from autograd through block_diag_multiply, hipgp.py:640-652).
    Forward: compute_knSkn's kernels.  Backward: dkn = g (S + S^T) kn through `hipgp_block_quadform_grad`, and, when S
    requires a gradient (`elbo` in the 'standard' parameterisation), dS_k = sum_b g_b kn_blk,b kn_blk,b^T through
    `hipgp_block_lam`."""

    @staticmethod
    def forward(ctx, kn, S, blk_idx):
        ctx.save_for_backward(kn, S, blk_idx)
        return row_dot(kn, block_diag_multiply(S, kn, blk_idx))

    @staticmethod
    def backward(ctx, grad_output):
        kn, S, idx = ctx.saved_tensors
        g = grad_output.contiguous()
        dkn = block_quadform_grad(S, kn, g, idx) if ctx.needs_input_grad[0] else None
        dS = block_lam(kn, g, idx, scale=1.0, diag=0.0).to(S.dtype) if ctx.needs_input_grad[1] else None
        return dkn, dS, None


class BlockToeplitzGP(MeanFieldToeplitzGP):
    """Block-diagonal variational family (ziggy/hipgp.py:527-690): q(u) = N(m, blockdiag(S_k)) with the blocks being
    neighbouring chunks of the WHITENED (2m-2)-grid.  `qm` is kept in Toeplitz ordering, the blocks in block ordering;
    the two contractions over k_n run through `hipgp_block_lam` / `hipgp_block_diag_multiply`, which read k_n through the
    index map (no permuted copies, no (bsz, num_blocks, bs, bs) outer products as in hipgp.py:252-255).  The ELBO /
    natural-gradient step and `predict` are the shared code of the mean-field class with this family's statistics;
    learn_kernel / learn_noise take the mean-field class's traced step with knSkn through `_BlockKnSkn`."""

    def __init__(self, kernel, xgrids, num_obs, xblock_size=10, block_sizes=None, sig2_init=1., ell_init=.05, noise2_init=1.,
                 init_Svar=.1, learn_kernel=False, learn_noise=False, dtype=torch.float, whitened_type='ziggy',
                 parameterization='expectation-family', jitter_val=1e-3):
        ToeplitzInducingGP.__init__(self, kernel, xgrids, num_obs, sig2_init=sig2_init, ell_init=ell_init,
                                    noise2_init=noise2_init, learn_kernel=learn_kernel, learn_noise=learn_noise, dtype=dtype,
                                    whitened_type=whitened_type, parameterization=parameterization, jitter_val=jitter_val)
        input_dim = len(xgrids)
        if block_sizes is not None:
            assert input_dim == len(block_sizes), "xgrids ndim = {}, block ndim = {}".format(input_dim, len(block_sizes))
        else:
            block_sizes = [xblock_size for _ in range(input_dim)]
        expanded_xgrids = self.get_expanded_xgrids(xgrids)
        self.block_idx, self.to_blocks, self.from_blocks = hutil.define_block_chunks(expanded_xgrids, block_sizes)
        self.num_blocks, self.block_size = self.block_idx.shape
        self._block_idx_dev = None
        eye = torch.eye(self.block_size, dtype=self.dtype)
        if self.parameterization == 'standard':
            self.global_m = nn.Parameter(torch.nn.init.xavier_normal_(torch.zeros(self.Mprime, 1, dtype=self.dtype)))
            self.global_S = nn.Parameter(torch.stack([init_Svar * eye for _ in range(self.num_blocks)]))
        else:
            self.global_theta1 = nn.Parameter(torch.nn.init.xavier_normal_(torch.zeros(self.Mprime, 1, dtype=self.dtype)))
            self.global_theta2 = nn.Parameter(torch.stack([(-.5 / init_Svar) * eye for _ in range(self.num_blocks)]))

    @property
    def name(self):
        return 'block'

    def get_expanded_xgrids(self, xgrids):
        return [torch.arange(2 * len(x) - 2) for x in xgrids]

    def _idx(self, device):
        if self._block_idx_dev is None or self._block_idx_dev.device != device:
            self._block_idx_dev = self.block_idx.to(device)
        return self._block_idx_dev

    def standard_variational_params(self):
        if self.parameterization == 'standard':
            return self.global_m, self.global_S
        S = self._spd_inverse(-2 * self.global_theta2.data)
        m = self.block_diag_multiply(S, self.global_theta1.data.t()).t()
        return m, S

    def block_diag_multiply(self, S_block, v):
        """S_block (num_blocks, bs, bs) times v (bsz, M') in Toeplitz ordering (hipgp.py:640-652)"""
        bsz, _ = v.shape
        Sv = block_diag_multiply(S_block, v, self._idx(v.device))
        assert Sv.shape == (bsz, self.num_blocks * self.block_size), Sv.shape
        return Sv

    @staticmethod
    def _spd_inverse(A):
        """batched inverse of the (num_blocks, bs, bs) precision blocks (library calls on small dense matrices).  The
        blocks are symmetric positive definite whenever q(u) is a proper Gaussian, so A^-1 = L^-T L^-1 from one batched
        Cholesky (5x faster than the LU route of `torch.inverse`, hipgp.py:634); anything else falls back to LU."""
        Lc, info = torch.linalg.cholesky_ex(A)
        if bool((info != 0).any()):
            return torch.inverse(A)
        eye = torch.eye(A.shape[-1], dtype=A.dtype, device=A.device).expand_as(A)
        Li = torch.linalg.solve_triangular(Lc, eye, upper=False)
        return Li.transpose(-1, -2) @ Li

    def get_S_from_lam(self, lam):
        return self._spd_inverse(lam)

    def compute_knSkn(self, kn, qS):
        return row_dot(kn, self.block_diag_multiply(qS, kn))

    def _knSkn_traced(self, kn, qS):
        """knSkn on the autograd tape (compute_batch_an under learn_kernel / learn_noise, and `elbo`)"""
        return _BlockKnSkn.apply(kn, qS, self._idx(kn.device))

    def get_identity_for_lam(self):
        return torch.eye(self.block_size, device=self.xgrids[0].device, dtype=self.dtype)

    def get_lam(self, ivar_noise, kn, bscale=1, add_identity=True):
        """Lambda = bscale * sum_n 1/sigma_n^2 kn kn^T (+ I), (num_blocks, bs, bs)  (hipgp.py:666-685)"""
        return block_lam(kn, ivar_noise, self._idx(kn.device), scale=bscale, diag=1.0 if add_identity else 0.0)

    def get_kl_to_prior(self, qm=None, qS=None):
        """stats.py:15-29 block_kl_to_standard (Cholesky log-determinants of the jittered blocks)"""
        if qm is None or qS is None:
            qm, qS = self.standard_variational_params()
        I = torch.eye(qS.shape[1], dtype=qS.dtype, device=qS.device)
        Schol = torch.linalg.cholesky(qS + 1e-4 * I)
        lndet = 2.0 * torch.sum(torch.log(torch.diagonal(Schol, dim1=-2, dim2=-1)))
        D = qS.shape[0] * qS.shape[1]
        Strace = torch.sum(torch.diagonal(qS, dim1=-2, dim2=-1))
        return .5 * (Strace + torch.sum(qm * qm) - lndet - D)

    def _row_stats(self, kn, qm, qS):
        st = meanfield_rowstats(kn, qm, torch.zeros_like(qm))
        return st[0], st[1], self.compute_knSkn(kn, qS)

    def _batch_stats(self, kn, bdiff, ivar_noise):
        dm_sum, _ = meanfield_colstats(kn, bdiff, ivar_noise)
        return dm_sum, block_lam(kn, ivar_noise, self._idx(kn.device), scale=1.0, diag=0.0)

    def _natural_gradient(self, dm, lam_sum, qm, bscale):
        """hipgp.py:251-261"""
        lam_block = bscale * lam_sum + self.get_identity_for_lam().to(lam_sum.device)[None]
        dS = -.5 * lam_block - self.global_theta2.data
        dSdeta1 = self.block_diag_multiply(dS, -2 * qm[None, :, 0])
        return dm + dSdeta1.squeeze().unsqueeze(-1), dS


class FullRankToeplitzGP(ToeplitzInducingGP):
    """The reference's full-rank family (ziggy/hipgp.py:693-797) stores a dense (M', M') variational covariance -- 0.5 TB in fp32 at
    BASELINE config 3 -- and is the reference's own small-problem baseline, outside the structured hot path (SURVEY.md 8,
    DESIGN.md 0).  The name exists so that a switch-over fails with a pointer instead of an AttributeError."""

    def __init__(self, *args, **kwargs):
        raise NotImplementedError("hipgp_b200 implements the mean-field and block-diagonal families (MeanFieldToeplitzGP, "
                                  "BlockToeplitzGP); the dense full-rank family of ziggy/hipgp.py:693-797 is out of scope")
