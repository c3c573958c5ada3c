/* hipgp_b200.h -- C ABI of libhipgp_b200.so: the B200 (sm_100a) implementation of HIP-GP's
 * structured-kernel hot path.  Plain pointers and sizes only; every function returns 0 on success and a
 * negative status otherwise (the message is available from hipgp_last_error(), thread-local).
 * All device pointers must be contiguous, of the plan's dtype, on the plan's device.  Work is enqueued on
 * `stream` (a cudaStream_t passed as void*; NULL = default stream); calls that report scalars to the host
 * (hipgp_pcg, *_host) synchronise that stream before returning.
 *
 * Each entry point names the reference interface (suyashk12/hipgp, package `ziggy`) it replaces.
 */
#ifndef HIPGP_B200_H
#define HIPGP_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hipgp_plan hipgp_plan;

enum { HIPGP_F32 = 0, HIPGP_F64 = 1 };

/* matvec modes                     reference (ziggy/misc/toeplitz_tensor.py : toeplitz_expanded.py "multiply_type") */
enum {
    HIPGP_MV_K = 0,    /* K v            _matmul_by_K    :70-83   : "gram"     (B,M)  -> (B,M)  */
    HIPGP_MV_CINV = 1, /* C^-1 block v   _matmul_by_Cinv :114-125 : "circ_inv" (B,M)  -> (B,M)  */
    HIPGP_MV_RT = 2,   /* R^T v          _matmul_by_RT   :85-97   : "RTv"      (B,M)  -> (B,M') */
    HIPGP_MV_R = 3     /* R w            _matmul_by_R    :99-112  : "Rv"       (B,M') -> (B,M)  */
};

/* which spectrum hipgp_plan_spectrum exports (attributes D, D_sqrt, Di, Di_sqrt; toeplitz_tensor.py:26-33) */
enum { HIPGP_SPEC_D = 0, HIPGP_SPEC_D_SQRT = 1, HIPGP_SPEC_DI = 2, HIPGP_SPEC_DI_SQRT = 3 };

/* kernel families (ziggy/kernels.py) and cross-covariance modes (ziggy/svi_gp.py:48-76) */
enum { HIPGP_K_SQEXP = 0, HIPGP_K_MATERN12 = 1, HIPGP_K_MATERN32 = 2, HIPGP_K_MATERN52 = 3, HIPGP_K_GNEITING = 4 };
enum {
    HIPGP_KXU_POINT = 0,         /* kernel(xbatch, xinduce)            kernels.py:73-79,108-117,145-158 */
    HIPGP_KXU_SEMI_ANALYTIC = 1, /* SqExp.k_semi (ray from the origin) kernels.py:85-90,223-237         */
    HIPGP_KXU_SEMI_MC = 2,       /* Kernel.k_semi_mc                   kernels.py:19-39                 */
    HIPGP_KXU_DERIV = 3,         /* kprime (1-D SqExp d/dx)            exact_gp_1d_derivatives.py:19-23 */
    HIPGP_KXU_DERIV2 = 4         /* kprime_double_full (1-D SqExp)     exact_gp_1d_derivatives.py:32-38 */
};

const char* hipgp_last_error(void);
int hipgp_version(void);

/* ---- plan: replaces ToeplitzTensor.__init__ / ToeplitzMatmul.__init__ (toeplitz_tensor.py:9-45,
 *      toeplitz_expanded.py:82-127).  m[ndim] are the grid extents (C order, last fastest). */
int hipgp_plan_create(int ndim, const int64_t* m, int dtype, int device, hipgp_plan** out);
int hipgp_plan_destroy(hipgp_plan* plan);
/* sizes: M = prod m_d, Mprime = prod (2 m_d - 2)  (1 for m_d == 1; ziggy/hipgp.py:72) */
int hipgp_plan_sizes(const hipgp_plan* plan, int64_t* M, int64_t* Mprime);
/* embedding lengths actually used: narrow (K, C^-1) and wide (R^T, R), ndim entries each */
int hipgp_plan_embedding(const hipgp_plan* plan, int64_t* L_narrow, int64_t* L_wide);

/* first row of K_uu (M values of the plan dtype, device; jitter already added -- toeplitz_tensor.py:127-133)
 * -> D = max(Re FFT(embed(column)), clamp) and the spectra of K, C^-1 (and lazily C^1/2).
 * `clamped_out` (host, optional) receives the number of clamped values among the M DISTINCT spectrum entries (the DCT-I of the
 * column; an interior entry stands for up to 2^ndim equal eigenvalues of the embedding). */
int hipgp_plan_set_first_row(hipgp_plan* plan, const void* column_dev, double clamp, int64_t* clamped_out, void* stream);
/* writes Mprime reals in the reference's (N_1..N_D) layout */
int hipgp_plan_spectrum(hipgp_plan* plan, int which, void* out_dev, void* stream);

/* ---- structured matvecs; `in`/`out` are (B, M) or (B, M') row-major device arrays */
int hipgp_matvec(hipgp_plan* plan, int mode, const void* in_dev, void* out_dev, int64_t B, void* stream);
/* same, host buffers in and out (H2D + D2H inside the call) */
int hipgp_matvec_host(hipgp_plan* plan, int mode, const void* in_host, void* out_host, int64_t B, void* stream);

/* Asynchronous variant for a stream of batches (two slots): submit queues upload (plan's H2D stream) -> whole solve (caller's
 * stream; the stopping rule of cg.py:70 lives on the device, so nothing polls) -> download (plan's D2H stream) and returns;
 * wait blocks until x_host of that slot is complete and reports the iteration count.  With both slots in flight the copies of
 * neighbouring batches run under the current solve.  Re-submitting a busy slot waits for it first.  Host buffers must be pinned
 * and must stay untouched between submit and wait. */
int hipgp_pcg_host_submit(hipgp_plan* plan, const void* b_host, void* x_host, int64_t B, int maxiter, double tol, int precond,
                          int slot, void* stream);
int hipgp_pcg_host_wait(hipgp_plan* plan, int slot, int* iters_out);

/* ---- PCG: replaces conj_grad2/conj_grad driven by ToeplitzTensor._solve / gram_solve
 *      (ziggy/misc/cg.py:5-80, toeplitz_tensor.py:54-68, toeplitz_expanded.py:17-58).
 * b, x: (B, M).  precond != 0 uses the HIP-GP preconditioner (upper-left block of C^-1).
 * Stops when all_b sqrt(r_b.r_b) < tol (checked after the x/r update, as the reference does) or after
 * maxiter iterations.  iters_out: iterations executed; callbacks_out: iterations that did not break
 * (= number of reference callback invocations).  resid_out (host, optional): B values of sqrt(r.r).
 * cb (optional) is called on the host after every non-breaking iteration with x valid on the device. */
typedef void (*hipgp_iter_cb)(int n, const void* x_dev, void* user);
int hipgp_pcg(hipgp_plan* plan, const void* b_dev, void* x_dev, int64_t B, int maxiter, double tol, int precond,
              int* iters_out, int* callbacks_out, double* resid_out, hipgp_iter_cb cb, void* user, void* stream);
/* the same solve split in two, for callers that own the stopping rule (a minibatch sharded over several GPUs must
 * stop on all_b over ALL ranks, cg.py:70): begin = everything before the loop; step = `niter` more iterations, then
 * (if any out pointer is given) a stream sync and done flag / iteration count / max_b sqrt(r_b.r_b) of this rank.
 * Pass tol < 0 to begin to disable the local stopping test. */
int hipgp_pcg_begin(hipgp_plan* plan, const void* b_dev, void* x_dev, int64_t B, double tol, int precond, void* stream);
int hipgp_pcg_step(hipgp_plan* plan, int niter, int* done_out, int* iters_out, double* max_resid_out, void* stream);
int hipgp_pcg_host(hipgp_plan* plan, const void* b_host, void* x_host, int64_t B, int maxiter, double tol, int precond,
                   int* iters_out, int* callbacks_out, double* resid_out, void* stream);
/* host-buffer solve with the copies hidden behind the solves: a first and a last group of `group` right-hand sides and one
 * big group in between (uniform groups of `group` when B < 4 group; <= 0: all at once); H2D of group g+1 and D2H of group
 * g-1 overlap the solve of group g (two plan-owned copy streams).  Each group is an
 * independent batched solve (the stopping rule of cg.py:70 spans one group); iters_out = max over groups.  Pinned buffers. */
int hipgp_pcg_host_pipelined(hipgp_plan* plan, const void* b_host, void* x_host, int64_t B, int maxiter, double tol,
                             int precond, int64_t group, int* iters_out, void* stream);
/* k_n = R^T K^-1 K_un  (ziggy/hipgp.py:139-146): PCG(precond) followed by R^T.  Knm (B,M) -> kn (B,M') */
int hipgp_compute_kn(hipgp_plan* plan, const void* Knm_dev, void* kn_dev, int64_t B, int maxiter, double tol,
                     int* iters_out, void* stream);

/* ---- fused CG vector updates for callers that bring their own A_mul / precond closures
 *      (cg.py:25-36 / :64-75).  All vectors (B, M) in the plan dtype; scalars (B) fp64 on the device. */
int hipgp_vec_dot(int dtype, const void* a_dev, const void* b_dev, double* out_dev, int64_t B, int64_t M, void* stream);
/* x += alpha p ; r -= alpha Ap with alpha = rs / pAp ; rr_out = r.r */
int hipgp_vec_xr_update(int dtype, void* x_dev, void* r_dev, const void* p_dev, const void* Ap_dev, const double* rs_dev,
                        const double* pAp_dev, double* rr_out_dev, int64_t B, int64_t M, void* stream);
/* p = z + (zr_new / zr_old) p */
int hipgp_vec_p_update(int dtype, void* p_dev, const void* z_dev, const double* zr_new_dev, const double* zr_old_dev,
                       int64_t B, int64_t M, void* stream);

/* ---- cross-covariances evaluated on the fly from the grid (ziggy/svi_gp.py:48-76 `_make_grams`).
 * x: (B, ndim) device; grids: the concatenated 1-D grid coordinates (sum m_d values, plan dtype, device);
 * ell: 1 or ndim host doubles (n_ell); out: (B, M) row-major.  mc_alphas: npts values (device, plan dtype)
 * for SEMI_MC -- the stratified offsets arange(npts)/npts + U/npts drawn by the caller (kernels.py:25-27). */
int hipgp_kxu(int dtype, int kernel_id, int mode, double sig2, const double* ell, int n_ell, double gneiting_alpha,
              const void* x_dev, int64_t B, int ndim, const int64_t* m, const void* grids_dev,
              const void* mc_alphas_dev, int npts, void* out_dev, void* stream);
/* the same kernels between two explicit point sets x (n, ndim) and y (m, ndim) -> out (n, m): the generic
 * Kernel.forward(x, y) (kernels.py:73-79,108-117,145-158) and k_semi / k_semi_mc / kprime with y the point set */
int hipgp_kernel_pairwise(int dtype, int kernel_id, int mode, double sig2, const double* ell, int n_ell, double gneiting_alpha,
                          const void* x_dev, int64_t n, const void* y_dev, int64_t m, int ndim,
                          const void* mc_alphas_dev, int npts, void* out_dev, void* stream);
/* hyper-parameter derivatives of K_xu for learn_kernel=True (the reference lets autograd differentiate kernels.py:73-79,
 * 145-158): per-block partial sums of G * {dk/dsig2, dk/dell_0, dk/dell_1, dk/dell_2} over the columns of row b; `partial` holds
 * B * ceil(M/1024) * 4 doubles, the caller adds them up.  Either the 1-D grids (grids != NULL, as hipgp_kxu) or an explicit
 * second point set ypts (n_y x ndim, as hipgp_kernel_pairwise).  Modes POINT and SEMI_MC with the SqExp / Matern kernels;
 * SEMI_ANALYTIC with SqExp (closed form of the derivative of the analytic line integral). */
int hipgp_kxu_param_grad(int dtype, int kernel_id, int mode, double sig2, const double* ell, int n_ell, const void* x_dev, int64_t B,
                         int ndim, const int64_t* m, const void* grids_dev, const void* ypts_dev, int64_t n_y, const void* mc_alphas_dev,
                         int npts, const void* G_dev, double* partial_dev, void* stream);
/* KernelDoublyDiagInterpolator.forward (kernels.py:199-218); table = distance_grid, slopes, knn (ntab each, device) */
int hipgp_doubly_diag(int dtype, const void* x_dev, int64_t B, int ndim, double sig2, const double* ell, int n_ell,
                      const void* distance_grid_dev, const void* slopes_dev, const void* knn_dev, int ntab,
                      void* out_dev, void* stream);
/* hyper-parameter derivatives of hipgp_doubly_diag for learn_kernel=True (the reference lets autograd differentiate
 * kernels.py:199-218): with out_b = ell^2 sig2 iv_b, d/dsig2 = ell^2 iv_b and d/dell = sig2 ell (2 iv_b - slope_b |x_b| / ell).
 * Scalar ell only (n_ell == 1).  g: upstream gradient (B, dtype).  partial holds ceil(B/256) * 2 doubles = per-block sums of
 * g * {d/dsig2, d/dell}; the caller adds them up.  B = 0 is a no-op. */
int hipgp_doubly_diag_param_grad(int dtype, const void* x_dev, int64_t B, int ndim, double sig2, const double* ell, int n_ell,
                                 const void* distance_grid_dev, const void* slopes_dev, const void* knn_dev, int ntab,
                                 const void* g_dev, double* partial_dev, void* stream);

/* ---- mean-field natural-gradient reductions over k_n (B, M') (ziggy/hipgp.py:241-250,395-397,439,524).
 * rowstats: out[0][b] = k_n[b].qm, out[1][b] = k_n[b].k_n[b], out[2][b] = sum_j k_n[b,j]^2 qS[j]   (3 x B, plan dtype)
 * colstats: dm[j] = sum_b w1[b] k_n[b,j], lam[j] = sum_b w2[b] k_n[b,j]^2                       (M' each) */
int hipgp_meanfield_rowstats(int dtype, const void* kn_dev, const void* qm_dev, const void* qS_dev, int64_t B, int64_t E,
                             void* out_dev, void* stream);
int hipgp_meanfield_colstats(int dtype, const void* kn_dev, const void* w1_dev, const void* w2_dev, int64_t B, int64_t E,
                             void* dm_dev, void* lam_dev, void* stream);

/* ---- block-diagonal variational family (ziggy/hipgp.py:527-690; index maps of ziggy/misc/util.py:79-126).
 * blk_idx (num_blocks x block_size, int64, device) is the permutation `define_block_chunks` returns; nblk * bs = M'.
 * block_lam:            lam[k][i][j] = scale * sum_n w[n] kn[n, idx[k,i]] kn[n, idx[k,j]] + diag * (i == j)
 *                       (get_lam, hipgp.py:666-685; the natural-gradient branch :251-257 with scale = N / bsz, diag = 1)
 * block_diag_multiply:  out[b, idx[k,i]] = sum_j S[k][i][j] v[b, idx[k,j]]   (= from_blocks(S to_blocks(v)), hipgp.py:640-652)
 * kn, v, out: (B, M'); w: (B); S, lam: (nblk, bs, bs); all in `dtype`. */
int hipgp_block_lam(int dtype, const void* kn_dev, const void* w_dev, const int64_t* blk_idx_dev, int64_t B, int64_t E,
                    int64_t nblk, int64_t bs, double scale, double diag, void* lam_dev, void* stream);
int hipgp_block_diag_multiply(int dtype, const void* S_dev, const void* v_dev, const int64_t* blk_idx_dev, int64_t B,
                              int64_t E, int64_t nblk, int64_t bs, void* out_dev, void* stream);
/* block_quadform_grad:  dkn[b, idx[k,i]] = g[b] sum_j (S[k][i][j] + S[k][j][i]) kn[b, idx[k,j]]
 *                       the gradient of knSkn_b = kn_b^T blockdiag(S) kn_b with upstream g (B), which the reference gets from
 *                       autograd through block_diag_multiply and the row sum of compute_batch_an (hipgp.py:640-652, :370-414)
 *                       when it traces kernel / noise hyper-parameters (:214-218).  S + S^T, so any S (the 'standard'
 *                       parameterisation does not keep it symmetric).  Deterministic (no atomics); B = 0 is a no-op;
 *                       dkn must not overlap kn. */
int hipgp_block_quadform_grad(int dtype, const void* S_dev, const void* kn_dev, const void* g_dev, const int64_t* blk_idx_dev,
                              int64_t B, int64_t E, int64_t nblk, int64_t bs, void* dkn_dev, void* stream);

/* ---- Toeplitz-column quadratic form: the kernel-hyper-parameter gradient of InvMatmul.backward
 * (ziggy/misc/_inv_matmul.py:39-55 -> gpt_toeplitz.py:169-209 sym_toeplitz_derivative_quadratic_form, evaluated there on
 * the FLATTENED M-vectors with 1-D FFTs of length 2M-1).  left/right: S pairs of M-vectors (device, row-major S x M);
 *   out[i] = scale * sum_j sum_k ( u_j[k+i] v_j[k] + v_j[k+i] u_j[k] )   (1 <= i < M),   out[0] = scale * sum_j u_j . v_j
 * over the flattened index.  InvMatmul.backward is this with S = B, u = left solves, v = right solves, scale = -1. */
int hipgp_toeplitz_quadform(hipgp_plan* plan, const void* left_dev, const void* right_dev, int64_t S, double scale,
                            void* out_dev, void* stream);
/* gradient of sum_b grad_out_b . (R^T vec_b) with respect to the Toeplitz column (learn_kernel=True; the reference gets it
 * from autograd through toeplitz_tensor.py:21-33,85-97: D_sqrt = sqrt(max(Re FFT C, 1e-6))).  vec (B,M), grad_out (B,M'),
 * out (M) in the plan dtype, multiplied by `scale`.  Clamped eigenvalues contribute nothing (torch.clamp's gradient). */
int hipgp_rt_column_grad(hipgp_plan* plan, const void* vec_dev, const void* grad_out_dev, int64_t B, double scale, void* out_dev,
                         void* stream);

/* ---- slab-decomposed 3-D grids (axis 0 split over `nranks` GPUs; K and C^-1 matvecs; one right-hand side).
 * The reference has no multi-GPU path; this is the grid-sharded route of SURVEY.md 8e.  What travels is the UN-PADDED output
 * of the row pass, split along the bins of the last axis; after the exchange a rank owns all (i0, i1) for its bins and runs
 * the three ordinary column passes locally:
 *   stage_a(in_slab -> send) ; all-to-all(send -> buf) ; stage_b(mode, buf in place) ; all-to-all(buf -> recv) ; stage_c(recv -> out_slab)
 * with the two all-to-alls issued by the caller (NCCL through torch.distributed), or the peer-memory exchange below.
 * Buffers: slab = (n0/nranks, m1, m2) reals; exchange = `exchange_complex` complex numbers = nranks equal blocks. */
int hipgp_plan_set_slab(hipgp_plan* plan, int rank, int nranks);
int hipgp_slab2_sizes(const hipgp_plan* plan, int64_t* slab_reals, int64_t* exchange_complex);
int hipgp_slab2_stage_a(hipgp_plan* plan, const void* in_slab_dev, void* send_buf_dev, void* stream);
int hipgp_slab2_stage_b(hipgp_plan* plan, int mode, void* buf_dev, void* stream);
int hipgp_slab2_stage_c(hipgp_plan* plan, const void* recv_buf_dev, void* out_slab_dev, void* stream);
/* Overlap: with `nchunks` > 1 (set before hipgp_slab2_sizes) the exchange buffer is laid out [chunk][rank][rows][bins/chunk], so
 * every chunk is a contiguous all-to-all of its own (exchange_complex / nchunks numbers) and stage_b can run on chunk c while
 * chunk c+1 is still on the wire and chunk c-1 already travels back. */
int hipgp_plan_set_slab_chunks(hipgp_plan* plan, int nchunks);
int hipgp_slab2_stage_b_chunk(hipgp_plan* plan, int mode, void* buf_dev, int chunk, void* stream);
/* Peer-memory exchange (one process per GPU on one NVLink / NVSwitch node): no collective library on the data path.
 * The plan owns two receive buffers; ranks swap their inter-process handles (64 bytes each, e.g. with an all-gather) and
 * open them; then the packing kernel's 16-byte stores go straight into the peers' buffers over NVLink:
 *   push_a(in_slab)      rows r2c, every destination's bins stored into ITS first buffer
 *   -- barrier across ranks (any stream-ordered collective) --
 *   push_b(mode, chunk)  the column passes in place on the own first buffer, results stored into the peers' second buffers
 *   -- barrier --
 *   finish(out_slab)     own second buffer -> rows c2r
 * The two barriers also order the buffers' reuse by the next matvec.  peer_set takes raw addresses instead of handles for
 * ranks that live in one process. */
int hipgp_slab2_peer_alloc(hipgp_plan* plan, void** r1_out, void** r2_out, void* handle1_64, void* handle2_64);
int hipgp_slab2_peer_open(hipgp_plan* plan, const void* handles1, const void* handles2);
int hipgp_slab2_peer_set(hipgp_plan* plan, void* const* r1_all, void* const* r2_all);
int hipgp_slab2_push_a(hipgp_plan* plan, const void* in_slab_dev, void* stream);
int hipgp_slab2_push_b(hipgp_plan* plan, int mode, int chunk, void* stream);
int hipgp_slab2_finish(hipgp_plan* plan, void* out_slab_dev, void* stream);
/* measurement aid: the transfer kernel of push_a (back = 0) or push_b (back = 1) alone, on whatever the buffers hold */
int hipgp_slab2_push_only(hipgp_plan* plan, int back, void* stream);

/* bytes of device memory the plan currently owns (spectra, twiddles, workspace) */
int hipgp_plan_device_bytes(const hipgp_plan* plan, size_t* bytes);
/* number of kernel launches issued through this plan since creation (for bench accounting) */
int hipgp_plan_launch_count(const hipgp_plan* plan, int64_t* launches);

/* per-kernel-class device timing (CUDA events around every launch while enabled); classes:
 * 0 rows_fwd (last-axis r2c pass), 1 cols_pass (strided axes, spectrum multiply), 2 rows_inv (c2r pass),
 * 3 stand-alone vector kernel.  Used by bench.py for the roofline figure; off by default. */
int hipgp_plan_profile(hipgp_plan* plan, int enable);
int hipgp_plan_profile_read(hipgp_plan* plan, int kernel_class, double* ms_total, int64_t* launches, int reset);

#ifdef __cplusplus
}
#endif
#endif
