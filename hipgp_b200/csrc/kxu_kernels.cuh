// kxu_kernels.cuh -- cross-covariance K_xu evaluated on the fly from the grid structure.
//
// The reference materialises an (n, M, D) difference tensor per minibatch (ziggy/kernels.py:78,149,112) and,
// for line integrals, an (n, M, 1, 1) batched matmul (kernels.py:228).  Here every output element is computed
// from the D grid coordinates of its column index; nothing but the (B, M) result touches HBM.
#pragma once
#include "cuda_emu.h"

namespace hipgp {

struct KxuParams {
    int kernel_id, mode, ndim, npts;
    int m[3];               // grid extents, right-aligned active axes are NOT required here: plain ndim
    int goff[3];            // offsets of each axis's coordinates inside `grids`
    double sig2, alpha;     // alpha: Gneiting exponent
    double ell[3];          // per-axis length scale (scalar ell replicated)
    double ell0;            // the scalar ell (Matern divides the unscaled distance by it, kernels.py:149)
    long B, M;
};

template <class T> struct M_ {};
template <> struct M_<float> {
    static __device__ __forceinline__ float exp(float x) { return ::expf(x); }
    static __device__ __forceinline__ float sqrt(float x) { return ::sqrtf(x); }
    static __device__ __forceinline__ float erf(float x) { return ::erff(x); }
    static __device__ __forceinline__ float cos(float x) { return ::cosf(x); }
    static __device__ __forceinline__ float sin(float x) { return ::sinf(x); }
    static __device__ __forceinline__ float pow(float x, float y) { return ::powf(x, y); }
};
template <> struct M_<double> {
    static __device__ __forceinline__ double exp(double x) { return ::exp(x); }
    static __device__ __forceinline__ double sqrt(double x) { return ::sqrt(x); }
    static __device__ __forceinline__ double erf(double x) { return ::erf(x); }
    static __device__ __forceinline__ double cos(double x) { return ::cos(x); }
    static __device__ __forceinline__ double sin(double x) { return ::sin(x); }
    static __device__ __forceinline__ double pow(double x, double y) { return ::pow(x, y); }
};

// k(x, u) for one pair; x, u given per axis.  Follows ziggy/kernels.py:73-79 (SqExp), :145-158 (Matern),
// :108-117 (Gneiting) operation by operation in the plan dtype.
template <class T>
__device__ __forceinline__ T eval_point(const KxuParams& P, const T* x, const T* u) {
    const T sig2 = (T)P.sig2;
    if (P.kernel_id == 0) {
        T sq = 0;
        for (int d = 0; d < P.ndim; ++d) { const T t = (x[d] - u[d]) / (T)P.ell[d]; sq += t * t; }
        return sig2 * M_<T>::exp(-sq / (T)2);
    }
    if (P.kernel_id == 4) {
        T sq = 0;
        for (int d = 0; d < P.ndim; ++d) { const T t = (x[d] - u[d]) / (T)P.ell[d]; sq += t * t; }
        const T t = M_<T>::sqrt(sq);
        if (t > (T)1) return sig2 * (T)0;
        const T pi = (T)3.14159265358979323846;
        const T cterms = ((T)1 - t) * M_<T>::cos(pi * t) + ((T)1 / pi) * M_<T>::sin(pi * t);
        const T base = (T)1 + M_<T>::pow(t, (T)P.alpha);
        return sig2 * (cterms / (base * base * base));
    }
    T sq = 0;
    for (int d = 0; d < P.ndim; ++d) { const T t = x[d] - u[d]; sq += t * t; }
    const T ell = (T)P.ell0;
    const T r = M_<T>::sqrt(sq);
    T k;
    if (P.kernel_id == 1) {
        k = M_<T>::exp(-r / ell);
    } else if (P.kernel_id == 2) {
        const T dp = (T)1.7320508075688772 * r / ell;
        k = ((T)1 + dp) * M_<T>::exp(-dp);
    } else {
        const T dp = (T)2.23606797749979 * r / ell;
        k = ((T)1 + dp + (T)(5. / 3.) * sq / (ell * ell)) * M_<T>::exp(-dp);
    }
    return sig2 * k;
}

// grid (ceil(M / (256*4)), B); block 256.  out[b][j]
template <class T>
__global__ void __launch_bounds__(256) kxu_kernel(KxuParams P, const T* __restrict__ xb, const T* __restrict__ grids,
                                                  const T* __restrict__ ypts, const T* __restrict__ alphas, T* __restrict__ out) {
    const long b = blockIdx.y;
    T x[3] = {0, 0, 0};
    for (int d = 0; d < P.ndim; ++d) x[d] = xb[b * P.ndim + d];
    // per-observation scalars of the analytic line integral (kernels.py:225-227,232-233)
    T a = 0, xnorm = 0;
    for (int d = 0; d < P.ndim; ++d) { a += x[d] * ((T)1 / ((T)P.ell[d] * (T)P.ell[d])) * x[d]; xnorm += x[d] * x[d]; }
    xnorm = M_<T>::sqrt(xnorm);
    const long j0 = (long)blockIdx.x * (blockDim.x * 4);
    for (int it = 0; it < 4; ++it) {
        const long j = j0 + it * blockDim.x + threadIdx.x;
        if (j >= P.M) break;
        long rem = j;
        T u[3] = {0, 0, 0};
        if (ypts) {   // explicit second point set (generic Kernel.forward); otherwise the C-order grid
            for (int d = 0; d < P.ndim; ++d) u[d] = ypts[j * P.ndim + d];
        } else {
            for (int d = P.ndim - 1; d >= 0; --d) { const int jd = (int)(rem % P.m[d]); rem /= P.m[d]; u[d] = grids[P.goff[d] + jd]; }
        }
        T val;
        if (P.mode == 0) {
            val = eval_point<T>(P, x, u);
        } else if (P.mode == 1) {
            // semi_integrated_sqe, kernels.py:223-237 with Sinv = diag(1/ell^2)
            T bq = 0, c = 0;
            for (int d = 0; d < P.ndim; ++d) {
                const T si = (T)1 / ((T)P.ell[d] * (T)P.ell[d]);
                bq += x[d] * si * u[d]; c += u[d] * si * u[d];
            }
            const T scale = M_<T>::sqrt((T)1 / a);
            const T loc = bq / a;
            const T coef = (T)P.sig2 * M_<T>::exp((bq * bq) / ((T)2 * a) - c / (T)2) * (T)2.5066282746310002 * scale;
            const T sqrt2 = (T)1.4142135623730951;
            const T ca = (T).5 * ((T)1 + M_<T>::erf(((T)1 - loc) / (scale * sqrt2)));
            const T cb = (T).5 * ((T)1 + M_<T>::erf(((T)0 - loc) / (scale * sqrt2)));
            val = coef * (ca - cb) * xnorm;
        } else if (P.mode == 2) {
            // k_semi_mc, kernels.py:19-39: mean over the stratified points alpha_t x, times |x|
            T acc = 0;
            for (int t = 0; t < P.npts; ++t) {
                T xa[3];
                const T al = alphas[t];
                for (int d = 0; d < P.ndim; ++d) xa[d] = x[d] * al;
                acc += eval_point<T>(P, u, xa);
            }
            val = (acc / (T)P.npts) * xnorm;
        } else if (P.mode == 3) {
            // kprime, exact_gp_1d_derivatives.py:19-23
            const T ell = (T)P.ell0;
            const T diff = x[0] - u[0];
            const T Kxy = (T)P.sig2 * M_<T>::exp((T)(-1. / 2.) * (diff * diff) / (ell * ell));
            val = -diff / (ell * ell) * Kxy;
        } else {
            // kprime_double_full, exact_gp_1d_derivatives.py:32-38
            const T ell = (T)P.ell0;
            const T diff = x[0] - u[0];
            const T dsq = diff * diff, esq = ell * ell;
            const T Kxy = (T)P.sig2 * M_<T>::exp((T)(-1. / 2.) * dsq / esq);
            val = Kxy / esq * ((T)1 - (T)1 / esq * dsq);
        }
        out[b * P.M + j] = val;
    }
}

// The table interval of KernelDoublyDiagInterpolator.forward (kernels.py:205-207) for observation b: the scaled distance
// |x_b / ell| and the index of the last table distance below it.
template <class T>
__device__ __forceinline__ int doubly_diag_lookup(const T* __restrict__ xb, long b, int ndim, const T* ell, const T* __restrict__ dgrid,
                                                  int ntab, T* dist_out) {
    T sq = 0;
    for (int d = 0; d < ndim; ++d) { const T t = xb[b * ndim + d] / ell[d]; sq += t * t; }
    const T dist = M_<T>::sqrt(sq);
    int cnt = 0;
    for (int t = 0; t < ntab; ++t) cnt += (dist > dgrid[t]) ? 1 : 0;
    int li = cnt - 1;
    if (li < 0) li += ntab;                 // python negative index wraps to the last entry (SURVEY 8a-bis)
    *dist_out = dist;
    return li;
}

// KernelDoublyDiagInterpolator.forward, kernels.py:199-218
template <class T>
__global__ void doubly_diag_kernel(const T* __restrict__ xb, long B, int ndim, double sig2, double ell0,
                                   const T* __restrict__ dgrid, const T* __restrict__ slopes, const T* __restrict__ knn, int ntab,
                                   T* __restrict__ out, double e0, double e1, double e2) {
    const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    const T ell[3] = {(T)e0, (T)e1, (T)e2};
    T dist;
    const int li = doubly_diag_lookup<T>(xb, b, ndim, ell, dgrid, ntab, &dist);
    const T diff = dist - dgrid[li];
    const T iv = knn[li] + slopes[li] * diff;
    out[b] = (T)ell0 * (T)ell0 * (T)sig2 * iv;
}

// ---- stand-alone fused CG vector kernels (generic closure path) -------------------------------------
template <class T> __device__ __forceinline__ double block_sum_256(double v) {
    __shared__ double red[8];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double t = 0;
    for (int i = 0; i < 8; ++i) t += red[i];
    return t;
}

// ---- hyper-parameter derivatives of the point kernels (learn_kernel = True; the reference lets autograd differentiate
// kernels.py:73-79,145-158).  dk/dsig2 = k / sig2;  dk/dell_d closed form: SqExp k t_d^2 / ell_d (t_d = (x_d-u_d)/ell_d);
// Matern-1/2 k r/ell^2;  Matern-3/2 sig2 a^2 e^-a / ell (a = sqrt3 r/ell);  Matern-5/2 sig2 (a^2/3)(1+a) e^-a / ell (a = sqrt5 r/ell).
template <class T>
__device__ __forceinline__ void eval_point_grad(const KxuParams& P, const T* x, const T* u, double* dsig2, double* dell) {
    dell[0] = dell[1] = dell[2] = 0.0;
    if (P.kernel_id == 0) {
        double sq = 0, td[3] = {0, 0, 0};
        for (int d = 0; d < P.ndim; ++d) { const double t = ((double)x[d] - (double)u[d]) / P.ell[d]; td[d] = t * t; sq += t * t; }
        const double e = ::exp(-0.5 * sq);
        *dsig2 = e;
        for (int d = 0; d < P.ndim; ++d) dell[d] = P.sig2 * e * td[d] / P.ell[d];
        return;
    }
    double sq = 0;
    for (int d = 0; d < P.ndim; ++d) { const double t = (double)x[d] - (double)u[d]; sq += t * t; }
    const double r = ::sqrt(sq), ell = P.ell0;
    if (P.kernel_id == 1) {
        const double e = ::exp(-r / ell);
        *dsig2 = e; dell[0] = P.sig2 * e * r / (ell * ell);
    } else if (P.kernel_id == 2) {
        const double a = 1.7320508075688772 * r / ell, e = ::exp(-a);
        *dsig2 = (1.0 + a) * e; dell[0] = P.sig2 * a * a * e / ell;
    } else {
        const double a = 2.23606797749979 * r / ell, e = ::exp(-a);
        *dsig2 = (1.0 + a + a * a / 3.0) * e; dell[0] = P.sig2 * (a * a / 3.0) * (1.0 + a) * e / ell;
    }
}

// partial[(b * gridDim.x + blockIdx.x) * 4 + {0, 1, 2, 3}] = sum over this block's columns of G[b][j] * {dk/dsig2, dk/dell_0..2}
// (modes POINT, SEMI_ANALYTIC and SEMI_MC; grid as kxu_kernel)
//
// SEMI_ANALYTIC (SqExp, kernels.py:223-237): k = sig2 |x| I0 with I_k = int_0^1 alpha^k e(alpha) dalpha,
// e(alpha) = exp(-(a alpha^2 - 2 b alpha + c) / 2), a = x^T S x, b = x^T S u, c = u^T S u, S = diag(1 / ell_d^2).
// Integration by parts (e' = -(a alpha - b) e) gives I1 = (b I0 + e(0) - e(1)) / a and I2 = (b I1 + I0 - e(1)) / a, so
// dk/dsig2 = |x| I0 and dk/dell_d = sig2 |x| / ell_d^3 (x_d^2 I2 - 2 x_d u_d I1 + u_d^2 I0).
template <class T>
__global__ void __launch_bounds__(256) kxu_grad_kernel(KxuParams P, const T* __restrict__ xb, const T* __restrict__ grids,
                                                       const T* __restrict__ ypts, const T* __restrict__ alphas,
                                                       const T* __restrict__ G, double* __restrict__ partial) {
    const long b = blockIdx.y;
    T x[3] = {0, 0, 0};
    for (int d = 0; d < P.ndim; ++d) x[d] = xb[b * P.ndim + d];
    double xnorm = 0;
    for (int d = 0; d < P.ndim; ++d) xnorm += (double)x[d] * (double)x[d];
    xnorm = ::sqrt(xnorm);
    double acc[4] = {0, 0, 0, 0};
    const long j0 = (long)blockIdx.x * (blockDim.x * 4);
    for (int it = 0; it < 4; ++it) {
        const long j = j0 + it * blockDim.x + threadIdx.x;
        if (j >= P.M) break;
        long rem = j;
        T u[3] = {0, 0, 0};
        if (ypts) { for (int d = 0; d < P.ndim; ++d) u[d] = ypts[j * P.ndim + d]; }
        else { for (int d = P.ndim - 1; d >= 0; --d) { const int jd = (int)(rem % P.m[d]); rem /= P.m[d]; u[d] = grids[P.goff[d] + jd]; } }
        const double g = (double)G[b * P.M + j];
        double ds, de[3];
        if (P.mode == 0) {
            eval_point_grad<T>(P, x, u, &ds, de);
            acc[0] += g * ds; acc[1] += g * de[0]; acc[2] += g * de[1]; acc[3] += g * de[2];
        } else if (P.mode == 1) {
            double a = 0, bq = 0, c = 0;
            for (int d = 0; d < P.ndim; ++d) {
                const double xd = (double)x[d], ud = (double)u[d], si = 1.0 / (P.ell[d] * P.ell[d]);
                a += xd * si * xd; bq += xd * si * ud; c += ud * si * ud;
            }
            const double r2a = ::sqrt(2.0 * a);
            const double I0 = ::exp(bq * bq / (2.0 * a) - 0.5 * c) * ::sqrt(1.5707963267948966 / a) *
                              (::erf((a - bq) / r2a) - ::erf(-bq / r2a));
            const double e0 = ::exp(-0.5 * c), e1 = ::exp(-0.5 * (a - 2.0 * bq + c));
            const double I1 = (bq * I0 + e0 - e1) / a;
            const double I2 = (bq * I1 + I0 - e1) / a;
            acc[0] += g * xnorm * I0;
            const double f = g * P.sig2 * xnorm;
#pragma unroll
            for (int d = 0; d < 3; ++d) {
                if (d < P.ndim) {
                    const double xd = (double)x[d], ud = (double)u[d], el = P.ell[d];
                    acc[1 + d] += f / (el * el * el) * (xd * xd * I2 - 2.0 * xd * ud * I1 + ud * ud * I0);
                }
            }
        } else {          // SEMI_MC: mean over the stratified points alpha_t x, times |x|
            double s0 = 0, s1 = 0, s2 = 0, s3 = 0;
            for (int t = 0; t < P.npts; ++t) {
                T xa[3];
                const T al = alphas[t];
                for (int d = 0; d < P.ndim; ++d) xa[d] = x[d] * al;
                eval_point_grad<T>(P, u, xa, &ds, de);
                s0 += ds; s1 += de[0]; s2 += de[1]; s3 += de[2];
            }
            const double f = g * xnorm / (double)P.npts;
            acc[0] += f * s0; acc[1] += f * s1; acc[2] += f * s2; acc[3] += f * s3;
        }
    }
    for (int c = 0; c < 4; ++c) {
        const double t = block_sum_256<T>(acc[c]);
        if (threadIdx.x == 0) partial[((size_t)b * gridDim.x + blockIdx.x) * 4 + c] = t;
    }
}

// Backward of doubly_diag_kernel for a scalar ell: out_b = ell^2 sig2 iv_b with iv_b = knn[i] + slopes[i] (dist_b - dgrid[i]) and
// dist_b = |x_b| / ell, so d out_b / d sig2 = ell^2 iv_b and d out_b / d ell = sig2 ell (2 iv_b - slopes[i] dist_b).
// grid ceil(B / 256), block 256: partial[blockIdx.x * 2 + {0, 1}] = this block's sums of g_b * {d/dsig2, d/dell}.
template <class T>
__global__ void __launch_bounds__(256) doubly_diag_grad_kernel(const T* __restrict__ xb, long B, int ndim, double sig2, double ell0,
                                                               const T* __restrict__ dgrid, const T* __restrict__ slopes,
                                                               const T* __restrict__ knn, int ntab, const T* __restrict__ g,
                                                               double* __restrict__ partial) {
    const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
    double ds = 0, de = 0;
    if (b < B) {
        const T ell[3] = {(T)ell0, (T)ell0, (T)ell0};
        T dist;
        const int li = doubly_diag_lookup<T>(xb, b, ndim, ell, dgrid, ntab, &dist);
        const double sl = (double)slopes[li];
        const double iv = (double)knn[li] + sl * ((double)dist - (double)dgrid[li]);
        const double gb = (double)g[b];
        ds = gb * ell0 * ell0 * iv;
        de = gb * sig2 * ell0 * (2.0 * iv - sl * (double)dist);
    }
    ds = block_sum_256<T>(ds);
    de = block_sum_256<T>(de);
    if (threadIdx.x == 0) { partial[(size_t)blockIdx.x * 2] = ds; partial[(size_t)blockIdx.x * 2 + 1] = de; }
}

// grid (nchunk, B), block 256; op 0: dot(a,b) | op 1: x += al p, r -= al Ap, dot(r,r) | op 2: p = z + be p
// (done: optional PCG early-exit flag, as in the fused passes)
template <class T>
__global__ void __launch_bounds__(256) vec_kernel(int op, T* x, T* r, const T* a, const T* b2, const double* s_num, const double* s_den,
                                                  double* partial, long M, int nchunk, const int* done) {
    if (done && *done) return;
    const long bb = blockIdx.y;
    const long per = (M + nchunk - 1) / nchunk;
    const long lo = (long)blockIdx.x * per, hi = lo + per < M ? lo + per : M;
    const size_t off = (size_t)bb * M;
    T coef = 0;
    if (op != 0) coef = (T)(s_num[bb] / s_den[bb]);
    double acc = 0;
    for (long i = lo + threadIdx.x; i < hi; i += 256) {
        if (op == 0) { acc += (double)(a[off + i] * b2[off + i]); }
        else if (op == 1) {
            x[off + i] = x[off + i] + coef * a[off + i];
            const T rv = r[off + i] - coef * b2[off + i];
            r[off + i] = rv; acc += (double)(rv * rv);
        } else { x[off + i] = a[off + i] + coef * x[off + i]; }
    }
    if (op != 2) {
        const double t = block_sum_256<T>(acc);
        if (threadIdx.x == 0) partial[bb * nchunk + blockIdx.x] = t;
    }
}
// ---- mean-field natural-gradient reductions over k_n (B x E) ------------------------------------------
// grid (nchunk, B), block 256: partial[(b*3 + t)*nchunk + chunk]
template <class T>
__global__ void __launch_bounds__(256) mf_rowstats_kernel(const T* __restrict__ kn, const T* __restrict__ qm, const T* __restrict__ qS,
                                                          double* partial, long E, int nchunk) {
    const long bb = blockIdx.y;
    const long per = (E + nchunk - 1) / nchunk;
    const long lo = (long)blockIdx.x * per, hi = lo + per < E ? lo + per : E;
    const T* row = kn + (size_t)bb * E;
    double a0 = 0, a1 = 0, a2 = 0;
    for (long j = lo + threadIdx.x; j < hi; j += 256) {
        const T k = row[j];
        a0 += (double)(k * qm[j]); a1 += (double)(k * k); a2 += (double)(k * k * qS[j]);
    }
    a0 = block_sum_256<T>(a0); a1 = block_sum_256<T>(a1); a2 = block_sum_256<T>(a2);
    if (threadIdx.x == 0) {
        partial[(bb * 3 + 0) * nchunk + blockIdx.x] = a0;
        partial[(bb * 3 + 1) * nchunk + blockIdx.x] = a1;
        partial[(bb * 3 + 2) * nchunk + blockIdx.x] = a2;
    }
}
template <class T>
__global__ void mf_rowstats_reduce_kernel(const double* partial, T* out, int nchunk, long B) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;   // over 3*B
    if (i >= 3 * B) return;
    const long bb = i / 3, t = i - bb * 3;
    double s = 0;
    for (int c = 0; c < nchunk; ++c) s += partial[i * nchunk + c];
    out[t * B + bb] = (T)s;
}
// thread per column j, coalesced across j; loops over the B rows
template <class T>
__global__ void __launch_bounds__(256) mf_colstats_kernel(const T* __restrict__ kn, const T* __restrict__ w1, const T* __restrict__ w2,
                                                          T* __restrict__ dm, T* __restrict__ lam, long B, long E) {
    const long j = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= E) return;
    T a = 0, l = 0;
    for (long b = 0; b < B; ++b) {
        const T k = kn[(size_t)b * E + j];
        a += w1[b] * k; l += w2[b] * k * k;
    }
    dm[j] = a; lam[j] = l;
}

__global__ void vec_reduce_kernel(const double* partial, double* out, int nchunk, long B, const int* done) {
    if (done && *done) return;
    const long bb = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (bb >= B) return;
    double t = 0;
    for (int i = 0; i < nchunk; ++i) t += partial[bb * nchunk + i];
    out[bb] = t;
}

}  // namespace hipgp
