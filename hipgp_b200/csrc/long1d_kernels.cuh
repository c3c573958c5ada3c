// long1d_kernels.cuh -- four-step FFT convolution along a last grid axis too long for the one-block row pass (1-D grids,
// and the last axis of 2-D / 3-D grids).
//
// The last axis' embedding length factors as L = L1 * L2 and a sample index as n = L2 * n1 + n2 (n2 contiguous).  Data of
// one packed pair of right-hand sides (x_a + i x_b) along one row of the leading axes is a complex [L1][L2] array in the
// workspace W[pair][row][L1][L2].  A pass runs on `nrows` rows per pair, CTA line index = pair * nrows + row (a 1-D grid
// has one row).  Its input / output rows are the right-hand sides' [row][n] arrays, partner b one vector (nrows * n
// values) after partner a.  A transform of the last axis is made of three passes:
//   cols_fwd : strided L1-point DIF over n1 of the zero-padded input (only the first ceil(n_in / L2) rows are loaded), then
//              the twiddle W_L^(n2 k1) on the way out.  Row p of the workspace holds k1 = rev1(p).
//   rows     : contiguous L2-point lines: DIF (LR_FWD), DIF times the spectrum then DIT back (LR_CONV, the middle of a 1-D
//              convolution), or DIT alone (LR_INV, after the column passes of a 2-D / 3-D grid).  The spectrum is stored
//              [p1][p2] in the same digit-reversed order, because set-up builds it with these passes.
//   cols_inv : conjugate twiddle, strided L1-point DIT back to n1, crop to n_out, unpack into the two real output rows.
// Every operator is a circular convolution with a real first column: K and C^-1 have real spectra, R^T a real or Hermitian
// one and R its conjugate, so the real and imaginary parts of a packed pair never mix.
#pragma once
#include "conv_kernels.cuh"

namespace hipgp {

enum LongRowsMode { LR_FWD = 0, LR_CONV = 1, LR_INV = 2 };

template <class T>
struct LongParams {
    const T* in;              // cols_fwd: B vectors of nrows real rows of n_in samples
    T* out;                   // cols_inv: B vectors of nrows real rows of n_out samples
    cplx<T>* W;               // [pair][W_rows][L1][L2]
    long B, n_in, n_out;
    int nrows;                // rows per pair this pass runs on: grid.x = ntiles * pairs * nrows (< 2^31)
    long W_rows;              // rows per pair in W (>= nrows)
    int L1, L2;
    LineFft<T> f1, f2;        // L1-point (strided) and L2-point (contiguous) line FFTs
    const cplx<T>* twh;       // W_L1^j, j < L1     (W_L^(n2 k1) = twh[j / L2] * twl[j % L2], j = n2 k1 < L)
    const cplx<T>* twl;       // W_L^j,  j < L2
    int TB, TBP;              // lines per CTA and padded line count (shared-memory line stride)
    int ntiles;               // CTAs per line
    int rows_mode;            // rows: LongRowsMode
    const void* spec; int spec_kind;   // rows, LR_CONV
    const int* done_flag;     // optional PCG early-exit flag
};

template <class T>
__device__ __forceinline__ cplx<T> long_twiddle(const LongParams<T>& P, long n2, int k1) {
    const long j = n2 * (long)k1;                          // < L1 L2: no reduction needed
    return ldg_c(P.twh + j / P.L2) * ldg_c(P.twl + j % P.L2);
}

template <class T>
__global__ void __launch_bounds__(256) long_cols_fwd_kernel(LongParams<T> P) {
    HIPGP_DYN_SMEM(smem_raw);
    cplx<T>* s = reinterpret_cast<cplx<T>*>(smem_raw);
    const int tid = threadIdx.x, nthreads = blockDim.x;
    if (P.done_flag && *P.done_flag) return;
    const int line = blockIdx.x / P.ntiles, pair = line / P.nrows, row = line % P.nrows;
    const long c0 = (long)(blockIdx.x % P.ntiles) * P.TB;
    const int L1 = P.L1, TB = P.TB, TBP = P.TBP;
    const long rows_nz = (P.n_in + P.L2 - 1) / P.L2;
    const long vec = (long)P.nrows * P.n_in;
    const T* ina = P.in + (size_t)(2 * pair) * vec + (size_t)row * P.n_in;
    const bool has_b = 2 * pair + 1 < P.B;
    for (int w = tid; w < L1 * TB; w += nthreads) {
        const int c = w % TB, i = w / TB;
        const long n = (long)i * P.L2 + c0 + c;
        cplx<T> v = mk<T>(0, 0);
        if (i < rows_nz && c0 + c < P.L2 && n < P.n_in) v = mk<T>(ina[n], has_b ? ina[vec + n] : (T)0);
        s[(size_t)i * TBP + c] = v;
    }
    __syncthreads();
    fft_forward(s, TBP, TB, P.f1, tid, nthreads);
    cplx<T>* W = P.W + ((size_t)pair * P.W_rows + row) * L1 * P.L2 + c0;
    for (int w = tid; w < L1 * TB; w += nthreads) {
        const int c = w % TB, p = w / TB;
        if (c0 + c < P.L2) W[(size_t)p * P.L2 + c] = s[(size_t)p * TBP + c] * long_twiddle(P, c0 + c, P.f1.rev[p]);
    }
}

template <class T>
__global__ void __launch_bounds__(256) long_rows_kernel(LongParams<T> P) {
    HIPGP_DYN_SMEM(smem_raw);
    cplx<T>* s = reinterpret_cast<cplx<T>*>(smem_raw);
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
    if (P.done_flag && *P.done_flag) return;
    const int wline = blockIdx.x / P.ntiles, pair = wline / P.nrows, row = wline % P.nrows;
    const int r0 = (blockIdx.x % P.ntiles) * P.TB;
    const int L2 = P.L2, TB = P.TB, TBP = P.TBP;
    const int nl = P.L1 - r0 < TB ? P.L1 - r0 : TB;
    cplx<T>* W = P.W + (((size_t)pair * P.W_rows + row) * P.L1 + r0) * L2;
    for (int line = warp; line < TB; line += nwarps)
        for (int q = lane; q < L2; q += 32) s[(size_t)q * TBP + line] = line < nl ? W[(size_t)line * L2 + q] : mk<T>(0, 0);
    __syncthreads();
    if (P.rows_mode != LR_INV) fft_forward(s, TBP, TB, P.f2, tid, nthreads);
    if (P.rows_mode == LR_CONV) {
        for (int w = tid; w < L2 * TB; w += nthreads) {
            const int line = w % TB, q = w / TB;
            if (line < nl) s[(size_t)q * TBP + line] = apply_spec(s[(size_t)q * TBP + line], P.spec, P.spec_kind, (size_t)(r0 + line) * L2 + q);
        }
        __syncthreads();
    }
    if (P.rows_mode != LR_FWD) fft_inverse(s, TBP, TB, P.f2, tid, nthreads);
    for (int line = warp; line < nl; line += nwarps)
        for (int q = lane; q < L2; q += 32) W[(size_t)line * L2 + q] = s[(size_t)q * TBP + line];
}

template <class T>
__global__ void __launch_bounds__(256) long_cols_inv_kernel(LongParams<T> P) {
    HIPGP_DYN_SMEM(smem_raw);
    cplx<T>* s = reinterpret_cast<cplx<T>*>(smem_raw);
    const int tid = threadIdx.x, nthreads = blockDim.x;
    if (P.done_flag && *P.done_flag) return;
    const int line = blockIdx.x / P.ntiles, pair = line / P.nrows, row = line % P.nrows;
    const long c0 = (long)(blockIdx.x % P.ntiles) * P.TB;
    const int L1 = P.L1, TB = P.TB, TBP = P.TBP;
    const cplx<T>* W = P.W + ((size_t)pair * P.W_rows + row) * L1 * P.L2 + c0;
    for (int w = tid; w < L1 * TB; w += nthreads) {
        const int c = w % TB, p = w / TB;
        cplx<T> v = mk<T>(0, 0);
        if (c0 + c < P.L2) v = mulc(W[(size_t)p * P.L2 + c], long_twiddle(P, c0 + c, P.f1.rev[p]));
        s[(size_t)p * TBP + c] = v;
    }
    __syncthreads();
    fft_inverse(s, TBP, TB, P.f1, tid, nthreads);
    const long rows_out = (P.n_out + P.L2 - 1) / P.L2;
    const long vec = (long)P.nrows * P.n_out;
    T* outa = P.out + (size_t)(2 * pair) * vec + (size_t)row * P.n_out;
    const bool has_b = 2 * pair + 1 < P.B;
    for (int w = tid; w < (int)(rows_out < L1 ? rows_out : L1) * TB; w += nthreads) {
        const int c = w % TB, i = w / TB;
        const long n = (long)i * P.L2 + c0 + c;
        if (c0 + c < P.L2 && n < P.n_out) {
            const cplx<T> v = s[(size_t)i * TBP + c];
            outa[n] = v.x;
            if (has_b) outa[vec + n] = v.y;
        }
    }
}

// ---- Bluestein DCT-I of length m (set-up of long 1-D plans, fp64) -------------------------------------------------
// DCT-I(c)[k] = Re FFT_N(x)[k], x the even extension of c (N = 2m - 2), and FFT_N(x)[k] = w_k sum_n (x_n w_n) conj(w_{k-n})
// with the chirp w_n = exp(-i pi n^2 / N): a circular convolution of length Lb >= 2N - 1 on the four-step passes.  Chirp
// angles use the exact reduction n^2 mod 2N in 64-bit integers.
__device__ __forceinline__ void chirp(long n, long N, double* c, double* s) {
    const long r = (long)(((unsigned long long)n * (unsigned long long)n) % (unsigned long long)(2 * N));
    sincospi((double)r / (double)N, s, c);          // exp(-i pi r / N) = c - i s
}

// b[2][Lb] planar: b_j = conj(w_j) at circular lags j in (-N, N), 0 elsewhere
__global__ void blu_chirp_kernel(double* __restrict__ b, long N, long Lb) {
    for (long j = (long)blockIdx.x * blockDim.x + threadIdx.x; j < Lb; j += (long)gridDim.x * blockDim.x) {
        const long lag = j < N ? j : (j > Lb - N ? Lb - j : -1);
        double c = 0, s = 0;
        if (lag >= 0) chirp(lag, N, &c, &s);
        b[j] = c; b[Lb + j] = s;
    }
}

// a[2][N] planar: a_n = x_n w_n, x the even extension of in[m]
__global__ void blu_premul_kernel(const double* __restrict__ in, double* __restrict__ a, long m, long N) {
    for (long n = (long)blockIdx.x * blockDim.x + threadIdx.x; n < N; n += (long)gridDim.x * blockDim.x) {
        const double x = in[n < m ? n : N - n];
        double c, s;
        chirp(n, N, &c, &s);
        a[n] = x * c; a[N + n] = -x * s;
    }
}

// out[k] = scale Re(w_k (y_re + i y_im)[k]), k < m
__global__ void blu_post_kernel(const double* __restrict__ y, double* __restrict__ out, long m, long N, double scale) {
    for (long k = (long)blockIdx.x * blockDim.x + threadIdx.x; k < m; k += (long)gridDim.x * blockDim.x) {
        double c, s;
        chirp(k, N, &c, &s);
        out[k] = scale * (c * y[k] + s * y[m + k]);
    }
}

// the stop test of the fused passes (pcg_finalize, DOT_RR) for solves whose updates run as separate vector kernels
__global__ void long_pcg_stop_kernel(PcgDev st) {
    if (threadIdx.x == 0 && blockIdx.x == 0 && !st.flags[0]) pcg_stop_test(st);
}

}  // namespace hipgp
