// setup_kernels.cuh -- spectrum set-up (runs once per plan / per kernel-hyperparameter change).
//
// The reference builds D = max(Re FFT_N(embed(column)), 1e-6) with N_d = 2 m_d - 2
// (ziggy/misc/toeplitz_tensor.py:19-33).  The embedded first row is the even extension of the column, so
// Re FFT_N is exactly the separable DCT-I of the (m_1..m_D) column and D is even per axis.  Hence every
// operator the reference applies -- C' = F^-1 D F, C'^-1, C'^(1/2) -- is a block-circulant whose first
// column is again a DCT-I of an (m_1..m_D) array.  Set-up therefore is:  DCT-I -> clamp -> {id, 1/x, sqrt}
// -> DCT-I (first columns c', g, s), all in fp64, followed by a forward FFT of the re-embedded columns at a
// smooth length L_d (done with the matvec's own forward passes, so the spectra come out in the pipeline's
// digit-reversed layout).
#pragma once
#include "fft_engine.cuh"

namespace hipgp {

// out[o][k][i] = sum_j w_j in[o][j][i] cos(pi j k / (m-1)),  w_0 = w_{m-1} = 1, else 2.   (DCT-I, unnormalised;
// applying it twice multiplies by N = 2(m-1)).  costab[t] = cos(pi t / (m-1)), t in [0, 2(m-1)).
// It is the one genuine matrix product of the path -- (m x m cosine matrix) x (m x inner) per outer index -- so it runs as a
// TILED fp64 contraction (a one-output-per-thread kernel spent 1.13 ms per launch at config 2, 8 launches per spectrum
// set-up).  64 x 64 output tile per CTA, 16-deep k tiles in shared memory,
// 16 x 16 threads with 4 x 4 fp64 accumulators each; the cosine operand is generated from the length-N table (index
// (j k) mod N) while its tile is staged, so no m x m matrix is stored (axes longer than 2048 points; shorter axes take
// dct1_sym_kernel below).
//   LAST == false: out[o][k][i] = scale * sum_j w_j cos(pi j k / (m-1)) in[o][j][i]      (tile rows = k, tile columns = i)
//   LAST == true : inner == 1:  out[o][k]   = scale * sum_j in[o][j] w_j cos(pi j k / (m-1))  (tile rows = o, tile columns = k)
template <bool LAST>
__global__ void __launch_bounds__(256) dct1_tile_kernel(const double* __restrict__ in, double* __restrict__ out,
                                                        const double* __restrict__ costab, int m, long inner, long outer, double scale) {
    constexpr int RM = 8;                   // rows per thread: 8 x 4 outputs per thread, 12 shared-memory loads per 32 DFMA
    constexpr int TM = 16 * RM, TN = 64, TK = 16;
    __shared__ double As[TK][TM + 2];      // As[jj][row]
    __shared__ double Bs[TK][TN + 2];      // Bs[jj][col]
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const int N = m > 1 ? 2 * (m - 1) : 1;
    const long r0 = (long)blockIdx.y * TM, c0 = (long)blockIdx.x * TN;
    const long o = LAST ? 0 : (long)blockIdx.z;
    const long nrows = LAST ? outer : m, ncols = LAST ? m : inner;
    const double* inb = in + (LAST ? 0 : (size_t)o * m * inner);
    double acc[RM][4];
#pragma unroll
    for (int a = 0; a < RM; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
    for (int j0 = 0; j0 < m; j0 += TK) {
        // stage the two operand tiles
        for (int e = threadIdx.x; e < TK * TM; e += 256) {
            if (LAST) {          // A(row = o, j) = in[o][j]: consecutive threads walk j (contiguous)
                const int jj = e % TK, rr = e / TK;
                const long row = r0 + rr; const int j = j0 + jj;
                As[jj][rr] = (row < nrows && j < m) ? inb[(size_t)row * m + j] : 0.0;
            } else {             // A(row = k, j) = w_j cos(pi j k / (m-1))
                const int rr = e % TM, jj = e / TM;
                const long k = r0 + rr; const int j = j0 + jj;
                double v = 0.0;
                if (k < nrows && j < m) { const double w = (j == 0 || j == m - 1) ? 1.0 : 2.0; v = m > 1 ? w * costab[((unsigned)j * (unsigned)k) % (unsigned)N] : 1.0; }
                As[jj][rr] = v;
            }
        }
        for (int e = threadIdx.x; e < TK * TN; e += 256) {
            const int cc = e % TN, jj = e / TN;
            const long col = c0 + cc; const int j = j0 + jj;
            double v = 0.0;
            if (col < ncols && j < m) {
                if (LAST) { const double w = (j == 0 || j == m - 1) ? 1.0 : 2.0; v = m > 1 ? w * costab[((unsigned)j * (unsigned)col) % (unsigned)N] : 1.0; }
                else v = inb[(size_t)j * inner + col];
            }
            Bs[jj][cc] = v;
        }
        __syncthreads();
#pragma unroll
        for (int jj = 0; jj < TK; ++jj) {
            double a[RM], b[4];
#pragma unroll
            for (int t = 0; t < RM; ++t) a[t] = As[jj][ty * RM + t];
#pragma unroll
            for (int t = 0; t < 4; ++t) b[t] = Bs[jj][tx * 4 + t];
#pragma unroll
            for (int x = 0; x < RM; ++x)
#pragma unroll
                for (int y = 0; y < 4; ++y) acc[x][y] += a[x] * b[y];
        }
        __syncthreads();
    }
    double* outb = out + (LAST ? 0 : (size_t)o * m * inner);
#pragma unroll
    for (int x = 0; x < RM; ++x) {
        const long row = r0 + ty * RM + x;
        if (row >= nrows) continue;
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            const long col = c0 + tx * 4 + y;
            if (col < ncols) outb[(size_t)row * (LAST ? m : inner) + col] = acc[x][y] * scale;
        }
    }
}

// ---- DCT-I with the reflection symmetry of the cosine matrix folded in: HALF the multiply-adds -------------------------
// w_j cos(pi (m-1-j) k / (m-1)) = (-1)^k w_j cos(pi j k / (m-1)), so with hj = ceil(m / 2) folded inputs
//   out[2k'+p] = sum_{j < hj} Cw[j][2k'+p] (x[j] + (-1)^p x[m-1-j])          (the unpaired middle input of an odd m counts once)
// i.e. two products of half the size, one per output parity p.  The parity-split matrix Cw2[p][j][k'] = Cw[j][2k'+p] (row pitch
// hk0 = ceil(m / 2)) is cached per axis; the fold happens while the input tile is staged.  Same tile shape as dct1_tile_kernel.
__global__ void dct1_cosmat_sym_kernel(const double* __restrict__ costab, double* __restrict__ cw2, int m) {
    const unsigned N = m > 1 ? 2u * (unsigned)(m - 1) : 1u;
    const int hj = (m + 1) / 2, hk0 = (m + 1) / 2;
    const long total = 2L * hj * hk0;
    for (long i = (long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long)gridDim.x * blockDim.x) {
        const int kp = (int)(i % hk0), j = (int)((i / hk0) % hj), p = (int)(i / ((long)hk0 * hj));
        const int k = 2 * kp + p;
        const double w = (j == 0 || j == m - 1) ? 1.0 : 2.0;
        cw2[i] = (k < m && m > 1) ? w * costab[((unsigned)j * (unsigned)k) % N] : (m > 1 ? 0.0 : 1.0);
    }
}
template <bool LAST>
__global__ void __launch_bounds__(256) dct1_sym_kernel(const double* __restrict__ in, double* __restrict__ out, const double* __restrict__ cw2,
                                                       int m, long inner, long outer, double scale, int nty) {
    constexpr int RM = 8;
    constexpr int TM = 16 * RM, TN = 64, TK = 16;
    __shared__ double As[TK][TM + 2];
    __shared__ double Bs[TK][TN + 2];
    const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
    const int hj = (m + 1) / 2, hk0 = (m + 1) / 2;
    // parity and tile coordinates:  !LAST: grid (inner tiles, 2 * nty, outer);  LAST: grid (k' tiles, outer tiles, 2)
    const int p = LAST ? (int)blockIdx.z : (int)(blockIdx.y / nty);
    const long r0 = (LAST ? (long)blockIdx.y : (long)(blockIdx.y - p * nty)) * TM, c0 = (long)blockIdx.x * TN;
    const int hk = (m - p + 1) / 2;                             // outputs of this parity
    const long o = LAST ? 0 : (long)blockIdx.z;
    const long nrows = LAST ? outer : hk, ncols = LAST ? hk : inner;
    const double* inb = in + (LAST ? 0 : (size_t)o * m * inner);
    const double* cwp = cw2 + (size_t)p * hj * hk0;
    const double sgn = p ? -1.0 : 1.0;
    double acc[RM][4];
#pragma unroll
    for (int a = 0; a < RM; ++a)
#pragma unroll
        for (int b = 0; b < 4; ++b) acc[a][b] = 0.0;
    for (int j0 = 0; j0 < hj; j0 += TK) {
        for (int e = threadIdx.x; e < TK * TM; e += 256) {
            if (LAST) {          // A(row = o, j) = in[o][j] +- in[o][m-1-j]
                const int jj = e % TK, rr = e / TK;
                const long row = r0 + rr; const int j = j0 + jj;
                double v = 0.0;
                if (row < nrows && j < hj) {
                    const int jm = m - 1 - j;
                    v = inb[(size_t)row * m + j];
                    v = jm == j ? (p ? 0.0 : v) : v + sgn * inb[(size_t)row * m + jm];
                }
                As[jj][rr] = v;
            } else {             // A(row = k', j) = Cw2[p][j][k']
                const int rr = e % TM, jj = e / TM;
                const long k = r0 + rr; const int j = j0 + jj;
                As[jj][rr] = (k < nrows && j < hj) ? cwp[(size_t)j * hk0 + k] : 0.0;
            }
        }
        for (int e = threadIdx.x; e < TK * TN; e += 256) {
            const int cc = e % TN, jj = e / TN;
            const long col = c0 + cc; const int j = j0 + jj;
            double v = 0.0;
            if (col < ncols && j < hj) {
                if (LAST) v = cwp[(size_t)j * hk0 + col];
                else {
                    const int jm = m - 1 - j;
                    v = inb[(size_t)j * inner + col];
                    v = jm == j ? (p ? 0.0 : v) : v + sgn * inb[(size_t)jm * inner + col];
                }
            }
            Bs[jj][cc] = v;
        }
        __syncthreads();
#pragma unroll
        for (int jj = 0; jj < TK; ++jj) {
            double a[RM], b[4];
#pragma unroll
            for (int t = 0; t < RM; ++t) a[t] = As[jj][ty * RM + t];
#pragma unroll
            for (int t = 0; t < 4; ++t) b[t] = Bs[jj][tx * 4 + t];
#pragma unroll
            for (int x = 0; x < RM; ++x)
#pragma unroll
                for (int y = 0; y < 4; ++y) acc[x][y] += a[x] * b[y];
        }
        __syncthreads();
    }
    double* outb = out + (LAST ? 0 : (size_t)o * m * inner);
#pragma unroll
    for (int x = 0; x < RM; ++x) {
        const long row = r0 + ty * RM + x;
        if (row >= nrows) continue;
#pragma unroll
        for (int y = 0; y < 4; ++y) {
            const long col = c0 + tx * 4 + y;
            if (col >= ncols) continue;
            if (LAST) outb[(size_t)row * m + (2 * col + p)] = acc[x][y] * scale;
            else outb[(size_t)(2 * row + p) * inner + col] = acc[x][y] * scale;
        }
    }
}

template <class T>
__global__ void to_double_kernel(const T* __restrict__ in, double* __restrict__ out, long n) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (double)in[i];
}

// D (fp64 DCT output) -> rounded to the plan dtype, clamped (toeplitz_tensor.py:26), then the three
// derived spectra in fp64.  counts[0] += number of clamped entries.
template <class T>
__global__ void clamp_derive_kernel(const double* __restrict__ Draw, double* __restrict__ D, double* __restrict__ Dinv,
                                    double* __restrict__ Dsqrt, long n, double clampv, unsigned* counts) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    T d = (T)Draw[i];
    if (d < (T)clampv) { d = (T)clampv; atomicAdd(counts, 1u); }
    const double dd = (double)d;
    D[i] = dd; Dinv[i] = 1.0 / dd; Dsqrt[i] = sqrt(dd);
}

struct EmbedDims {
    int D;
    int m[3];      // column extents
    int N[3];      // 2m-2 (1 if m == 1)
    int L[3];      // embedding length
    int wide[3];   // 0: Toeplitz-block embedding (K, Cinv)  1: full-circulant-output embedding (RT / R)
};

__host__ __device__ __forceinline__ int embed_index(int i, int m, int N, int L, int wide) {
    // returns the column index in [0,m) feeding embedded position i, or -1 for the zero gap
    if (!wide) {
        if (i < m) return i;
        if (i > L - m) return L - i;
        return -1;
    }
    if (wide == 2) {
        // SYMMETRIC wide embedding (needs L >= 2N - 1): taps s[lag mod N] for every lag in (-N, N).  The rectangular product
        // R^T v (outputs [0, N), inputs [0, m)) only reads lags in [-(m-1), N-1]; the mirrored taps at lags (-N, -m] land on
        // circular positions that no (output, input) pair reaches, and they make the tap sequence even, i.e. the spectrum REAL.
        const int lag = i < N ? i : (i > L - N ? L - i : -1);
        if (lag < 0) return -1;
        return lag < m ? lag : N - lag;
    }
    if (i < N) return i < m ? i : N - i;
    if (i > L - m) return L - i;
    return -1;
}

// h[i1][i2][i3] (real, extents L) from col[(m1,m2,m3)]
__global__ void embed_kernel(const double* __restrict__ col, double* __restrict__ h, EmbedDims e) {
    const long total = (long)e.L[0] * e.L[1] * e.L[2];
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int i3 = (int)(idx % e.L[2]);
        const int i2 = (int)((idx / e.L[2]) % e.L[1]);
        const int i1 = (int)(idx / ((long)e.L[2] * e.L[1]));
        const int j1 = embed_index(i1, e.m[0], e.N[0], e.L[0], e.wide[0]);
        const int j2 = embed_index(i2, e.m[1], e.N[1], e.L[1], e.wide[1]);
        const int j3 = embed_index(i3, e.m[2], e.N[2], e.L[2], e.wide[2]);
        double v = 0.0;
        if (j1 >= 0 && j2 >= 0 && j3 >= 0) v = col[((size_t)j1 * e.m[1] + j2) * e.m[2] + j3];
        h[idx] = v;
    }
}

// raw forward-pipeline output (fp64 complex) -> stored spectrum in the plan dtype, scaled.
template <class T>
__global__ void store_spec_real_kernel(const cplx<double>* __restrict__ raw, T* __restrict__ out, long n, double scale) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (T)(raw[i].x * scale);
}
template <class T>
__global__ void store_spec_cplx_kernel(const cplx<double>* __restrict__ raw, cplx<T>* __restrict__ out, long n, double scale) {
    const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = mk<T>((T)(raw[i].x * scale), (T)(raw[i].y * scale));
}

// D-shaped (m_1..m_D) fp64 -> reference layout (N_1..N_D) in the plan dtype (even extension), for the
// `D`, `D_sqrt`, `Di` attributes of the drop-in ToeplitzTensor.
template <class T>
__global__ void expand_even_kernel(const double* __restrict__ Dm, T* __restrict__ out, EmbedDims e, int op) {
    const long total = (long)e.N[0] * e.N[1] * e.N[2];
    for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
        const int i3 = (int)(idx % e.N[2]);
        const int i2 = (int)((idx / e.N[2]) % e.N[1]);
        const int i1 = (int)(idx / ((long)e.N[2] * e.N[1]));
        const int j1 = i1 < e.m[0] ? i1 : e.N[0] - i1;
        const int j2 = i2 < e.m[1] ? i2 : e.N[1] - i2;
        const int j3 = i3 < e.m[2] ? i3 : e.N[2] - i3;
        const double d = Dm[((size_t)j1 * e.m[1] + j2) * e.m[2] + j3];
        T v = (T)d;
        if (op == 1) v = (T)sqrt((double)v);            // D_sqrt = sqrt(D)      (toeplitz_tensor.py:29)
        else if (op == 2) v = (T)1 / v;                 // Di = 1 / D            (toeplitz_tensor.py:30)
        else if (op == 3) v = (T)sqrt((double)((T)1 / v));   // Di_sqrt = sqrt(Di)    (toeplitz_tensor.py:33)
        out[idx] = v;
    }
}

}  // namespace hipgp
