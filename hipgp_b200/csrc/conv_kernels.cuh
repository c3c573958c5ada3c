// conv_kernels.cuh -- the pruned FFT-convolution passes of the structured matvec.
//
//   rows_fwd : last grid axis.  real rows (n_in samples, implicit zero pad to L) -> half spectrum
//              (H = L/2 complex FFT + in-place split), written in digit-reversed order, H+1 entries/row.
//              Optional fused PCG vector update on load (p = z + beta p | x += a p, r -= a Ap, r.r).
//   cols_pass: any other axis, strided lines, TB neighbouring lines per CTA.
//              FWD (pad + DIF) | INV (DIT + crop) | FUSED (pad + DIF, x spectrum, DIT + crop).
//   rows_inv : merge + H-point DIT + crop, real rows out.  Optional spectrum multiply on load (1-D
//              grids have no cols pass) and fused dot product of the output with a second vector.
//
// Frequency data layout: W[batch][i_1]...[i_{D-1}][q], q in [0,H]; q < H holds frequency rev(q) of the
// last axis, q == H holds the Nyquist term.  All other axes are in DIF position order after their pass.
#pragma once
#include "fft_engine.cuh"

namespace hipgp {

enum RowsFwdMode { RF_PLAIN = 0, RF_PUPDATE = 1, RF_XRUPDATE = 2, RF_SELFDOT = 3 };
enum RowsInvMode { RI_PLAIN = 0, RI_DOT = 1 };
enum DotKind { DOT_PAP = 0, DOT_ZR = 1, DOT_RR = 2 };
enum ColsMode { CM_FWD = 0, CM_INV = 1, CM_FUSED = 2 };
enum SpecKind { SPEC_NONE = 0, SPEC_REAL = 1, SPEC_CPLX = 2, SPEC_CPLX_CONJ = 3 };

// Device-resident PCG scalars (all fp64; one entry per right-hand side).
struct PcgDev {
    double* zr;        // r.z of the current iterate
    double* zr_prev;   // r.z of the previous iterate
    double* pAp;
    double* rr;
    const double* rr_all;   // all B residual norms when `rr` points into a group of right-hand sides (nullptr: rr itself)
    double* partial;   // one slot per global row
    unsigned* row_cnt; // [B] rows finished for this rhs (self-resetting)
    unsigned* rhs_cnt; // [1] rhs finished (self-resetting)
    int* flags;        // [0] done, [1] iterations executed (x/r updates), [2] first-iteration marker
    double tol;
    int B;
    int cg_mode;       // no preconditioner: z aliases r, so r.r also serves as r.z
};

template <class T> __device__ __forceinline__ T warp_sum(T v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// The stopping rule all_b sqrt(r_b.r_b) < tol (cg.py:70), run by one thread once r.r of every right-hand side is in.
__device__ __forceinline__ void pcg_stop_test(const PcgDev& st) {
    bool all = true;
    const volatile double* rr = st.rr_all ? st.rr_all : st.rr;
    for (int i = 0; i < st.B; ++i) all = all && (sqrt(rr[i]) < st.tol);
    st.flags[1] += 1;
    st.flags[2] = 0;
    if (all) st.flags[0] = 1;
}

// Deterministic finalisation: called by every thread of the CTA after it has written the per-row partials
// of rows [g0, g1).  The CTA that completes a right-hand side sums that rhs's partials in a fixed order.
__device__ __forceinline__ void pcg_finalize(const PcgDev& st, int kind, long g0, long g1, int nrows, int tid, int nthreads) {
    __shared__ unsigned s_last;
    __shared__ double s_red[32];
    const int b0 = (int)(g0 / nrows), b1 = (int)((g1 - 1) / nrows);
    for (int b = b0; b <= b1; ++b) {
        const long lo = g0 > (long)b * nrows ? g0 : (long)b * nrows;
        const long hi = g1 < (long)(b + 1) * nrows ? g1 : (long)(b + 1) * nrows;
        __syncthreads();
        if (tid == 0) {
            __threadfence();
            const unsigned done = atomicAdd(st.row_cnt + b, (unsigned)(hi - lo)) + (unsigned)(hi - lo);
            s_last = (done == (unsigned)nrows);
        }
        __syncthreads();
        if (!s_last) continue;
        __threadfence();
        // fixed-order tree: thread t sums partial[t], partial[t+nthreads], ...; then warps; then warp 0
        double acc = 0.0;
        const volatile double* part = st.partial + (long)b * nrows;
        for (int i = tid; i < nrows; i += nthreads) acc += part[i];
        acc = warp_sum(acc);
        if ((tid & 31) == 0) s_red[tid >> 5] = acc;
        __syncthreads();
        if (tid < 32) {
            double v = tid < (nthreads >> 5) ? s_red[tid] : 0.0;
            v = warp_sum(v);
            if (tid == 0) {
                st.row_cnt[b] = 0;
                if (kind == DOT_PAP) st.pAp[b] = v;
                else if (kind == DOT_ZR) { st.zr_prev[b] = st.zr[b]; st.zr[b] = v; }
                else {
                    st.rr[b] = v;
                    if (st.cg_mode) { st.zr_prev[b] = st.zr[b]; st.zr[b] = v; }
                }
                __threadfence();
                if (kind == DOT_RR) {
                    const unsigned nb = atomicAdd(st.rhs_cnt, 1u) + 1u;
                    if (nb == (unsigned)st.B) {
                        __threadfence();
                        st.rhs_cnt[0] = 0;
                        pcg_stop_test(st);
                    }
                }
            }
        }
    }
}

// ------------------------------------------------------------------------------------------------
template <class T>
struct RowsParams {
    const T* in;          // RF_PLAIN: rows in; RF_PUPDATE: z; RF_XRUPDATE: Ap
    T* out;               // rows_inv output
    T* v0;                // RF_PUPDATE: p (rw); RF_XRUPDATE: r (rw); RI_DOT: other vector (ro)
    T* v1;                // RF_XRUPDATE: x (rw)
    const T* v2;          // RF_XRUPDATE: p (ro)
    cplx<T>* W;           // frequency data
    long total_rows;      // B * nrows
    int nrows;            // rows per right-hand side
    int n_real;           // samples per row in (fwd) / out (inv)
    int L, H;             // real length, H = L/2
    long W_pitch;         // complex entries per row (>= H+1)
    int W_rows;           // rows per rhs in W (>= nrows): W row of global row g is (g/nrows)*W_rows + g%nrows
    LineFft<T> f;         // H-point complex FFT
    const cplx<T>* twL;   // exp(-2 pi i k / L), k < H
    const cplx<T>* twLp;  // twL in position order: twLp[q] = twL[rev[q]]
    const int* part;      // partner position of q in the r2c split: pos[H - rev[q]] (q > 0)
    const int* pairq;     // the H/2 + 1 positions q with q <= part[q] (one per (k, H-k) pair), ascending
    // specialised kernels: (k, H-k) pairs as records {q, q2} + twLp[q], in pairq order (the first npair0 = digit group
    // 0, or all of them when the list has one stage), and quads {a, b} + (twLp[a], twLp[a+1]): even positions whose
    // bins (a, a+1) mirror onto (b+1, b), a <= b
    const int* pairs; const cplx<T>* pairw; int npair0;
    const int* quadq; const cplx<T>* quadw; int nquad;
    int RB, RBP;          // rows per CTA, padded smem line count
    int mode, dot_kind, do_fft;
    int vec_ok;           // all row pointers are aligned for 2-element vector access
    int vec16_ok;         // ... and for 16-byte access (specialised kernels stream rows in 16-byte chunks)
    int tma_op;           // specialised kernels move aligned row blocks with 1-D bulk-asynchronous (TMA) copies; 1 = so do the
                          // operands of a fused PCG update (they land in the idle tile buffer, which is big enough)
    const void* spec; int spec_kind;   // rows_inv only (1-D grids)
    PcgDev st;
};

template <class T>
__global__ void __launch_bounds__(256) rows_fwd_kernel(RowsParams<T> P) {
    HIPGP_DYN_SMEM(smem_raw);
    cplx<T>* s = reinterpret_cast<cplx<T>*>(smem_raw);
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
    if (P.mode != RF_PLAIN && P.st.flags[0]) return;
    const long g0 = (long)blockIdx.x * P.RB;
    const long g1 = g0 + P.RB < P.total_rows ? g0 + P.RB : P.total_rows;
    const int nl = (int)(g1 - g0);
    const int H = P.H, RBP = P.RBP, n = P.n_real;

    // ---- load (one warp per row), fused vector update, pack x[2k] + i x[2k+1] -------------------
    for (int line = warp; line < P.RB; line += nwarps) {
        if (line >= nl) {
            if (P.do_fft) for (int k = lane; k < H; k += 32) s[(size_t)k * RBP + line] = mk<T>(0, 0);
            continue;
        }
        const long g = g0 + line;
        const int b = (int)(g / P.nrows);
        const size_t off = (size_t)g * n;
        T acc = 0;
        T coef = 0;
        bool first = false;
        if (P.mode == RF_PUPDATE) {
            first = P.st.flags[2] != 0;
            coef = first ? (T)0 : (T)(P.st.zr[b] / P.st.zr_prev[b]);
        } else if (P.mode == RF_XRUPDATE) {
            coef = (T)(P.st.zr[b] / P.st.pAp[b]);
        }
        for (int k = lane; k < H; k += 32) {
            T e[2];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int i = 2 * k + h;
                T val = 0;
                if (i < n) {
                    if (P.mode == RF_PLAIN) {
                        val = P.in[off + i];
                    } else if (P.mode == RF_PUPDATE) {
                        const T z = P.in[off + i];
                        val = first ? z : z + coef * P.v0[off + i];
                        P.v0[off + i] = val;
                    } else if (P.mode == RF_SELFDOT) {
                        val = P.in[off + i];
                        acc += val * val;
                    } else {
                        const T pv = P.v2[off + i];
                        P.v1[off + i] = P.v1[off + i] + coef * pv;
                        val = P.v0[off + i] - coef * P.in[off + i];
                        P.v0[off + i] = val;
                        acc += val * val;
                    }
                }
                e[h] = val;
            }
            if (P.do_fft) s[(size_t)k * RBP + line] = mk<T>(e[0], e[1]);
        }
        if (P.mode == RF_XRUPDATE || P.mode == RF_SELFDOT) {
            const double tot = warp_sum((double)acc);
            if (lane == 0) P.st.partial[g] = tot;
        }
    }
    if (P.mode == RF_XRUPDATE) pcg_finalize(P.st, DOT_RR, g0, g1, P.nrows, tid, nthreads);
    if (P.mode == RF_SELFDOT) pcg_finalize(P.st, DOT_ZR, g0, g1, P.nrows, tid, nthreads);
    if (!P.do_fft) return;
    __syncthreads();

    fft_forward(s, RBP, P.RB, P.f, tid, nthreads);

    // ---- split: Z (H-point spectrum of the packed row) -> 2 X[k], k = 0..H, in place -----------------
    for (int w = tid; w < H * P.RB; w += nthreads) {
        const int line = w % P.RB, p = w / P.RB;
        const int k = P.f.rev[p];
        if (k == 0) {
            const cplx<T> z = s[line];
            s[line] = mk<T>((T)2 * (z.x + z.y), 0);
            s[(size_t)H * RBP + line] = mk<T>((T)2 * (z.x - z.y), 0);
        } else {
            const int k2 = H - k;
            if (k <= k2) {
                const int p2 = P.f.pos[k2];
                const cplx<T> a = s[(size_t)p * RBP + line], c = conj(s[(size_t)p2 * RBP + line]);
                const cplx<T> E = a + c;
                const cplx<T> d = a - c;
                const cplx<T> O = mk<T>(d.y, -d.x);                 // -i d
                const cplx<T> t = P.twL[k] * O;
                s[(size_t)p * RBP + line] = E + t;
                if (k != k2) s[(size_t)p2 * RBP + line] = conj(E - t);
            }
        }
    }
    __syncthreads();

    // ---- store H+1 entries per row --------------------------------------------------------------
    for (int line = warp; line < nl; line += nwarps) {
        const long g = g0 + line;
        cplx<T>* dst = P.W + ((size_t)(g / P.nrows) * P.W_rows + (g % P.nrows)) * P.W_pitch;
        for (int q = lane; q <= H; q += 32) dst[q] = s[(size_t)q * RBP + line];
    }
}

template <class T>
__device__ __forceinline__ cplx<T> apply_spec(cplx<T> v, const void* spec, int kind, size_t idx) {
    if (kind == SPEC_REAL) return v * reinterpret_cast<const T*>(spec)[idx];
    const cplx<T> sv = reinterpret_cast<const cplx<T>*>(spec)[idx];
    return kind == SPEC_CPLX ? v * sv : mulc(v, sv);
}

template <class T>
__global__ void __launch_bounds__(256) rows_inv_kernel(RowsParams<T> P) {
    HIPGP_DYN_SMEM(smem_raw);
    cplx<T>* s = reinterpret_cast<cplx<T>*>(smem_raw);
    const int tid = threadIdx.x, nthreads = blockDim.x;
    const int warp = tid >> 5, lane = tid & 31, nwarps = nthreads >> 5;
    if (P.mode != RI_PLAIN && P.st.flags[0]) return;
    const long g0 = (long)blockIdx.x * P.RB;
    const long g1 = g0 + P.RB < P.total_rows ? g0 + P.RB : P.total_rows;
    const int nl = (int)(g1 - g0);
    const int H = P.H, RBP = P.RBP, n = P.n_real;

    for (int line = warp; line < P.RB; line += nwarps) {
        if (line >= nl) {
            for (int q = lane; q <= H; q += 32) s[(size_t)q * RBP + line] = mk<T>(0, 0);
            continue;
        }
        const long g = g0 + line;
        const cplx<T>* src = P.W + ((size_t)(g / P.nrows) * P.W_rows + (g % P.nrows)) * P.W_pitch;
        for (int q = lane; q <= H; q += 32) {
            cplx<T> v = src[q];
            if (P.spec_kind != SPEC_NONE) v = apply_spec(v, P.spec, P.spec_kind, (size_t)q);
            s[(size_t)q * RBP + line] = v;
        }
    }
    __syncthreads();

    // ---- merge: Y[k], k = 0..H  ->  2 Z[k] (H-point spectrum of the packed row), in place -------------
    for (int w = tid; w < H * P.RB; w += nthreads) {
        const int line = w % P.RB, p = w / P.RB;
        const int k = P.f.rev[p];
        if (k == 0) {
            const T y0 = s[line].x, yh = s[(size_t)H * RBP + line].x;
            s[line] = mk<T>(y0 + yh, y0 - yh);
        } else {
            const int k2 = H - k;
            if (k <= k2) {
                const int p2 = P.f.pos[k2];
                const cplx<T> a = s[(size_t)p * RBP + line], c = conj(s[(size_t)p2 * RBP + line]);
                const cplx<T> E = a + c;
                const cplx<T> O = mulc(a - c, P.twL[k]);           // conj(w^k) (Y[k] - conj Y[k'])
                const cplx<T> iO = mk<T>(-O.y, O.x);
                s[(size_t)p * RBP + line] = E + iO;
                if (k != k2) s[(size_t)p2 * RBP + line] = conj(E - iO);   // conj(E) + i conj(O)
            }
        }
    }
    __syncthreads();

    fft_inverse(s, RBP, P.RB, P.f, tid, nthreads);

    for (int line = warp; line < nl; line += nwarps) {
        const long g = g0 + line;
        const size_t off = (size_t)g * n;
        T acc = 0;
        for (int k = lane; k < H; k += 32) {
            const cplx<T> z = s[(size_t)k * RBP + line];
            const int i = 2 * k;
            if (i < n) { P.out[off + i] = z.x; if (P.mode == RI_DOT) acc += z.x * P.v0[off + i]; }
            if (i + 1 < n) { P.out[off + i + 1] = z.y; if (P.mode == RI_DOT) acc += z.y * P.v0[off + i + 1]; }
        }
        if (P.mode == RI_DOT) {
            const double tot = warp_sum((double)acc);
            if (lane == 0) P.st.partial[g] = tot;
        }
    }
    if (P.mode == RI_DOT) pcg_finalize(P.st, P.dot_kind, g0, g1, P.nrows, tid, nthreads);
}

// ------------------------------------------------------------------------------------------------
template <class T>
struct ColsParams {
    const cplx<T>* in;
    cplx<T>* out;
    int n_in, n_out;              // lines are zero padded from n_in to L (fwd) / cropped to n_out (inv)
    long inner;                   // number of valid lines (fast index) per outer slice
    long pitch;                   // elements between consecutive positions along the axis
    long in_ostride, in_bstride, out_ostride, out_bstride;   // grid.y = outer, grid.z = batch
    LineFft<T> f;                 // L-point complex FFT along the axis
    int TB, TBP;                  // lines per CTA, padded
    int mode;
    const void* spec; int spec_kind;   // FUSED: spectrum indexed [pos * spec_pitch + line]
    long spec_pitch;              // 0 = same as pitch
    int spec_stage;               // specialised kernels: real spectrum tile staged through shared memory
    int in_stage;                 // specialised kernels: input rows prefetched through the shared-memory side buffer
    int nx, ny, nz;               // specialised (persistent) kernels: tile grid = line tiles x outer x batch
    int tma_in, tma_in_rows, tma_in_nbox;   // block-local column kernel: input rows arrive as tma_in_nbox TMA boxes of tma_in_rows rows
    int tma_spec;                 // ... and the real spectrum tile as ONE padded TMA box
    int batch_fastest;            // ... walked batch-fastest (big spectra: a spectrum tile is reused by the CTAs running side by side)
    const int* done_flag;         // optional PCG early-exit flag
};

template <class T>
__global__ void __launch_bounds__(512) cols_pass_kernel(ColsParams<T> P) {
    HIPGP_DYN_SMEM(smem_raw);
    cplx<T>* s = reinterpret_cast<cplx<T>*>(smem_raw);
    const int tid = threadIdx.x, nthreads = blockDim.x;
    if (P.done_flag && *P.done_flag) return;
    const long c0 = (long)blockIdx.x * P.TB;
    const int nc = (int)(P.inner - c0 < P.TB ? P.inner - c0 : P.TB);
    const int L = P.f.Ln, TB = P.TB, TBP = P.TBP;
    const cplx<T>* in = P.in + (size_t)blockIdx.y * P.in_ostride + (size_t)blockIdx.z * P.in_bstride + c0;
    cplx<T>* out = P.out + (size_t)blockIdx.y * P.out_ostride + (size_t)blockIdx.z * P.out_bstride + c0;

    const int rows_in = P.mode == CM_INV ? L : P.n_in;
    for (int w = tid; w < L * TB; w += nthreads) {
        const int c = w % TB, i = w / TB;
        cplx<T> v = mk<T>(0, 0);
        if (i < rows_in && c < nc) v = in[(size_t)i * P.pitch + c];
        s[(size_t)i * TBP + c] = v;
    }
    __syncthreads();

    if (P.mode != CM_INV) fft_forward(s, TBP, TB, P.f, tid, nthreads);
    if (P.mode == CM_FUSED) {
        for (int w = tid; w < L * TB; w += nthreads) {
            const int c = w % TB, i = w / TB;
            if (c < nc) s[(size_t)i * TBP + c] = apply_spec(s[(size_t)i * TBP + c], P.spec, P.spec_kind, (size_t)i * (P.spec_pitch ? P.spec_pitch : P.pitch) + c0 + c);
        }
        __syncthreads();
    }
    if (P.mode != CM_FWD) fft_inverse(s, TBP, TB, P.f, tid, nthreads);

    const int rows_out = P.mode == CM_FWD ? L : P.n_out;
    for (int w = tid; w < rows_out * TB; w += nthreads) {
        const int c = w % TB, i = w / TB;
        if (c < nc) out[(size_t)i * P.pitch + c] = s[(size_t)i * TBP + c];
    }
}

// ---- plain fused vector kernels (CG without preconditioner, and the generic closure path) ----------
// x += a p ; r -= a Ap ; partial r.r  -- is RF_XRUPDATE with do_fft = 0 (rows_fwd_kernel).
// z = r copy is avoided by pointing `in` of RF_PUPDATE at r.

}  // namespace hipgp
