// fast_kernels.cuh -- compile-time specialised versions of the three matvec passes on the lane engine (lane_fft.cuh).
//
// Same math and the same digit-reversed ordering as conv_kernels.cuh (the generic, runtime-radix kernels stay as the
// fallback for lengths without an instantiation).  What is different:
//   * a thread owns (butterfly, lane): 16-byte lanes (two fp32 lines / one fp64 line), LDS.128 / STS.128 only, packed
//     f32x2 arithmetic across the two lines of a lane, all butterfly legs at [base + immediate];
//   * the frequency workspace is kept in LANE layout (lane_fft.cuh), so the column pass moves lanes between global
//     memory and registers with plain 16-byte accesses;
//   * COLUMN pass: persistent CTAs; the first forward stage reads its operands from a shared-memory SIDE buffer that was
//     filled with cp.async while the previous tile was in its inverse stages (zero padding = skipped reads and a pruned
//     butterfly); the same buffer then receives the tile's real spectrum behind the forward stages; last forward stage,
//     spectrum multiply and first inverse stage run back to back in registers; the last inverse stage writes straight
//     to global memory (crop = skipped stores).  Tiles are wide (4 lanes, 512 threads at 2048 points) because the
//     per-butterfly twiddle loads are shared by all lanes of a tile;
//   * ROW passes: small tiles on purpose (2 fp32 rows, 8 CTAs per SM at 1024 points): a row tile is a latency chain.
//     Vectors stream in 16-byte chunks, one row per (sub-)warp team, with the PCG vector updates fused and deterministic
//     row sums; PLAIN row blocks move with one bulk-asynchronous TMA copy (cp.async.bulk + mbarrier); the r2c split /
//     c2r merge works on QUADS -- two neighbouring bins and their two mirror bins -- so one thread turns four
//     shared-memory lanes into 16-byte global accesses, all loads of a thread issued up front and branch-free (the few
//     bins of digit group 0, whose mirrors are irregular, go through a scalar path).
#pragma once
#include "lane_fft.cuh"

namespace hipgp {

template <class T> __device__ __forceinline__ void ld2(const T* p, bool vec, T& a, T& b, bool ok0, bool ok1) {
    if (vec && ok1) { const cplx<T> t = ld_stream(reinterpret_cast<const cplx<T>*>(p)); a = t.x; b = t.y; }
    else { a = ok0 ? ld_stream(p) : (T)0; b = ok1 ? ld_stream(p + 1) : (T)0; }
}
template <class T> __device__ __forceinline__ void st2(T* p, bool vec, T a, T b, bool ok0, bool ok1) {
    if (vec && ok1) { st_stream(reinterpret_cast<cplx<T>*>(p), mk<T>(a, b)); }
    else { if (ok0) st_stream(p, a); if (ok1) st_stream(p + 1, b); }
}

// sum over an aligned team of `tw` lanes (tw a power of two <= 32); every lane of the warp takes part
__device__ __forceinline__ double team_sum(double v, int tw) {
    for (int o = tw >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// spectrum factor(s) of one lane, read from global memory: `idx` = index of the lane's first line in the spectrum
__device__ __forceinline__ Lane<float> lane_spec(Lane<float> v, const void* spec, int kind, size_t idx) {
    if (kind == SPEC_REAL) {
        const cplx<float> sv = ld_stream(reinterpret_cast<const cplx<float>*>(reinterpret_cast<const float*>(spec) + idx));   // two reals
        return lmul_real2(v, sv.x, sv.y);
    }
    const cplx<float>* sp = reinterpret_cast<const cplx<float>*>(spec) + idx;
    const cplx<float> w0 = ld_stream(sp), w1 = ld_stream(sp + 1);
    return kind == SPEC_CPLX ? lmul_cplx2<false>(v, w0, w1) : lmul_cplx2<true>(v, w0, w1);
}
__device__ __forceinline__ Lane<double> lane_spec(Lane<double> v, const void* spec, int kind, size_t idx) {
    if (kind == SPEC_REAL) return lscale(v, ld_stream(reinterpret_cast<const double*>(spec) + idx));
    const cplx<double> w = ld_stream(reinterpret_cast<const cplx<double>*>(spec) + idx);
    return kind == SPEC_CPLX ? lmul(v, w) : lmulc(v, w);
}
// real spectrum factor(s) of one lane staged in shared memory (8 bytes per lane)
__device__ __forceinline__ Lane<float> lane_spec_smem(Lane<float> v, const void* p) {
    const float2 s2 = *reinterpret_cast<const float2*>(p);      // stays a register pair: the packed multiply takes it as is
    Lane<float> r; r.re = __fmul2_rn(v.re, s2); r.im = __fmul2_rn(v.im, s2); return r;
}
__device__ __forceinline__ Lane<double> lane_spec_smem(Lane<double> v, const void* p) { return lscale(v, *reinterpret_cast<const double*>(p)); }

// =====================================================================================================
// Column pass.  PERSISTENT: the grid is sized to the machine and every CTA walks tiles t = blockIdx.x, + gridDim.x, ...
// A tile = NL lanes (= NL * LPT neighbouring lines) of one (outer, batch) slice; tile index = ((bz * ny) + by) * nx + bx,
// so CTAs that run side by side work on neighbouring lines (their 32-byte row segments share DRAM bursts).
// Dynamic shared memory: the tile, then a SIDE buffer that is time-shared: it receives the next tile's input rows with
// cp.async while this tile is in its inverse stages, and this tile's (real) spectrum while it is in its forward stages,
// so neither latency sits on the critical path.
// =====================================================================================================
template <class T, int NL, int NT, int MINB, int R0, int... Rs>
__global__ void __launch_bounds__(NT, MINB) cols_fast_kernel(ColsParams<T> P) {
    using G = TileGeo<T, NL, R0, Rs...>;
    constexpr int Ln = G::Ln, NST = G::NST, RLAST = G::RLAST, LPT = LaneInfo<T>::LPT, TBL = NL * LPT, S0 = Ln / R0;
    HIPGP_DYN_SMEM(smem_raw);
    Lane<T>* s = reinterpret_cast<Lane<T>*>(smem_raw);
    const int tid = threadIdx.x;
    if (P.done_flag && *P.done_flag) return;
    const int mode = P.mode;
    const size_t pitch = (size_t)P.pitch;
    const size_t spitch = P.spec_pitch ? (size_t)P.spec_pitch : (size_t)P.pitch;
    const long ntiles = (long)P.nx * P.ny * P.nz;
    auto tile_origin = [&](long t, long& c0, size_t& ioff, size_t& ooff) {
        long bx, by, bz;
        if (P.batch_fastest) { bz = t % P.nz; const long r = t / P.nz; bx = r % P.nx; by = r / P.nx; }   // spectrum tile reused by neighbours
        else { bx = t % P.nx; const long r = t / P.nx; by = r % P.ny; bz = r / P.ny; }
        c0 = bx * TBL;
        ioff = (size_t)by * P.in_ostride + (size_t)bz * P.in_bstride + c0;
        ooff = (size_t)by * P.out_ostride + (size_t)bz * P.out_bstride + c0;
    };

    if constexpr (NST == 1) {
        // the whole line lives in one thread's registers
        for (long t = blockIdx.x; t < ntiles; t += gridDim.x) {
            long c0; size_t ioff, ooff;
            tile_origin(t, c0, ioff, ooff);
            const long nvalid = P.inner - c0;
            const cplx<T>* in = P.in + ioff;
            cplx<T>* out = P.out + ooff;
            for (int lane = tid; lane < NL; lane += NT) {
                if ((long)lane * LPT >= nvalid) continue;
                const int rows_in = mode == CM_INV ? Ln : P.n_in;
                const int rows_out = mode == CM_FWD ? Ln : P.n_out;
                Lane<T> v[R0];
#pragma unroll
                for (int r = 0; r < R0; ++r)
                    v[r] = r < rows_in ? lane_from_global(in + (size_t)r * P.pitch + lane * LPT) : lzero<T>();
                if (mode != CM_INV) lbfly<R0, false, T>(v);
                if (mode == CM_FUSED) {
#pragma unroll
                    for (int r = 0; r < R0; ++r) v[r] = lane_spec(v[r], P.spec, P.spec_kind, (size_t)r * spitch + c0 + lane * LPT);
                }
                if (mode != CM_FWD) lbfly<R0, true, T>(v);
#pragma unroll
                for (int r = 0; r < R0; ++r)
                    if (r < rows_out) lane_to_global(out + (size_t)r * P.pitch + lane * LPT, v[r]);
            }
        }
        return;
    } else {
        constexpr int LEG0 = G::leg(S0);
        constexpr int SPEC_LANE = 8;                                  // bytes of real spectrum per lane (2 x fp32 or 1 x fp64)
        constexpr int SIDE_SLOTS = Ln + Ln / RLAST;                   // side buffer: SIDE_SLOTS * NL * 8 bytes
        constexpr int SIDE_LANES = SIDE_SLOTS * NL / 2;               // ... = this many 16-byte lanes
        unsigned char* side = smem_raw + G::smem_bytes();
        auto sslot = [](int p) { return p + (p >> G::LOGRL); };       // padded position of the staged spectrum
        const cplx<T>* tw0 = P.f.twst + P.f.twoff[0];
        const bool spec_smem = P.spec_stage != 0;                     // FUSED with a real spectrum
        const int n_in = P.n_in, n_out = P.n_out;
        const bool stage_in = P.in_stage != 0;                        // input rows go through the side buffer
        const bool zero_hi = is_pow2(R0) && n_in <= Ln / 2;
        const bool out_lo = is_pow2(R0) && n_out <= Ln / 2;
        const size_t rstep = (size_t)S0 * pitch;

        // asynchronous copy of a tile's input rows (row i, lane l -> side lane i * NL + l)
        auto prefetch_input = [&](long t) {
            long c0; size_t ioff, ooff;
            tile_origin(t, c0, ioff, ooff);
            const long nvalid = P.inner - c0;
            const cplx<T>* in = P.in + ioff;
            constexpr int NIT = (SIDE_LANES + NT - 1) / NT;
            const int total = n_in * NL;
#pragma unroll
            for (int k = 0; k < NIT; ++k) {
                const int w = tid + k * NT;
                const int i = w / NL, lane = w - i * NL;
                if (w < total && (long)lane * LPT < nvalid) cp_async<16>(side + (size_t)w * 16, in + (size_t)i * pitch + lane * LPT);
            }
            cp_async_commit();
        };

        long t = blockIdx.x;
        if (stage_in && t < ntiles) prefetch_input(t);
        for (; t < ntiles; t += gridDim.x) {
            long c0; size_t ioff, ooff;
            tile_origin(t, c0, ioff, ooff);
            const long nvalid = P.inner - c0;                   // lines of this tile that exist
            const cplx<T>* in = P.in + ioff;
            cplx<T>* out = P.out + ooff;
            // the previous tile's last stage has to be done with the tile buffer, and this tile's input must have landed
            cp_async_wait_all();
            __syncthreads();

            // ---- first forward stage: operands from the side buffer or straight from global memory (zero padding = skipped loads) ----
            if (mode != CM_INV) {
#pragma unroll 1
                for (int it = tid; it < S0 * NL; it += NT) {
                    const int lane = it % NL, j = it / NL;
                    const bool ok = (long)lane * LPT < nvalid;
                    cplx<T> w[R0];
                    lane_twiddles<R0, S0>(w, tw0, j);
                    Lane<T> v[R0];
                    if (stage_in) {
                        const Lane<T>* sp = reinterpret_cast<const Lane<T>*>(side) + (j * NL + lane);
                        if (zero_hi) {
#pragma unroll
                            for (int r = 0; r < R0 / 2; ++r) v[r] = (ok && j + r * S0 < n_in) ? sp[r * S0 * NL] : lzero<T>();
                            lbfly_zero_hi<R0, T>(v);
                        } else {
#pragma unroll
                            for (int r = 0; r < R0; ++r) v[r] = (ok && j + r * S0 < n_in) ? sp[r * S0 * NL] : lzero<T>();
                            lbfly<R0, false, T>(v);
                        }
                    } else {
                        const cplx<T>* gp = in + (size_t)j * pitch + lane * LPT;
                        if (zero_hi) {
#pragma unroll
                            for (int r = 0; r < R0 / 2; ++r) v[r] = (ok && j + r * S0 < n_in) ? lane_from_global(gp + r * rstep) : lzero<T>();
                            lbfly_zero_hi<R0, T>(v);
                        } else {
#pragma unroll
                            for (int r = 0; r < R0; ++r) v[r] = (ok && j + r * S0 < n_in) ? lane_from_global(gp + r * rstep) : lzero<T>();
                            lbfly<R0, false, T>(v);
                        }
                    }
#pragma unroll
                    for (int r = 1; r < R0; ++r) v[r] = lmul(v[r], w[r]);
                    Lane<T>* base = s + (G::slot(j) * NL + lane);
#pragma unroll
                    for (int r = 0; r < R0; ++r) base[r * LEG0] = v[r];
                }
                __syncthreads();
                // ---- spectrum tile -> side buffer (free now), asynchronously behind the forward middle stages ----
                if (spec_smem) {
                    const unsigned char* sp = reinterpret_cast<const unsigned char*>(P.spec) + (size_t)c0 * sizeof(T);
                    constexpr int ROWB = NL * SPEC_LANE;                      // bytes per position
                    constexpr int CH = ROWB >= 16 ? 16 : 8, NCH = ROWB / CH;
                    constexpr int NIT = (Ln * NCH + NT - 1) / NT;
#pragma unroll
                    for (int k = 0; k < NIT; ++k) {
                        const int w = tid + k * NT;
                        const int p = w / NCH, c = w - p * NCH;
                        if (w < Ln * NCH) cp_async<CH>(side + (size_t)sslot(p) * ROWB + c * CH, sp + (size_t)p * spitch * sizeof(T) + c * CH);
                    }
                    cp_async_commit();
                }
                LaneMidFwd<G, T, NL, NT, Ln / R0, 1, Rs...>::run(s, P.f, tid);
                if (spec_smem) { cp_async_wait_all(); __syncthreads(); }
            }

            // ---- last forward stage + spectrum + first inverse stage: RLAST neighbouring positions, in registers ----
            {
#pragma unroll 2
                for (int it = tid; it < (Ln / RLAST) * NL; it += NT) {
                    const int lane = it % NL, bf = it / NL;
                    const bool ok = (long)lane * LPT < nvalid;
                    const int p0 = bf * RLAST;
                    Lane<T>* base = s + (G::slot(p0) * NL + lane);
                    Lane<T> v[RLAST];
                    if (mode == CM_INV) {
                        const cplx<T>* gp = in + (size_t)p0 * P.pitch + lane * LPT;
#pragma unroll
                        for (int r = 0; r < RLAST; ++r) v[r] = ok ? lane_from_global(gp + r * pitch) : lzero<T>();
                    } else {
#pragma unroll
                        for (int r = 0; r < RLAST; ++r) v[r] = base[r * NL];
                        lbfly<RLAST, false, T>(v);
                    }
                    if (mode == CM_FUSED) {
                        if (spec_smem) {
                            const unsigned char* sp = side + ((size_t)sslot(p0) * NL + lane) * SPEC_LANE;
#pragma unroll
                            for (int r = 0; r < RLAST; ++r) v[r] = lane_spec_smem(v[r], sp + r * NL * SPEC_LANE);
                        } else if (ok) {
                            const size_t sidx = (size_t)p0 * spitch + c0 + lane * LPT;
#pragma unroll
                            for (int r = 0; r < RLAST; ++r) v[r] = lane_spec(v[r], P.spec, P.spec_kind, sidx + (size_t)r * spitch);
                        }
                    }
                    if (mode == CM_FWD) {
                        if (ok) {
                            cplx<T>* gp = out + (size_t)p0 * P.pitch + lane * LPT;
#pragma unroll
                            for (int r = 0; r < RLAST; ++r) lane_to_global(gp + r * pitch, v[r]);
                        }
                    } else {
                        lbfly<RLAST, true, T>(v);
#pragma unroll
                        for (int r = 0; r < RLAST; ++r) base[r * NL] = v[r];
                    }
                }
                __syncthreads();
            }
            // ---- the side buffer is free again: next tile's input rows travel behind the inverse stages ----
            if (stage_in && t + gridDim.x < ntiles) prefetch_input(t + gridDim.x);
            if (mode == CM_FWD) continue;

            // ---- inverse middle stages, then the last inverse stage straight to global memory (crop = skipped stores) ----
            LaneMidInv<G, T, NL, NT, Ln / R0, 1, Rs...>::run(s, P.f, tid);
            {
#pragma unroll 1
                for (int it = tid; it < S0 * NL; it += NT) {
                    const int lane = it % NL, j = it / NL;
                    const bool ok = (long)lane * LPT < nvalid;
                    cplx<T> w[R0];
                    lane_twiddles<R0, S0>(w, tw0, j);
                    const Lane<T>* base = s + (G::slot(j) * NL + lane);
                    Lane<T> v[R0];
#pragma unroll
                    for (int r = 0; r < R0; ++r) v[r] = base[r * LEG0];
#pragma unroll
                    for (int r = 1; r < R0; ++r) v[r] = lmulc(v[r], w[r]);
                    cplx<T>* gp = out + (size_t)j * pitch + lane * LPT;
                    lbfly<R0, true, T>(v);
                    if (ok) {
                        if (out_lo) {
#pragma unroll
                            for (int r = 0; r < R0 / 2; ++r) if (j + r * S0 < n_out) lane_to_global(gp + r * rstep, v[r]);
                        } else {
#pragma unroll
                            for (int r = 0; r < R0; ++r) if (j + r * S0 < n_out) lane_to_global(gp + r * rstep, v[r]);
                        }
                    }
                }
            }
        }
    }
}

// =====================================================================================================
// Row passes.  H = product of the radix list; a CTA owns NL lanes = NL * LPT rows.
// =====================================================================================================
struct __align__(8) QuadIdx { int a, b; };     // even positions of a quad: bins (a, a+1) mirror bins (b+1, b)

template <class T, int NL, int NT, int MINB, int R0, int... Rs>
__global__ void __launch_bounds__(NT, MINB) rows_fwd_fast_kernel(RowsParams<T> P) {
    using G = TileGeo<T, NL, R0, Rs...>;
    constexpr int H = G::Ln, NST = G::NST, RLAST = G::RLAST, LPT = LaneInfo<T>::LPT, NROW = NL * LPT, S0 = H / R0;
    constexpr int LEG0 = G::leg(NST > 1 ? S0 : 1);
    HIPGP_DYN_SMEM(smem_raw);
    Lane<T>* s = reinterpret_cast<Lane<T>*>(smem_raw);
    const int tid = threadIdx.x;
    if (P.mode != RF_PLAIN && P.st.flags[0]) return;
    const long g0 = (long)blockIdx.x * NROW;
    const long g1 = g0 + NROW < P.total_rows ? g0 + NROW : P.total_rows;
    const int nl = (int)(g1 - g0);
    const int n = P.n_real;
    const int mode = P.mode;
    const bool vec = ((n & 1) == 0) && P.vec_ok;             // rows start on even offsets => 2-element accesses are aligned
    const bool first_it = (mode == RF_PUPDATE) && (P.st.flags[2] != 0);
    const bool want_dot = (mode == RF_XRUPDATE || mode == RF_SELFDOT);
    // per-row scalars, computed once (the 64-bit divisions stay out of the element loops)
    __shared__ T s_coef[32];
    __shared__ long s_wbase[32];
    __shared__ double s_part[32];
    if (tid < NROW && tid < nl) {
        const long gr = g0 + tid;
        const long b = gr / P.nrows;
        s_wbase[tid] = (b * P.W_rows + (gr - b * P.nrows)) * P.W_pitch;
        T coef = 0;
        if (mode == RF_PUPDATE) coef = first_it ? (T)0 : (T)(P.st.zr[b] / P.st.zr_prev[b]);
        else if (mode == RF_XRUPDATE) coef = (T)(P.st.zr[b] / P.st.pAp[b]);
        s_coef[tid] = coef;
    }
    __syncthreads();

    // ---- streaming phase: one warp per row, 16-byte accesses; the fused PCG vector update happens here; the FFT input
    //      row goes to the side buffer (row-major, SROW reals per row, zero-filled behind n); deterministic row sums ----
    const int SROW = (n + 3) & ~3;
    T* side = reinterpret_cast<T*>(smem_raw + G::smem_bytes());
    bool streamed = false;
#ifndef HIPGP_EMU
    // Bulk-asynchronous (TMA) streaming: the tile's rows are one contiguous block of every vector.  The FFT input lands in
    // the side buffer and the other operands of a fused PCG update in the (still idle) tile buffer -- one instruction per
    // vector, no register staging; the update then runs shared memory -> shared memory and the updated vector leaves with
    // one bulk store.  Only x of the x/r update (read AND written) goes through ordinary 16-byte accesses.
    bool bulk_store_pending = false;
    if (P.vec16_ok && SROW == n && (mode == RF_PLAIN || mode == RF_SELFDOT || P.tma_op)) {
        constexpr int CH = 16 / (int)sizeof(T);
        __shared__ __align__(8) unsigned long long s_mbar;
        const unsigned bytes = (unsigned)((size_t)nl * n * sizeof(T));
        const size_t goff = (size_t)g0 * n;
        T* bufA = reinterpret_cast<T*>(smem_raw);                  // operand landing zones inside the tile buffer
        T* bufB = bufA + (size_t)NROW * SROW;
        const bool two = mode == RF_PUPDATE && !first_it, three = mode == RF_XRUPDATE;
        if (tid == 0) { mbar_init(&s_mbar, 1); fence_proxy_async(); }
        __syncthreads();
        if (tid == 0) {
            mbar_arrive_expect_tx(&s_mbar, bytes * (three ? 3u : (two ? 2u : 1u)));
            bulk_g2s(side, P.in + goff, bytes, &s_mbar);                                   // in / z / Ap
            if (two) bulk_g2s(bufA, (const T*)P.v0 + goff, bytes, &s_mbar);                // p
            if (three) { bulk_g2s(bufA, (const T*)P.v0 + goff, bytes, &s_mbar); bulk_g2s(bufB, P.v2 + goff, bytes, &s_mbar); }   // r, p
        }
        // row teams (same dealing as the register path below)
        constexpr int NW = NT / 32, WPR = NW > NROW ? NW / NROW : 1;
        constexpr int tws = WPR > 1 ? 32 : (H / CH >= 32 ? 32 : (H / CH >= 16 ? 16 : (H / CH >= 8 ? 8 : 4)));
        constexpr int rpw = 32 / tws, TW = WPR > 1 ? 32 * WPR : tws, rstep = WPR > 1 ? NW / WPR : NW * rpw;
        const int warp = tid >> 5, l32 = tid & 31;
        const int ln = WPR > 1 ? l32 + 32 * (warp % WPR) : l32 % tws;
        const int nch = n / CH;
        mbar_wait(&s_mbar, 0);
        if (mode != RF_PLAIN && !(mode == RF_PUPDATE && first_it)) {
            for (int rbase = WPR > 1 ? warp / WPR : warp * rpw; rbase < nl; rbase += rstep) {
                const int row = rbase + (WPR > 1 ? 0 : l32 / tws);
                const bool ractive = row < nl;
                double acc = 0.0;
                if (ractive) {
                    T* srow = side + (size_t)row * SROW;
                    const T* arow = bufA + (size_t)row * SROW;
                    const T* brow = bufB + (size_t)row * SROW;
                    const size_t off = goff + (size_t)row * n;
                    const T coef = s_coef[row];
                    if (three) {
                        constexpr int BS = 4;                   // x: ordinary loads, a batch in flight
                        for (int cb = ln; cb < nch; cb += TW * BS) {
                            Vec16<T> xv[BS];
#pragma unroll
                            for (int k = 0; k < BS; ++k) { const int c = cb + TW * k; if (c < nch) xv[k] = ldv_stream((const T*)P.v1 + off + (size_t)c * CH); }
#pragma unroll
                            for (int k = 0; k < BS; ++k) {
                                const int c = cb + TW * k;
                                if (c < nch) {
                                    Vec16<T> q = *reinterpret_cast<const Vec16<T>*>(srow + c * CH);          // Ap
                                    const Vec16<T> rv = *reinterpret_cast<const Vec16<T>*>(arow + c * CH);   // r
                                    const Vec16<T> pv = *reinterpret_cast<const Vec16<T>*>(brow + c * CH);   // p
#pragma unroll
                                    for (int e = 0; e < CH; ++e) { xv[k].v[e] = xv[k].v[e] + coef * pv.v[e]; q.v[e] = rv.v[e] - coef * q.v[e]; acc += (double)(q.v[e] * q.v[e]); }
                                    stv_stream(P.v1 + off + (size_t)c * CH, xv[k]);
                                    *reinterpret_cast<Vec16<T>*>(srow + c * CH) = q;                          // r_new = FFT input
                                }
                            }
                        }
                    } else if (two) {
                        for (int c = ln; c < nch; c += TW) {
                            Vec16<T> z = *reinterpret_cast<const Vec16<T>*>(srow + c * CH);
                            const Vec16<T> pv = *reinterpret_cast<const Vec16<T>*>(arow + c * CH);
#pragma unroll
                            for (int e = 0; e < CH; ++e) z.v[e] = z.v[e] + coef * pv.v[e];
                            *reinterpret_cast<Vec16<T>*>(srow + c * CH) = z;                                  // p_new = FFT input
                        }
                    } else {        // RF_SELFDOT
                        for (int c = ln; c < nch; c += TW) {
                            const Vec16<T> z = *reinterpret_cast<const Vec16<T>*>(srow + c * CH);
#pragma unroll
                            for (int e = 0; e < CH; ++e) acc += (double)(z.v[e] * z.v[e]);
                        }
                    }
                }
                if (want_dot) {
                    acc = team_sum(acc, WPR > 1 ? 32 : tws);
                    if (ractive && (WPR > 1 ? l32 == 0 : ln == 0)) s_part[row * WPR + warp % WPR] = acc;
                }
            }
        }
        if (mode == RF_PUPDATE || mode == RF_XRUPDATE) {       // the updated vector (p or r) = the side buffer -> global
            fence_proxy_async();
            __syncthreads();
            if (tid == 0) {
                asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(P.v0 + goff), "r"((unsigned)__cvta_generic_to_shared(side)), "r"(bytes) : "memory");
                asm volatile("cp.async.bulk.commit_group;" ::: "memory");
            }
            bulk_store_pending = true;
        }
        if (want_dot) {
            __syncthreads();
            if (tid < nl) { double a = 0.0; for (int k = 0; k < WPR; ++k) a += s_part[tid * WPR + k]; P.st.partial[g0 + tid] = a; }
        }
        streamed = true;
    }
#endif
    if (!streamed) {
        constexpr int CH = 16 / (int)sizeof(T);
        // Teams: WPR warps share a row when there are more warps than rows; short rows are dealt to sub-warp teams of
        // `tws` lanes so that all 32 lanes of a warp stream.  TW = lanes per row, `rstep` = rows per sweep of the CTA.
        constexpr int NW = NT / 32, WPR = NW > NROW ? NW / NROW : 1;
        const bool chunked = P.vec16_ok && (n % CH == 0);
        // (team width fixed at compile time from the row length the transform was chosen for: n ~ H reals = H / CH chunks)
        constexpr int tws = WPR > 1 ? 32 : (H / CH >= 32 ? 32 : (H / CH >= 16 ? 16 : (H / CH >= 8 ? 8 : 4)));
        constexpr int rpw = 32 / tws;                              // rows per warp
        constexpr int TW = WPR > 1 ? 32 * WPR : tws;
        const int warp = tid >> 5, l32 = tid & 31;
        const int ln = WPR > 1 ? l32 + 32 * (warp % WPR) : l32 % tws;
        constexpr int rstep = WPR > 1 ? NW / WPR : NW * rpw;
        for (int rbase = WPR > 1 ? warp / WPR : warp * rpw; rbase < nl; rbase += rstep) {
            const int row = rbase + (WPR > 1 ? 0 : l32 / tws);
            const bool ractive = row < nl;
            T* srow = side + (size_t)(ractive ? row : 0) * SROW;
            const size_t off = (size_t)(g0 + (ractive ? row : 0)) * n;
            const T coef = s_coef[ractive ? row : 0];
            double acc = 0.0;
            if (!ractive) {
            } else if (chunked) {
                // batches of BS chunks per lane: all loads of a batch are in flight before the first use
                const int nch = n / CH;
                auto finish = [&](int c, Vec16<T> a) {
                    if (want_dot) {
#pragma unroll
                        for (int k = 0; k < CH; ++k) acc += (double)(a.v[k] * a.v[k]);
                    }
                    *reinterpret_cast<Vec16<T>*>(srow + c * CH) = a;
                };
                // two register sets, software-pipelined: the loads of batch b+1 are issued before batch b is consumed,
                // so a full batch of 16-byte loads per lane is always in flight
#define HIPGP_PIPE(LOAD, PROC)                                                                              \
                {                                                                                           \
                    const int step = TW * BS;                                                               \
                    int cb = ln;                                                                            \
                    LOAD(0, cb);                                                                            \
                    for (; cb < nch; cb += 2 * step) {                                                      \
                        if (cb + step < nch) { LOAD(1, cb + step); }                                        \
                        PROC(0, cb);                                                                        \
                        if (cb + 2 * step < nch) { LOAD(0, cb + 2 * step); }                                \
                        if (cb + step < nch) { PROC(1, cb + step); }                                        \
                    }                                                                                       \
                }
                if (mode == RF_XRUPDATE) {
                    constexpr int BS = 1;
                    Vec16<T> a[2][BS], pv[2][BS], xv[2][BS], rv[2][BS];
#define HIPGP_LD(S, CB)                                                                                     \
                    _Pragma("unroll") for (int k = 0; k < BS; ++k) {                                        \
                        const int c = (CB) + TW * k;                                                        \
                        if (c < nch) {                                                                      \
                            const size_t o = off + (size_t)c * CH;                                          \
                            a[S][k] = ldv_stream(P.in + o); pv[S][k] = ldv_stream(P.v2 + o);                \
                            xv[S][k] = ldv_stream((const T*)P.v1 + o); rv[S][k] = ldv_stream((const T*)P.v0 + o); \
                        }                                                                                   \
                    }
#define HIPGP_PR(S, CB)                                                                                     \
                    _Pragma("unroll") for (int k = 0; k < BS; ++k) {                                        \
                        const int c = (CB) + TW * k;                                                        \
                        if (c < nch) {                                                                      \
                            const size_t o = off + (size_t)c * CH;                                          \
                            _Pragma("unroll") for (int e = 0; e < CH; ++e) {                                \
                                xv[S][k].v[e] = xv[S][k].v[e] + coef * pv[S][k].v[e];                       \
                                a[S][k].v[e] = rv[S][k].v[e] - coef * a[S][k].v[e];                         \
                            }                                                                               \
                            stv_stream(P.v1 + o, xv[S][k]);                                                 \
                            stv_stream(P.v0 + o, a[S][k]);                                                  \
                            finish(c, a[S][k]);                                                             \
                        }                                                                                   \
                    }
                    HIPGP_PIPE(HIPGP_LD, HIPGP_PR)
#undef HIPGP_LD
#undef HIPGP_PR
                } else if (mode == RF_PUPDATE && !first_it) {
                    constexpr int BS = 2;
                    Vec16<T> a[2][BS], pv[2][BS];
#define HIPGP_LD(S, CB)                                                                                     \
                    _Pragma("unroll") for (int k = 0; k < BS; ++k) {                                        \
                        const int c = (CB) + TW * k;                                                        \
                        if (c < nch) { const size_t o = off + (size_t)c * CH; a[S][k] = ldv_stream(P.in + o); pv[S][k] = ldv_stream((const T*)P.v0 + o); } \
                    }
#define HIPGP_PR(S, CB)                                                                                     \
                    _Pragma("unroll") for (int k = 0; k < BS; ++k) {                                        \
                        const int c = (CB) + TW * k;                                                        \
                        if (c < nch) {                                                                      \
                            _Pragma("unroll") for (int e = 0; e < CH; ++e) a[S][k].v[e] = a[S][k].v[e] + coef * pv[S][k].v[e]; \
                            stv_stream(P.v0 + off + (size_t)c * CH, a[S][k]);                               \
                            finish(c, a[S][k]);                                                             \
                        }                                                                                   \
                    }
                    HIPGP_PIPE(HIPGP_LD, HIPGP_PR)
#undef HIPGP_LD
#undef HIPGP_PR
                } else {
                    constexpr int BS = 4;
                    const bool wr = mode == RF_PUPDATE;      // first iteration: p = z
                    Vec16<T> a[2][BS];
#define HIPGP_LD(S, CB)                                                                                     \
                    _Pragma("unroll") for (int k = 0; k < BS; ++k) { const int c = (CB) + TW * k; if (c < nch) a[S][k] = ldv_stream(P.in + off + (size_t)c * CH); }
#define HIPGP_PR(S, CB)                                                                                     \
                    _Pragma("unroll") for (int k = 0; k < BS; ++k) {                                        \
                        const int c = (CB) + TW * k;                                                        \
                        if (c < nch) { if (wr) stv_stream(P.v0 + off + (size_t)c * CH, a[S][k]); finish(c, a[S][k]); } \
                    }
                    HIPGP_PIPE(HIPGP_LD, HIPGP_PR)
#undef HIPGP_LD
#undef HIPGP_PR
                }
#undef HIPGP_PIPE
            } else {
                for (int i = ln; i < n; i += TW) {
                    const size_t o = off + i;
                    T a = ld_stream(P.in + o);
                    if (mode == RF_PUPDATE) {
                        if (!first_it) a = a + coef * ld_stream((const T*)P.v0 + o);
                        st_stream(P.v0 + o, a);
                    } else if (mode == RF_XRUPDATE) {
                        const T pv = ld_stream(P.v2 + o);
                        st_stream(P.v1 + o, ld_stream((const T*)P.v1 + o) + coef * pv);
                        a = ld_stream((const T*)P.v0 + o) - coef * a;
                        st_stream(P.v0 + o, a);
                    }
                    if (want_dot) acc += (double)(a * a);
                    srow[i] = a;
                }
            }
            if (ractive) for (int i = n + ln; i < SROW; i += TW) srow[i] = (T)0;
            if (want_dot) {
                acc = team_sum(acc, WPR > 1 ? 32 : tws);
                if (ractive && (WPR > 1 ? l32 == 0 : ln == 0)) s_part[row * WPR + warp % WPR] = acc;
            }
        }
        if (want_dot) {      // fixed-order sum of the WPR partials of a row
            __syncthreads();
            if (tid < nl) { double a = 0.0; for (int k = 0; k < WPR; ++k) a += s_part[tid * WPR + k]; P.st.partial[g0 + tid] = a; }
        }
    }
    __syncthreads();
    if (want_dot) pcg_finalize(P.st, mode == RF_XRUPDATE ? DOT_RR : DOT_ZR, g0, g1, P.nrows, tid, NT);

    // ---- first DIF stage, operands from the side buffer (packed complex e = x[2e] + i x[2e+1]; zero padding = skipped reads) ----
    {
        const bool zero_hi = is_pow2(R0) && R0 > 1 && (n + 1) / 2 <= H / 2;
        const cplx<T>* tw0 = P.f.twst + P.f.twoff[0];
#pragma unroll 1
        for (int it = tid; it < S0 * NL; it += NT) {
            const int lane = it % NL, j = it / NL;
            cplx<T> w[R0];
            if (NST > 1) lane_twiddles<R0, S0>(w, tw0, j);
            const T* srow0 = side + (size_t)(lane * LPT) * SROW;
            const T* srow1 = side + (size_t)(lane * LPT + LPT - 1) * SROW;
            const bool ok0 = lane * LPT < nl, ok1 = lane * LPT + LPT - 1 < nl;
            auto elem = [&](int r) -> Lane<T> {
                const int i = 2 * (j + r * S0);
                const bool in_row = i < SROW;
                const cplx<T> e0 = (ok0 && in_row) ? *reinterpret_cast<const cplx<T>*>(srow0 + i) : mk<T>(0, 0);
                const cplx<T> e1 = (LPT == 2 && ok1 && in_row) ? *reinterpret_cast<const cplx<T>*>(srow1 + i) : mk<T>(0, 0);
                return lane_make(e0, e1);
            };
            Lane<T> v[R0];
            if (zero_hi) {
#pragma unroll
                for (int r = 0; r < R0 / 2; ++r) v[r] = elem(r);
                lbfly_zero_hi<R0, T>(v);
            } else {
#pragma unroll
                for (int r = 0; r < R0; ++r) v[r] = elem(r);
                lbfly<R0, false, T>(v);
            }
            if (NST > 1) {
#pragma unroll
                for (int r = 1; r < R0; ++r) v[r] = lmul(v[r], w[r]);
            }
            Lane<T>* base = s + (G::slot(j) * NL + lane);
#pragma unroll
            for (int r = 0; r < R0; ++r) base[r * LEG0] = v[r];
        }
    }
    __syncthreads();

    if constexpr (NST > 1) {
        LaneMidFwd<G, T, NL, NT, H / R0, 1, Rs...>::run(s, P.f, tid);
        lane_stage<G, T, NL, NT, RLAST, RLAST, false>(s, P.f.twst, tid);
        __syncthreads();
    }

    // ---- r2c split, straight to global memory ----
    // (a) pairs (k, H-k) of digit group 0 (all pairs when the list has a single stage): scalar W accesses
    constexpr int NPAIR0 = NST > 1 ? RLAST / 2 + 1 : H / 2 + 1;
    constexpr int NQUAD = NST > 1 ? (H - RLAST) / 4 : 0;
#pragma unroll 1
    for (int it = tid; it < NPAIR0 * NL; it += NT) {
        const int lane = it % NL, pi = it / NL;
        const QuadIdx pq = reinterpret_cast<const QuadIdx*>(P.pairs)[pi];
        const int q = pq.a, q2 = pq.b;
        Lane<T> Xa, Xb;
        bool two;
        if (q == 0) {
            const Lane<T> z = s[lane];
            Lane<T> zs; zs.re = z.im; zs.im = z.re;
            Xa = lscale(z + zs, (T)2); Xb = lscale(z - zs, (T)2);       // .re = 2 (re +- im); imaginary parts are zero
            Xa.im = lzero<T>().im; Xb.im = lzero<T>().im;
            two = true;
        } else {
            const cplx<T> wq = ldg_c(P.pairw + pi);
            const Lane<T> a = s[G::slot(q) * NL + lane], c = lconj(s[G::slot(q2) * NL + lane]);
            const Lane<T> E = a + c;
            const Lane<T> t = lmul(lmi<false>(a - c), wq);
            Xa = E + t; Xb = lconj(E - t);
            two = q2 != q;
        }
#pragma unroll
        for (int l = 0; l < LPT; ++l) {
            const int row = lane * LPT + l;
            if (row < nl) {
                cplx<T>* dst = P.W + s_wbase[row];
                WRow<T>::store1(dst, q, lane_get(Xa, l));
                if (two) WRow<T>::store1(dst, q2, lane_get(Xb, l));
            }
        }
    }
    // (b) quads: bins (a, a+1) and their mirrors (b+1, b): four lanes in, 16-byte stores out.  The table loads of
    //     all of a thread's quads are issued up front.
    if constexpr (NQUAD > 0) {
        constexpr int QIT = (NQUAD * NL + NT - 1) / NT;
        QuadIdx qq[QIT]; cplx<T> wa[QIT], wa1[QIT];
#pragma unroll
        for (int k = 0; k < QIT; ++k) {
            const int it = tid + k * NT, qi = it / NL;
            if (it < NQUAD * NL) { qq[k] = reinterpret_cast<const QuadIdx*>(P.quadq)[qi]; wa[k] = ldg_c(P.quadw + 2 * qi); wa1[k] = ldg_c(P.quadw + 2 * qi + 1); }
        }
#pragma unroll
        for (int k = 0; k < QIT; ++k) {
            const int it = tid + k * NT, lane = it % NL;
            if (it < NQUAD * NL) {
                const Lane<T>* pa = s + (G::slot(qq[k].a) * NL + lane);
                const Lane<T>* pb = s + (G::slot(qq[k].b) * NL + lane);
                const Lane<T> za = pa[0], za1 = pa[NL], zb = pb[0], zb1 = pb[NL];
                // bin a with mirror b+1
                Lane<T> c = lconj(zb1);
                Lane<T> E = za + c;
                Lane<T> t = lmul(lmi<false>(za - c), wa[k]);
                const Lane<T> Xa = E + t, Xb1 = lconj(E - t);
                // bin a+1 with mirror b
                c = lconj(zb);
                E = za1 + c;
                t = lmul(lmi<false>(za1 - c), wa1[k]);
                const Lane<T> Xa1 = E + t, Xb = lconj(E - t);
                const bool self = qq[k].a == qq[k].b;    // the quad mirrors onto itself: bins (a, a+1) are each other's mirror
#pragma unroll
                for (int l = 0; l < LPT; ++l) {
                    const int row = lane * LPT + l;
                    if (row < nl) {
                        cplx<T>* dst = P.W + s_wbase[row];
                        if (self) WRow<T>::store2(dst, qq[k].a, lane_get(Xa, l), lane_get(Xb1, l));
                        else { WRow<T>::store2(dst, qq[k].a, lane_get(Xa, l), lane_get(Xa1, l)); WRow<T>::store2(dst, qq[k].b, lane_get(Xb, l), lane_get(Xb1, l)); }
                    }
                }
            }
        }
    }
#ifndef HIPGP_EMU
    if (bulk_store_pending && tid == 0) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");   // the side buffer has been read
#endif
}

template <class T, int NL, int NT, int MINB, int R0, int... Rs>
__global__ void __launch_bounds__(NT, MINB) rows_inv_fast_kernel(RowsParams<T> P) {
    using G = TileGeo<T, NL, R0, Rs...>;
    constexpr int H = G::Ln, NST = G::NST, RLAST = G::RLAST, LPT = LaneInfo<T>::LPT, NROW = NL * LPT, S0 = H / R0;
    constexpr int LEG0 = G::leg(NST > 1 ? S0 : 1);
    HIPGP_DYN_SMEM(smem_raw);
    Lane<T>* s = reinterpret_cast<Lane<T>*>(smem_raw);
    const int tid = threadIdx.x;
    if (P.mode != RI_PLAIN && P.st.flags[0]) return;
    const long g0 = (long)blockIdx.x * NROW;
    const long g1 = g0 + NROW < P.total_rows ? g0 + NROW : P.total_rows;
    const int nl = (int)(g1 - g0);
    const int n = P.n_real;

    __shared__ long s_wbase[32];
    __shared__ double s_part[32];
    if (tid < NROW && tid < nl) {
        const long gr = g0 + tid;
        const long b = gr / P.nrows;
        s_wbase[tid] = (b * P.W_rows + (gr - b * P.nrows)) * P.W_pitch;
    }
    __syncthreads();

    // ---- c2r merge, straight from global memory into shared memory ----
    const int spec_kind = P.spec_kind;
    constexpr int NPAIR0 = NST > 1 ? RLAST / 2 + 1 : H / 2 + 1;
    constexpr int NQUAD = NST > 1 ? (H - RLAST) / 4 : 0;
    // (a) pairs of digit group 0 (all pairs when the list has a single stage)
#pragma unroll 1
    for (int it = tid; it < NPAIR0 * NL; it += NT) {
        const int lane = it % NL, pi = it / NL;
        const QuadIdx pq = reinterpret_cast<const QuadIdx*>(P.pairs)[pi];
        const int q = pq.a, q2 = pq.b;
        const cplx<T> wq = ldg_c(P.pairw + pi);
        cplx<T> ya[LPT], yc[LPT];
#pragma unroll
        for (int l = 0; l < LPT; ++l) {
            const int row = lane * LPT + l;
            ya[l] = mk<T>(0, 0); yc[l] = mk<T>(0, 0);
            if (row < nl) {
                const cplx<T>* src = P.W + s_wbase[row];
                ya[l] = WRow<T>::load1(src, q); yc[l] = WRow<T>::load1(src, q2);
                if (spec_kind != SPEC_NONE) { ya[l] = apply_spec(ya[l], P.spec, spec_kind, (size_t)q); yc[l] = apply_spec(yc[l], P.spec, spec_kind, (size_t)q2); }
            }
        }
        const Lane<T> a = lane_make(ya[0], ya[LPT - 1]);
        Lane<T> c = lane_make(yc[0], yc[LPT - 1]);
        if (q == 0) {
            // Z[0] = (Y0 + YH) + i (Y0 - YH), real parts only
            Lane<T> z; z.re = (a + c).re; z.im = (a - c).re;
            s[lane] = z;
        } else {
            // bin q (frequency k):  E + i O with O = conj(w^k)(Y[k] - conj Y[k']);  bin q2 is conj(E - i O)
            c = lconj(c);
            const Lane<T> E = a + c;
            const Lane<T> iO = lmi<true>(lmulc(a - c, wq));
            s[G::slot(q) * NL + lane] = E + iO;
            if (q2 != q) s[G::slot(q2) * NL + lane] = lconj(E - iO);
        }
    }
    // (b) quads: the table and workspace loads of all of a thread's quads are issued up front, branch-free (rows past
    //     the end of the batch read the last valid row and are dropped at the very end), so they are all in flight together
    if constexpr (NQUAD > 0) {
        constexpr int QIT = (NQUAD * NL + NT - 1) / NT;
        QuadIdx qq[QIT]; cplx<T> wa[QIT], wa1[QIT];
        cplx<T> ya[QIT][LPT], ya1[QIT][LPT], yb[QIT][LPT], yb1[QIT][LPT];
#pragma unroll
        for (int k = 0; k < QIT; ++k) {
            int it = tid + k * NT;
            it = it < NQUAD * NL ? it : NQUAD * NL - 1;
            const int qi = it / NL;
            qq[k] = reinterpret_cast<const QuadIdx*>(P.quadq)[qi]; wa[k] = ldg_c(P.quadw + 2 * qi); wa1[k] = ldg_c(P.quadw + 2 * qi + 1);
        }
#pragma unroll
        for (int k = 0; k < QIT; ++k) {
            int it = tid + k * NT;
            it = it < NQUAD * NL ? it : NQUAD * NL - 1;
            const int lane = it % NL;
#pragma unroll
            for (int l = 0; l < LPT; ++l) {
                const int row = lane * LPT + l;
                const cplx<T>* src = P.W + s_wbase[row < nl ? row : nl - 1];
                WRow<T>::load2(src, qq[k].a, ya[k][l], ya1[k][l]);
                WRow<T>::load2(src, qq[k].b, yb[k][l], yb1[k][l]);
            }
        }
#pragma unroll
        for (int k = 0; k < QIT; ++k) {
            const int it = tid + k * NT, lane = it % NL;
            if (it < NQUAD * NL) {
                const bool self = qq[k].a == qq[k].b;
                if (spec_kind != SPEC_NONE) {
#pragma unroll
                    for (int l = 0; l < LPT; ++l) {
                        ya[k][l] = apply_spec(ya[k][l], P.spec, spec_kind, (size_t)qq[k].a); ya1[k][l] = apply_spec(ya1[k][l], P.spec, spec_kind, (size_t)qq[k].a + 1);
                        yb[k][l] = apply_spec(yb[k][l], P.spec, spec_kind, (size_t)qq[k].b); yb1[k][l] = apply_spec(yb1[k][l], P.spec, spec_kind, (size_t)qq[k].b + 1);
                    }
                }
                const Lane<T> A = lane_make(ya[k][0], ya[k][LPT - 1]), A1 = lane_make(ya1[k][0], ya1[k][LPT - 1]);
                const Lane<T> Bn = lane_make(yb[k][0], yb[k][LPT - 1]), B1 = lane_make(yb1[k][0], yb1[k][LPT - 1]);
                Lane<T>* pa = s + (G::slot(qq[k].a) * NL + lane);
                Lane<T>* pb = s + (G::slot(qq[k].b) * NL + lane);
                // bin a with mirror b+1
                Lane<T> c = lconj(B1);
                Lane<T> E = A + c;
                Lane<T> iO = lmi<true>(lmulc(A - c, wa[k]));
                pa[0] = E + iO;
                pb[NL] = lconj(E - iO);
                if (!self) {   // bin a+1 with mirror b
                    c = lconj(Bn);
                    E = A1 + c;
                    iO = lmi<true>(lmulc(A1 - c, wa1[k]));
                    pa[NL] = E + iO;
                    pb[0] = lconj(E - iO);
                }
            }
        }
    }
    __syncthreads();

    if constexpr (NST > 1) {
        lane_stage<G, T, NL, NT, RLAST, RLAST, true>(s, P.f.twst, tid);
        __syncthreads();
        LaneMidInv<G, T, NL, NT, H / R0, 1, Rs...>::run(s, P.f, tid);
    }

    // ---- last inverse stage into the side buffer (row-major, SROW reals per row) ----
    const int SROW = (n + 3) & ~3;
    T* side = reinterpret_cast<T*>(smem_raw + G::smem_bytes());
    const bool want_dot = P.mode == RI_DOT;
    {
        const bool out_lo = is_pow2(R0) && R0 > 1 && (n + 1) / 2 <= H / 2;
        const cplx<T>* tw0 = P.f.twst + P.f.twoff[0];
#pragma unroll 1
        for (int it = tid; it < S0 * NL; it += NT) {
            const int lane = it % NL, j = it / NL;
            cplx<T> w[R0];
            if (NST > 1) lane_twiddles<R0, S0>(w, tw0, j);
            const Lane<T>* base = s + (G::slot(j) * NL + lane);
            Lane<T> v[R0];
#pragma unroll
            for (int r = 0; r < R0; ++r) v[r] = base[r * LEG0];
            if (NST > 1) {
#pragma unroll
                for (int r = 1; r < R0; ++r) v[r] = lmulc(v[r], w[r]);
            }
            lbfly<R0, true, T>(v);
            T* srow0 = side + (size_t)(lane * LPT) * SROW;
            T* srow1 = side + (size_t)(lane * LPT + LPT - 1) * SROW;
            auto put = [&](int r) {
                const int i = 2 * (j + r * S0);
                if (i < SROW) {
                    *reinterpret_cast<cplx<T>*>(srow0 + i) = lane_get(v[r], 0);
                    if (LPT == 2) *reinterpret_cast<cplx<T>*>(srow1 + i) = lane_get(v[r], LPT - 1);
                }
            };
            if (out_lo) {
#pragma unroll
                for (int r = 0; r < R0 / 2; ++r) put(r);
            } else {
#pragma unroll
                for (int r = 0; r < R0; ++r) put(r);
            }
        }
    }
#ifndef HIPGP_EMU
    const bool tma_any = P.vec16_ok && SROW == n;
    const bool tma_out = !want_dot && tma_any;
    const bool tma_dot = want_dot && tma_any;       // fused dot: the rows still leave with ONE bulk store; the warps only read
    if (tma_any) fence_proxy_async();        // this thread's shared-memory writes become visible to the async proxy
#else
    const bool tma_out = false, tma_dot = false;
#endif
    __syncthreads();
#ifndef HIPGP_EMU
    if (tma_out) {      // plain rows: the tile's output rows are one contiguous block -> a single bulk-asynchronous store
        if (tid == 0) bulk_s2g(P.out + (size_t)g0 * n, side, (unsigned)((size_t)nl * n * sizeof(T)));
        return;
    }
    if (tma_dot && tid == 0) bulk_s2g_issue(P.out + (size_t)g0 * n, side, (unsigned)((size_t)nl * n * sizeof(T)));
#endif
    // ---- streaming phase: one warp per row, 16-byte accesses: store (crop) and the fused dot product ----
    {
        constexpr int CH = 16 / (int)sizeof(T);
        constexpr int NW = NT / 32, WPR = NW > NROW ? NW / NROW : 1;
        const bool chunked = P.vec16_ok && (n % CH == 0);
        constexpr int tws = WPR > 1 ? 32 : (H / CH >= 32 ? 32 : (H / CH >= 16 ? 16 : (H / CH >= 8 ? 8 : 4)));
        constexpr int rpw = 32 / tws;
        constexpr int TW = WPR > 1 ? 32 * WPR : tws;
        const int warp = tid >> 5, l32 = tid & 31;
        const int ln = WPR > 1 ? l32 + 32 * (warp % WPR) : l32 % tws;
        constexpr int rstep = WPR > 1 ? NW / WPR : NW * rpw;
        for (int rbase = WPR > 1 ? warp / WPR : warp * rpw; rbase < nl; rbase += rstep) {
            const int row = rbase + (WPR > 1 ? 0 : l32 / tws);
            const bool ractive = row < nl;
            const T* srow = side + (size_t)(ractive ? row : 0) * SROW;
            const size_t off = (size_t)(g0 + (ractive ? row : 0)) * n;
            double acc = 0.0;
            if (!ractive) {
            } else if (chunked) {
                const int nch = n / CH;
                constexpr int BS = 8;
                for (int cb = ln; cb < nch; cb += TW * BS) {
                    Vec16<T> ov[BS];
                    if (want_dot) {
#pragma unroll
                        for (int k = 0; k < BS; ++k) { const int c = cb + TW * k; if (c < nch) ov[k] = ldv_stream((const T*)P.v0 + off + (size_t)c * CH); }
                    }
#pragma unroll
                    for (int k = 0; k < BS; ++k) {
                        const int c = cb + TW * k;
                        if (c < nch) {
                            const Vec16<T> y = *reinterpret_cast<const Vec16<T>*>(srow + c * CH);
                            if (want_dot) {
#pragma unroll
                                for (int e = 0; e < CH; ++e) acc += (double)(y.v[e] * ov[k].v[e]);
                            }
                            if (!tma_dot) stv_stream(P.out + off + (size_t)c * CH, y);
                        }
                    }
                }
            } else if (sizeof(T) == 4 && (n & 1) == 0 && P.vec_ok) {
                // 8-byte chunks: rows of even length that are not a multiple of 4 (N = 2m - 2 outputs of R^T)
                for (int c = ln; c < n / 2; c += TW) {
                    const cplx<T> y = *reinterpret_cast<const cplx<T>*>(srow + 2 * c);
                    if (want_dot) {
                        const cplx<T> ov = ld_stream(reinterpret_cast<const cplx<T>*>((const T*)P.v0 + off + 2 * c));
                        acc += (double)(y.x * ov.x) + (double)(y.y * ov.y);
                    }
                    st_stream(reinterpret_cast<cplx<T>*>(P.out + off + 2 * c), y);
                }
            } else {
                for (int i = ln; i < n; i += TW) {
                    const T y = srow[i];
                    if (want_dot) acc += (double)(y * ld_stream((const T*)P.v0 + off + i));
                    st_stream(P.out + off + i, y);
                }
            }
            if (want_dot) {
                acc = team_sum(acc, WPR > 1 ? 32 : tws);
                if (ractive && (WPR > 1 ? l32 == 0 : ln == 0)) s_part[row * WPR + warp % WPR] = acc;
            }
        }
    }
#ifndef HIPGP_EMU
    if (tma_dot && tid == 0) bulk_s2g_wait();       // the bulk store has read the side buffer
#endif
    if (want_dot) {
        __syncthreads();
        constexpr int WPR2 = (NT / 32) > NROW ? (NT / 32) / NROW : 1;
        if (tid < nl) { double a = 0.0; for (int k = 0; k < WPR2; ++k) a += s_part[tid * WPR2 + k]; P.st.partial[g0 + tid] = a; }
        pcg_finalize(P.st, P.dot_kind, g0, g1, P.nrows, tid, NT);
    }
}

}  // namespace hipgp
