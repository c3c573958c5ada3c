// cols_blk_kernel.cuh -- column pass for three-stage radix lists (R0, R1, R2) with BLOCK-LOCAL middle sections (round 2).
//
// After the first DIF stage (radix R0, stride S0 = Ln / R0) a line is R0 independent sub-transforms of BS = Ln / R0
// neighbouring positions: the second forward stage, the last forward stage, the spectrum multiply, the first inverse stage
// and the second inverse stage never leave their block of BS positions.  Only the first forward and the last inverse stage
// couple the blocks.  cols_fast_kernel separates ALL stages by CTA barriers, which keeps the 16 warps of an SM in lock step:
// everybody loads, then everybody computes, then everybody stores (ncu, profiles/ncu_full_r1j.json: FMA pipe 42 %, shared-memory
// wavefronts 41 %, and the two do not overlap).  Here block b belongs to the GS = NT / R0 threads [b GS, (b+1) GS) -- one
// warp at 2048 points -- which run the three block-local sections back to back with only a group barrier (__syncwarp when GS
// is 32, a named barrier otherwise): the warps of an SM drift apart and the shared-memory phases of one overlap the
// arithmetic of the others.  CTA barriers per tile: 3 instead of 6.
//   * spectrum staging is block-local too (every group copies and waits for its own BS positions);
//   * the next tile's input rows are prefetched behind the LAST inverse stage (the side buffer holds spectrum until every
//     group has left its block-local sections);
//   * TMA: when the pass reads a plain [batch][row][bin] workspace, the tile's input rows arrive as a few 3-D tensor boxes
//     (cp.async.bulk.tensor, zero fill past the last row = the zero padding of the transform, so the first stage loads
//     without predicates) and the real spectrum tile as ONE box whose middle extent is one larger than the tensor's -- the
//     out-of-bounds row is exactly the bank-conflict padding of the staged layout; one thread issues, an mbarrier completes.
//     (ncu on the cp.async version: the per-thread LDGSTS address registers sat on the long scoreboard, 9 % of all samples.)
//   * per-stage twiddle tables live in shared memory when they fit (fp32): with 209 KB of the SM carved out for shared memory
//     the L1 keeps almost nothing (ncu: 12 % hit rate), so every table load of cols_fast_kernel is an L2 round trip at the
//     head of a section.
// Same math, same digit-reversed layout, same modes as cols_fast_kernel.
#pragma once
#include "fast_kernels.cuh"
#include "tma_maps.cuh"

namespace hipgp {

#ifdef HIPGP_EMU
static inline void nbar_sync(int id, int count) { emu::g_named_barrier[id].sync(count); }
static inline void warp_sync_all() {
    const int tid = (int)(threadIdx.x + blockDim.x * (threadIdx.y + blockDim.y * threadIdx.z));
    emu::g_warp_barrier[tid >> 5].wait();
}
#else
__device__ __forceinline__ void nbar_sync(int id, int count) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory"); }
__device__ __forceinline__ void warp_sync_all() { __syncwarp(); }
#endif

template <int GS> __device__ __forceinline__ void blk_sync(int b) {
    if (GS == 32) warp_sync_all(); else nbar_sync(1 + b, GS);
}

// The SHARED-memory twiddle tables are always PAIRED (fft_engine.cuh: TwPair, one 16-byte load for two fp32 twiddles): single
// 8-byte loads made the tables 28 % of the kernel's shared-memory INSTRUCTIONS.  The global tables are paired in fp32 only.
template <int R, int S, class T>
__device__ __forceinline__ void blk_fill_pairs(TwPair<T>* dst, const cplx<T>* tab, int tid, int nt) {
    for (int i = tid; i < TwPairs<R>::n * S; i += nt) { const int p = i / S; dst[i] = tw_pair_global<R, S, T>(tab, p, i - p * S); }
}
template <int R, int S, bool SM, class T> __device__ __forceinline__ TwPair<T> blk_pair(const cplx<T>* tab, int p, int j) {
    return SM ? reinterpret_cast<const TwPair<T>*>(tab)[p * S + j] : tw_pair_global<R, S, T>(tab, p, j);
}

// twiddles w^{j r}, r = 1..R-1, of a stage: from the shared-memory copy or from global memory
template <int R, int S, bool SM, class T>
__device__ __forceinline__ void blk_twiddles(cplx<T>* w, const cplx<T>* tab, int j) {
#pragma unroll
    for (int p = 0; p < TwPairs<R>::n; ++p) {
        const TwPair<T> e = blk_pair<R, S, SM, T>(tab, p, j);
        w[2 * p + 1] = e.a;
        if (2 * p + 2 < R) w[2 * p + 2] = e.b;
    }
}

// v[r] *= w^{j r} (or its conjugate), r = 1..R-1, with the table loads issued in chunks of CH / 2 pairs: at radix 16 the 15
// twiddles of a butterfly would otherwise all be live next to its 16 lanes (94 of 128 registers) and the kernel spills -- and a
// spill reload is an L2 round trip here, because with 225 KB of the SM carved out for shared memory there is no L1 to speak of.
template <int R, int S, bool SM, bool CONJ, int CH, class T>
__device__ __forceinline__ void blk_twiddle_mul(Lane<T>* v, const cplx<T>* tab, int j) {
    constexpr int PC = CH / 2 > 0 ? CH / 2 : 1;                 // pairs per chunk
#pragma unroll
    for (int p0 = 0; p0 < TwPairs<R>::n; p0 += PC) {
        TwPair<T> e[PC];
#pragma unroll
        for (int c = 0; c < PC; ++c) if (p0 + c < TwPairs<R>::n) e[c] = blk_pair<R, S, SM, T>(tab, p0 + c, j);
#pragma unroll
        for (int c = 0; c < PC; ++c) if (p0 + c < TwPairs<R>::n) {
            const int r = 2 * (p0 + c) + 1;
            v[r] = CONJ ? lmulc(v[r], e[c].a) : lmul(v[r], e[c].a);
            if (r + 1 < R) v[r + 1] = CONJ ? lmulc(v[r + 1], e[c].b) : lmul(v[r + 1], e[c].b);
        }
#ifndef HIPGP_EMU
        if (p0 + PC < TwPairs<R>::n) asm volatile("" ::: "memory");   // keeps the next chunk's loads behind this chunk's arithmetic
#endif
    }
}

template <class T, int NL, int NT, int MINB, int R0, int R1, int R2>
struct ColsBlkCfg {
    using G = TileGeo<T, NL, R0, R1, R2>;
    static constexpr int Ln = G::Ln, BS = Ln / R0, GS = NT / R0;
    static constexpr int IB2 = (BS / R1) * NL, IB3 = (BS / R2) * NL;         // items of one block in the middle / last stage
    static constexpr bool ok = (NT % R0 == 0) && (GS % 32 == 0) && (GS == 32 || R0 <= 15) && (IB2 % GS == 0) && (IB3 % GS == 0) &&
                               ((IB2 / GS) * R1 <= 16) && ((IB3 / GS) * R2 <= 16) && (BS % R2 == 0);
    static constexpr size_t tw_bytes = 2 * sizeof(cplx<T>) * (size_t)((R0 / 2) * (Ln / R0) + (R1 / 2) * (BS / R1));   // pairs
    static constexpr size_t side_bytes = (size_t)(Ln + Ln / R2) * NL * 8;
    // (MINB resident CTAs per SM must keep fitting: 228 KB per SM, 1 KB reserved per CTA)
    static constexpr bool tw_smem = (size_t)MINB * (G::smem_bytes() + side_bytes + tw_bytes + 1024) <= 228 * 1024;
    static constexpr size_t smem_bytes = G::smem_bytes() + side_bytes + (tw_smem ? tw_bytes : 0);
};

template <class T, int NL, int NT, int MINB, int R0, int R1, int R2>
__global__ void __launch_bounds__(NT, MINB) cols_blk_kernel(const HIPGP_GRID_CONSTANT ColsParams<T> P, const HIPGP_GRID_CONSTANT ColsTmaMaps maps) {
    using Cfg = ColsBlkCfg<T, NL, NT, MINB, R0, R1, R2>;
    using G = typename Cfg::G;
    constexpr int Ln = G::Ln, RLAST = R2, LPT = LaneInfo<T>::LPT, TBL = NL * LPT, S0 = Ln / R0;
    constexpr int BS = Cfg::BS, GS = Cfg::GS, S1 = BS / R1;
    constexpr bool TWS = Cfg::tw_smem;
    constexpr int TWCH = R0 >= 16 ? 5 : R0;                      // twiddle loads per chunk in the first / last stage
    static_assert(Cfg::ok, "radix list / tile shape not usable with block-local middle sections");
    constexpr int LEG0 = G::leg(S0), LEG1 = G::leg(S1);
    constexpr int SPEC_LANE = 8;                                  // bytes of real spectrum per lane (2 x fp32 or 1 x fp64)
    constexpr int SIDE_SLOTS = Ln + Ln / RLAST;
    constexpr int SIDE_LANES = SIDE_SLOTS * NL / 2;
    HIPGP_DYN_SMEM(smem_raw);
    Lane<T>* s = reinterpret_cast<Lane<T>*>(smem_raw);
    unsigned char* side = smem_raw + G::smem_bytes();
    const int tid = threadIdx.x;
    if (P.done_flag && *P.done_flag) return;
    const int blk = tid / GS, u = tid - blk * GS;                 // this thread's block of BS positions / its rank in the group

    // per-stage twiddle tables: shared-memory copies (persistent kernel: filled once per CTA)
    const cplx<T>* tw0 = P.f.twst + P.f.twoff[0];
    const cplx<T>* tw1 = P.f.twst + P.f.twoff[1];
    __shared__ unsigned long long s_bar[3];                       // [0] input rows, [1] spectrum tile (TMA completion), [2] "every warp has read its spectrum rows"
    const bool tma_in = P.tma_in != 0, tma_spec = P.tma_spec != 0;
    if ((tma_in || tma_spec) && tid == 0) { tma_bar_init(&s_bar[0]); tma_bar_init(&s_bar[1]); warps_bar_init(&s_bar[2], NT / 32); tma_fence_before_issue(); }
    if (tma_in || tma_spec) __syncthreads();
    if (TWS) {
        TwPair<T>* t0 = reinterpret_cast<TwPair<T>*>(side + Cfg::side_bytes);
        TwPair<T>* t1 = t0 + TwPairs<R0>::n * S0;
        blk_fill_pairs<R0, S0, T>(t0, tw0, tid, NT);
        blk_fill_pairs<R1, S1, T>(t1, tw1, tid, NT);
        tw0 = reinterpret_cast<const cplx<T>*>(t0); tw1 = reinterpret_cast<const cplx<T>*>(t1);
        __syncthreads();
    }

    const int mode = P.mode;
    const size_t pitch = (size_t)P.pitch;
    const size_t spitch = P.spec_pitch ? (size_t)P.spec_pitch : (size_t)P.pitch;
    const long ntiles = (long)P.nx * P.ny * P.nz;
    // (32-bit tile arithmetic: the launcher guarantees ntiles < 2^31; 64-bit divisions cost ~100 instructions per thread and tile)
    unsigned tile_bz = 0;                                          // batch index of the tile tile_origin() was last asked about
    auto tile_origin = [&](long t, long& c0, size_t& ioff, size_t& ooff) {
        const unsigned tt = (unsigned)t, nx = (unsigned)P.nx, ny = (unsigned)P.ny, nz = (unsigned)P.nz;
        unsigned bx, by, bz;
        if (P.batch_fastest) { bz = tt % nz; const unsigned r = tt / nz; bx = r % nx; by = r / nx; }
        else { bx = tt % nx; const unsigned r = tt / nx; by = r % ny; bz = r / ny; }
        c0 = (long)bx * TBL;
        tile_bz = bz;
        ioff = (size_t)by * P.in_ostride + (size_t)bz * P.in_bstride + c0;
        ooff = (size_t)by * P.out_ostride + (size_t)bz * P.out_bstride + c0;
    };
    auto sslot = [](int p) { return p + (p >> G::LOGRL); };       // padded position of the staged spectrum
    const bool spec_smem = P.spec_stage != 0;
    const int n_in = P.n_in, n_out = P.n_out;
    const bool stage_in = P.in_stage != 0;
    const bool zero_hi = is_pow2(R0) && n_in <= Ln / 2;
    const bool out_lo = is_pow2(R0) && n_out <= Ln / 2;
    const size_t rstep = (size_t)S0 * pitch;

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

    // TMA version of the same: boxes of tma_in_rows rows x TBL bins of batch entry bz, dense in the side buffer (row i at
    // lane i * NL); rows >= n_in are outside the tensor and arrive as zeros.  Called by ONE thread.
    auto issue_input = [&](long t) {
        long c0; size_t ioff, ooff;
        tile_origin(t, c0, ioff, ooff);
        const unsigned box_bytes = (unsigned)P.tma_in_rows * NL * 16u;
        tma_fence_before_issue();
        tma_bar_expect(&s_bar[0], box_bytes * (unsigned)P.tma_in_nbox);
        for (int k = 0; k < P.tma_in_nbox; ++k)
            tma_load_box3(side + (size_t)k * box_bytes, &maps.in, (int)(2 * c0), k * P.tma_in_rows, (int)tile_bz, &s_bar[0]);
    };
    auto stage_next = [&](long tn) {
        if (tn >= ntiles) return;
        if (tma_in) { if (tid == 0) issue_input(tn); }
        else if (stage_in) prefetch_input(tn);
    };

    stage_next((long)blockIdx.x);
    // (the mbarrier phases are the parity of the tile iteration: both barriers complete exactly once per tile)
    for (unsigned iter = 0;; ++iter) {
        const long t = (long)blockIdx.x + (long)iter * gridDim.x;
        if (t >= ntiles) break;
        const unsigned ph = iter & 1u;
        long c0; size_t ioff, ooff;
        tile_origin(t, c0, ioff, ooff);
        const long nvalid = P.inner - c0;
        const cplx<T>* in = P.in + ioff;
        cplx<T>* out = P.out + ooff;
        // This tile's input must have landed.  The previous tile's last inverse stage and this tile's first forward stage touch
        // the SAME tile-buffer slots from the SAME thread (item (lane, j) reads / writes positions j + r S0), so nothing but
        // program order is needed between them: with TMA staging (every thread waits on the mbarrier itself) there is no CTA
        // barrier here and the warps run from one tile's last stage straight into the next tile's first stage.
        // (Forward-only passes end a tile in the block-local last forward stage, a different thread-to-slot mapping: barrier.)
        if (tma_in) { tma_bar_wait(&s_bar[0], ph, 8, NT); if (mode != CM_FUSED) __syncthreads(); }
        else { cp_async_wait_all(); __syncthreads(); }

        if (mode != CM_INV) {
            // ---- first forward stage (couples the blocks): operands from the side buffer or from global memory ----
#pragma unroll 1
            for (int it = tid; it < S0 * NL; it += NT) {
                const int lane = it % NL, j = it / NL;
                const bool ok = (long)lane * LPT < nvalid;
                Lane<T> v[R0];
                if (tma_in) {        // rows past n_in were zero-filled by the TMA unit; lanes past the last line carry padding bins
                    const Lane<T>* sp = reinterpret_cast<const Lane<T>*>(side) + (j * NL + lane);
#pragma unroll
                    for (int r = 0; r < R0 / 2; ++r) v[r] = sp[r * S0 * NL];
                    lbfly_zero_hi<R0, T>(v);
                } else if (stage_in) {
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
                blk_twiddle_mul<R0, S0, TWS, false, TWCH>(v, tw0, j);
                Lane<T>* base = s + (G::slot(j) * NL + lane);
#pragma unroll
                for (int r = 0; r < R0; ++r) base[r * LEG0] = v[r];
            }
            __syncthreads();
            // passes that stage no spectrum leave the side buffer idle from here on: the next tile's input rows start right away
            if (!(mode == CM_FUSED && spec_smem)) stage_next(t + gridDim.x);
        }

        // ======== block-local sections: group `blk` owns positions [blk BS, (blk + 1) BS) of every lane of the tile ========
        const int pb = blk * BS;
        if (mode == CM_FUSED && spec_smem && tma_spec) {
            // the whole real spectrum tile as ONE padded box (the out-of-bounds 17th row of every group of 16 positions is the
            // bank-conflict padding of the staged layout) -> side buffer (free now), behind the second forward stage
            if (tid == 0) {
                tma_fence_before_issue();
                tma_bar_expect(&s_bar[1], (unsigned)Cfg::side_bytes);
                tma_load_box3(side, &maps.spec, (int)c0, 0, 0, &s_bar[1]);
            }
        } else if (mode == CM_FUSED && spec_smem) {
            // this block's rows of the real spectrum tile -> side buffer (free now), behind the second forward stage
            const unsigned char* sp = reinterpret_cast<const unsigned char*>(P.spec) + (size_t)c0 * sizeof(T);
            constexpr int ROWB = NL * SPEC_LANE;
            constexpr int CH = ROWB >= 16 ? 16 : 8, NCH = ROWB / CH;
            constexpr int NIT = (BS * NCH + GS - 1) / GS;
#pragma unroll
            for (int k = 0; k < NIT; ++k) {
                const int w = u + k * GS;
                const int p = pb + w / NCH, c = w % NCH;
                if (w < BS * NCH) cp_async<CH>(side + (size_t)sslot(p) * ROWB + c * CH, sp + (size_t)p * spitch * sizeof(T) + c * CH);
            }
            cp_async_commit();
        }
        if (mode != CM_INV) {
            // ---- second forward stage: radix R1 inside the block ----
            constexpr int NIT = Cfg::IB2 / GS;
            Lane<T> v[NIT][R1];
            cplx<T> w[NIT][R1];
            Lane<T>* base[NIT];
#pragma unroll
            for (int k = 0; k < NIT; ++k) {
                const int q = u + k * GS;
                const int lane = q % NL, j = q / NL;
                base[k] = s + (G::slot(pb + j) * NL + lane);
                blk_twiddles<R1, S1, TWS>(w[k], tw1, j);
#pragma unroll
                for (int r = 0; r < R1; ++r) v[k][r] = base[k][r * LEG1];
            }
#pragma unroll
            for (int k = 0; k < NIT; ++k) {
                lbfly<R1, false, T>(v[k]);
#pragma unroll
                for (int r = 1; r < R1; ++r) v[k][r] = lmul(v[k][r], w[k][r]);
#pragma unroll
                for (int r = 0; r < R1; ++r) base[k][r * LEG1] = v[k][r];
            }
            if (mode == CM_FUSED && spec_smem) {
                if (tma_spec) tma_bar_wait(&s_bar[1], ph, 9, NT);
                else cp_async_wait_all();
            }
            blk_sync<GS>(blk);
        }
        // ---- last forward stage + spectrum + first inverse stage: RLAST neighbouring positions, in registers ----
        {
            constexpr int NIT = Cfg::IB3 / GS;
#pragma unroll
            for (int k = 0; k < NIT; ++k) {
                const int q = u + k * GS;
                const int lane = q % NL;
                const bool ok = (long)lane * LPT < nvalid;
                const int p0 = pb + (q / NL) * RLAST;
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
        }
        if (mode == CM_FWD) continue;
        // the side buffer held the spectrum: once EVERY warp is through the multiply it is free, and the next tile's input rows can
        // start travelling behind the second inverse stage already (one lane per warp arrives, thread 0 waits and issues)
        const bool early_in = tma_in && mode == CM_FUSED && spec_smem;
        if (early_in) {
            warp_sync_all();                                  // every lane of this warp is done with its spectrum rows
            if (tid == 0) { warps_bar_arrive_and_wait(&s_bar[2], ph, 10, NT / 32); stage_next(t + gridDim.x); }
            else if ((tid & 31) == 0) warps_bar_arrive(&s_bar[2], 10, NT / 32);
        }
        blk_sync<GS>(blk);
        // ---- second inverse stage: radix R1 inside the block ----
        {
            constexpr int NIT = Cfg::IB2 / GS;
            Lane<T> v[NIT][R1];
            cplx<T> w[NIT][R1];
            Lane<T>* base[NIT];
#pragma unroll
            for (int k = 0; k < NIT; ++k) {
                const int q = u + k * GS;
                const int lane = q % NL, j = q / NL;
                base[k] = s + (G::slot(pb + j) * NL + lane);
                blk_twiddles<R1, S1, TWS>(w[k], tw1, j);
#pragma unroll
                for (int r = 0; r < R1; ++r) v[k][r] = base[k][r * LEG1];
            }
#pragma unroll
            for (int k = 0; k < NIT; ++k) {
#pragma unroll
                for (int r = 1; r < R1; ++r) v[k][r] = lmulc(v[k][r], w[k][r]);
                lbfly<R1, true, T>(v[k]);
#pragma unroll
                for (int r = 0; r < R1; ++r) base[k][r * LEG1] = v[k][r];
            }
        }
        __syncthreads();
        // ---- every group is done with its spectrum rows: next tile's input rows travel behind the last inverse stage ----
        if (mode == CM_FUSED && spec_smem && !early_in) stage_next(t + gridDim.x);
        // ---- last inverse stage (couples the blocks) straight to global memory (crop = skipped stores) ----
        {
#pragma unroll 1
            for (int it = tid; it < S0 * NL; it += NT) {
                const int lane = it % NL, j = it / NL;
                const bool ok = (long)lane * LPT < nvalid;
                const Lane<T>* base = s + (G::slot(j) * NL + lane);
                Lane<T> v[R0];
#pragma unroll
                for (int r = 0; r < R0; ++r) v[r] = base[r * LEG0];
                blk_twiddle_mul<R0, S0, TWS, true, TWCH>(v, tw0, j);
                // (one 64-bit base per thread, 32-bit element offsets for the R0 / 2 row blocks: an embedded line spans < 2^31 elements)
                cplx<T>* gp = out + (size_t)((unsigned)j * (unsigned)P.pitch + (unsigned)(lane * LPT));
                const unsigned rs = (unsigned)S0 * (unsigned)P.pitch;
                if (out_lo) {
                    // the cropped result keeps at most the lower half of the line: the butterfly sits INSIDE the branch so that
                    // the arithmetic feeding only outputs R0/2 .. R0-1 is dead code here
                    lbfly<R0, true, T>(v);
                    if (ok) {
#pragma unroll
                        for (int r = 0; r < R0 / 2; ++r) if (j + r * S0 < n_out) lane_to_global(gp + (size_t)((unsigned)r * rs), v[r]);
                    }
                } else {
                    lbfly<R0, true, T>(v);
                    if (ok) {
#pragma unroll
                        for (int r = 0; r < R0; ++r) if (j + r * S0 < n_out) lane_to_global(gp + (size_t)((unsigned)r * rs), v[r]);
                    }
                }
            }
        }
    }
}

}  // namespace hipgp
