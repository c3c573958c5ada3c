// fast_launch.cuh -- tile configuration and launch code of the specialised kernels (included only by fast_inst.cu).
#pragma once
#include "plan_types.cuh"
#include "fast_kernels.cuh"
#include "cols_blk_kernel.cuh"

namespace hipgp {

constexpr int cfg_min(int a, int b) { return a < b ? a : b; }
constexpr int cfg_max(int a, int b) { return a > b ? a : b; }
constexpr int pow2_floor(int x) { return x <= 1 ? 1 : 2 * pow2_floor(x / 2); }

// Tile configuration of one (dtype, radix list).  Base rule: NL lanes per CTA so that the widest stage gives every one of
// ~256 threads one butterfly and the tile stays near 64 KB; register cap 128 (MINB = CTAs per SM by threads).  The row
// passes then take a QUARTER of that (NLR: many small latency chains per SM), the column pass widens one- and two-lane
// tiles (NLC: wider global segments, shared twiddle loads).  All of it is measured, see profiles/README.md.
template <class T, int... Rs>
struct FastCfg {
    using List = RL<Rs...>;
    static constexpr int Ln = RLInfo<List>::N;
    static constexpr int RMAX = RLMax<List>::value;
    static constexpr int BFN = Ln / RMAX;                       // butterflies per line in the widest stage
    static constexpr int NL0 = pow2_floor(cfg_max(1, cfg_min(256 / cfg_max(BFN, 1), 4096 / Ln)));
    static constexpr int NL = cfg_max(1, cfg_min(16, NL0));
    static constexpr int NT = cfg_min(512, cfg_max(32, (BFN * NL + 31) / 32 * 32));
    static constexpr int MINB = cfg_max(1, 512 / NT);
    static constexpr int LPT = LaneInfo<T>::LPT;
    static constexpr int S0 = Ln / (RLInfo<List>::count ? RLFirst<List>::value : 1);
    // row passes: their tiles are latency chains (stream in, FFT, split, stream out); smaller tiles = more independent
    // chains per SM at the same number of warps
    static constexpr int NLR = cfg_max(1, NL / 4);
    static constexpr int NTR = cfg_min(512, cfg_max(32, (BFN * NLR + 31) / 32 * 32));
    static constexpr int MINBR = cfg_max(1, 512 / NTR);
    // column pass: a single lane per tile would mean 16-byte row segments (half of every 32-byte sector wasted); when the
    // doubled tile and its side buffer still fit one SM, take two lanes and 512 threads (one CTA per SM)
    static constexpr int RLASTv = RLLast<List>::value;
    static constexpr bool WIDEN = (NL == 1) && (RLInfo<List>::count > 1) && ((size_t)(Ln + Ln / RLASTv) * 2 * 24 <= 222 * 1024);
    // ... and two-lane tiles are widened to four lanes (512 threads, one CTA per SM): the per-butterfly twiddle loads are
    // shared by twice as many lines (measured at 2048 points: 183 -> 170 us; wider tiles than that lose again)
    static constexpr int CMULF = 2;
    static constexpr bool CMUL = !WIDEN && NL == 2 && ((size_t)(Ln + Ln / RLASTv) * NL * CMULF * 24 <= 222 * 1024) && BFN * NL * CMULF <= 512;
    static constexpr int NLC = WIDEN ? 2 : (CMUL ? NL * CMULF : NL);
    static constexpr int NTC = (WIDEN || CMUL) ? cfg_min(512, cfg_max(32, (BFN * NLC + 31) / 32 * 32)) : NT;
    static constexpr int MINBC = (WIDEN || CMUL) ? cfg_max(1, 512 / NTC) : MINB;
};

static void launch_check(const char* what, int len, int nl, int nt, size_t smem, long grid) {
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess)
        throw Error(std::string(what) + " launch failed (length " + std::to_string(len) + ", lanes " + std::to_string(nl) + ", threads " + std::to_string(nt) +
                    ", shared " + std::to_string(smem) + " B, grid " + std::to_string(grid) + "): " + cudaGetErrorString(e));
}

// shared memory of a row-pass CTA: the tile, then the side buffer with the tile's real rows (row-major)
template <class T, int... Rs>
static size_t rows_fast_smem(long n_real) {
    using C = FastCfg<T, Rs...>;
    using G = TileGeo<T, C::NLR, Rs...>;
    return G::smem_bytes() + sizeof(T) * (size_t)((n_real + 3) & ~3L) * (C::NLR * C::LPT);
}

template <class T, int... Rs>
static void launch_rows_fast_t(hipgp_plan* pl, bool inverse, RowsParams<T>& P, cudaStream_t st) {
    using C = FastCfg<T, Rs...>;
    using G = TileGeo<T, C::NLR, Rs...>;
    constexpr int NROW = C::NLR * C::LPT;
    static_assert(NROW <= 32, "per-row scalars are held in 32-entry shared arrays");
    P.RB = NROW; P.RBP = NROW;
    {   // the kernels take the pair / quad structure of the digit-reversed order as compile-time facts
        constexpr int NST = G::NST, H = C::Ln;
        const int want_q = NST > 1 ? (H - G::RLAST) / 4 : 0, want_p = NST > 1 ? G::RLAST / 2 + 1 : H / 2 + 1;
        if (P.nquad != want_q || P.npair0 != want_p) throw Error("internal: unexpected r2c pair structure for H = " + std::to_string(H));
    }
    const size_t smem = rows_fast_smem<T, Rs...>(P.n_real);
    if (smem > kRowsFastSmemMax) throw Error("row pass: rows too long for the shared-memory side buffer");
    // operands of a fused update land in the tile buffer: two row blocks must fit in it
    P.tma_op = (!inverse && 2 * sizeof(T) * (size_t)((P.n_real + 3) & ~3) * NROW <= G::smem_bytes()) ? 1 : 0;
    dim3 grid((unsigned)((P.total_rows + NROW - 1) / NROW));
    PROF_BEGIN(pl, inverse ? 2 : 0, st);
    if (inverse) {
        auto k = rows_inv_fast_kernel<T, C::NLR, C::NTR, C::MINBR, Rs...>;
        if (smem > 40 * 1024) HIPGP_SET_MAX_SMEM(k, smem);   // (static shared memory counts against the 48 KB default too)
        HIPGP_LAUNCH(k, grid, dim3(C::NTR), smem, st, P);
    } else {
        auto k = rows_fwd_fast_kernel<T, C::NLR, C::NTR, C::MINBR, Rs...>;
        if (smem > 40 * 1024) HIPGP_SET_MAX_SMEM(k, smem);   // (static shared memory counts against the 48 KB default too)
        HIPGP_LAUNCH(k, grid, dim3(C::NTR), smem, st, P);
    }
    PROF_END(pl, st);
    launch_check("row pass", C::Ln, C::NLR, C::NTR, smem, (long)grid.x);
    pl->launches++;
}

// number of CTAs of `kernel` that fit the device at once (persistent kernels size their grid with this)
template <class K>
static int resident_ctas(K kernel, int nthreads, size_t smem) {
#ifdef HIPGP_EMU
    (void)kernel; (void)nthreads; (void)smem;
    return 3;
#else
    int dev = 0, sms = 0, per = 0;
    CK(cudaGetDevice(&dev));
    CK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per, kernel, nthreads, smem));
    return sms * (per > 0 ? per : 1);
#endif
}

template <class T, int LEN, int... Rs>
static void launch_cols_fast_t(hipgp_plan* pl, ColsParams<T>& P, long n_outer, long B, cudaStream_t st) {
    using C = FastCfg<T, Rs...>;
    using G = TileGeo<T, C::NLC, Rs...>;
    static_assert(C::Ln == LEN, "radix list does not multiply to the length");
    constexpr int TBL = C::NLC * C::LPT;
    P.TB = TBL; P.TBP = TBL;
    // side buffer (8 bytes per lane and padded position): next tile's input rows / this tile's real spectrum
    const size_t side_bytes = G::NST > 1 ? (size_t)(C::Ln + C::Ln / G::RLAST) * C::NLC * 8 : 0;
    P.spec_stage = (G::NST > 1 && P.mode == CM_FUSED && P.spec_kind == SPEC_REAL) ? 1 : 0;
    P.in_stage = (G::NST > 1 && P.mode != CM_INV && (size_t)P.n_in * C::NLC * 16 <= side_bytes) ? 1 : 0;
    const size_t smem = G::smem_bytes() + ((P.spec_stage || P.in_stage) ? side_bytes : 0);
    P.nx = (int)((P.inner + TBL - 1) / TBL); P.ny = (int)n_outer; P.nz = (int)B;
    // tile order: lines fastest keeps neighbouring CTAs on neighbouring 32/64-byte row segments (shared DRAM bursts); but a
    // spectrum that does not stay in L2 would then be re-read from DRAM for every right-hand side, so for big spectra and
    // tiles that are a full 128-byte segment wide the batch index runs fastest instead
    {
        const size_t spec_bytes = (size_t)G::Ln * (size_t)P.inner * (P.spec_kind == SPEC_REAL ? sizeof(T) : 2 * sizeof(T));
        P.batch_fastest = (P.mode == CM_FUSED && B > 1 && spec_bytes > ((size_t)48 << 20) && (size_t)TBL * sizeof(cplx<T>) >= 128) ? 1 : 0;
    }
    auto k = cols_fast_kernel<T, C::NLC, C::NTC, C::MINBC, Rs...>;
    if (smem > 40 * 1024) HIPGP_SET_MAX_SMEM(k, smem);   // (static shared memory counts against the 48 KB default too)
    const long ntiles = (long)P.nx * P.ny * P.nz;
    const long grid = std::min<long>(ntiles, resident_ctas(k, C::NTC, smem));
    PROF_BEGIN(pl, 1, st);
    HIPGP_LAUNCH(k, dim3((unsigned)grid), dim3(C::NTC), smem, st, P);
    PROF_END(pl, st);
    launch_check("column pass", C::Ln, C::NLC, C::NTC, smem, grid);
    pl->launches++;
}

// block-local variant of the column pass for three-stage lists (cols_blk_kernel.cuh); false = not applicable
template <class T, int LEN, int... Rs> struct ColsBlkLaunch {
    static bool run(hipgp_plan*, ColsParams<T>&, long, long, cudaStream_t) { return false; }
};
template <class T, int LEN, int R0, int R1, int R2> struct ColsBlkLaunch<T, LEN, R0, R1, R2> {
    using C = FastCfg<T, R0, R1, R2>;
    using Cfg = ColsBlkCfg<T, C::NLC, C::NTC, C::MINBC, R0, R1, R2>;
    static bool run(hipgp_plan* pl, ColsParams<T>& P, long n_outer, long B, cudaStream_t st) {
        // (measured, profiles/README.md r2c: a gain where the twiddle tables fit next to the tile -- fp32 --, a loss otherwise)
        if constexpr (!Cfg::ok) { (void)pl; (void)P; (void)n_outer; (void)B; (void)st; return false; }
        else {
            if ((long)((P.inner + C::NLC * C::LPT - 1) / (C::NLC * C::LPT)) * n_outer * B >= (1L << 31)) return false;
            using G = typename Cfg::G;
            constexpr int TBL = C::NLC * C::LPT;
            P.TB = TBL; P.TBP = TBL;
            P.spec_stage = (P.mode == CM_FUSED && P.spec_kind == SPEC_REAL) ? 1 : 0;
            P.in_stage = (P.mode != CM_INV && (size_t)P.n_in * C::NLC * 16 <= Cfg::side_bytes) ? 1 : 0;
            const size_t smem = Cfg::smem_bytes;
            P.nx = (int)((P.inner + TBL - 1) / TBL); P.ny = (int)n_outer; P.nz = (int)B;
            {
                const size_t spec_bytes = (size_t)G::Ln * (size_t)P.inner * (P.spec_kind == SPEC_REAL ? sizeof(T) : 2 * sizeof(T));
                P.batch_fastest = (P.mode == CM_FUSED && B > 1 && spec_bytes > ((size_t)48 << 20) && (size_t)TBL * sizeof(cplx<T>) >= 128) ? 1 : 0;
            }
            // TMA staging (tiled tensor maps): input rows when the pass reads a plain [batch][row][bin] array whose rows fill at
            // most half the transform (the tensor's row extent is n_in, so the zero padding is the unit's out-of-bounds fill);
            // the real spectrum tile as one padded box.  Anything else keeps the cp.async staging.
            ColsTmaMaps maps{};
            P.tma_in = P.tma_spec = 0;
            constexpr int HALF = C::Ln / 2;
            const int nbox = (HALF + 255) / 256;
            if (P.in_stage && P.n_in <= HALF && P.in_ostride == 0 && n_outer == 1 && HALF % nbox == 0 && is_pow2(R0)) {
                const unsigned long long dim[3] = {(unsigned long long)(2 * P.pitch), (unsigned long long)P.n_in, (unsigned long long)B};
                const unsigned long long bstr = (unsigned long long)(P.in_bstride ? P.in_bstride : (long)P.n_in * P.pitch);
                const unsigned long long str[2] = {(unsigned long long)P.pitch * sizeof(cplx<T>), bstr * sizeof(cplx<T>)};
                const unsigned box[3] = {(unsigned)(2 * TBL), (unsigned)(HALF / nbox), 1u};
                if (encode_map3(&maps.in, P.in, (int)sizeof(T), dim, str, box)) { P.tma_in = 1; P.tma_in_rows = HALF / nbox; P.tma_in_nbox = nbox; }
            }
            if (P.spec_stage && C::Ln / R2 <= 256 && (TBL * sizeof(T)) % 16 == 0) {
                const long sp = P.spec_pitch ? P.spec_pitch : P.pitch;
                const unsigned long long dim[3] = {(unsigned long long)sp, (unsigned long long)R2, (unsigned long long)(C::Ln / R2)};
                const unsigned long long str[2] = {(unsigned long long)sp * sizeof(T), (unsigned long long)sp * R2 * sizeof(T)};
                const unsigned box[3] = {(unsigned)TBL, (unsigned)(R2 + 1), (unsigned)(C::Ln / R2)};
                if (encode_map3(&maps.spec, P.spec, (int)sizeof(T), dim, str, box)) P.tma_spec = 1;
            }
            auto k = cols_blk_kernel<T, C::NLC, C::NTC, C::MINBC, R0, R1, R2>;
            if (smem > 40 * 1024) HIPGP_SET_MAX_SMEM(k, smem);
            const long ntiles = (long)P.nx * P.ny * P.nz;
            const long grid = std::min<long>(ntiles, resident_ctas(k, C::NTC, smem));
            PROF_BEGIN(pl, 1, st);
            HIPGP_LAUNCH(k, dim3((unsigned)grid), dim3(C::NTC), smem, st, P, maps);
            PROF_END(pl, st);
            launch_check("column pass (block-local)", C::Ln, C::NLC, C::NTC, smem, grid);
            pl->launches++;
            return true;
        }
    }
};

// the lane kernels move 16-byte lanes: pointers and strides must keep every lane aligned
template <class T>
static bool cols_lane_aligned(const ColsParams<T>& P) {
    constexpr long A = 16 / (long)sizeof(cplx<T>);          // complex elements per 16 bytes (2 for fp32, 1 for fp64)
    auto al = [&](long v) { return v % A == 0; };
    return ((uintptr_t)P.in % 16 == 0) && ((uintptr_t)P.out % 16 == 0) && ((uintptr_t)P.spec % 16 == 0) && al(P.pitch) && al(P.in_ostride) &&
           al(P.in_bstride) && al(P.out_ostride) && al(P.out_bstride) && al(P.spec_pitch);
}

template <class T, int LEN> struct FastList;
#define X(LEN, ...)                                                                                         \
    template <class T> struct FastList<T, LEN> {                                                            \
        static void rows(hipgp_plan* pl, bool inv, RowsParams<T>& P, cudaStream_t st) { launch_rows_fast_t<T, __VA_ARGS__>(pl, inv, P, st); } \
        static size_t rows_smem(long n_real) { return rows_fast_smem<T, __VA_ARGS__>(n_real); }                 \
        static void cols(hipgp_plan* pl, ColsParams<T>& P, long no, long B, cudaStream_t st) {         \
            if (!ColsBlkLaunch<T, LEN, __VA_ARGS__>::run(pl, P, no, B, st)) launch_cols_fast_t<T, LEN, __VA_ARGS__>(pl, P, no, B, st); } \
    };
HIPGP_FAST_LIST(X)
#undef X
template <class T, int LEN> void launch_rows_fast_len(hipgp_plan* pl, bool inverse, RowsParams<T>& P, cudaStream_t st) { FastList<T, LEN>::rows(pl, inverse, P, st); }
template <class T, int LEN> bool rows_fast_fits_len(long n_real) { return FastList<T, LEN>::rows_smem(n_real) <= kRowsFastSmemMax; }
template <class T, int LEN> void launch_cols_fast_len(hipgp_plan* pl, ColsParams<T>& P, long n_outer, long B, cudaStream_t st) {
    if (!cols_lane_aligned<T>(P)) throw Error("column pass: pointers / strides are not 16-byte aligned");
    FastList<T, LEN>::cols(pl, P, n_outer, B, st);
}
}  // namespace hipgp
