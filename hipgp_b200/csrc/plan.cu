// plan.cu -- host side of libhipgp_b200: plan construction, spectrum set-up, matvec pipelines, PCG
// driver and the C ABI (include/hipgp_b200.h).
#include "plan_types.cuh"
#include "setup_kernels.cuh"
#include "kxu_kernels.cuh"
#include "long1d_kernels.cuh"

namespace hipgp {
thread_local std::string g_err;
}

namespace hipgp {

template <class T> struct Tag {};
static Geom<float>& geom(hipgp_plan* p, bool wide, Tag<float>) { return wide ? p->gw32 : p->gn32; }
static Geom<double>& geom(hipgp_plan* p, bool wide, Tag<double>) { return wide ? p->gw64 : p->gn64; }

template <class T> static size_t rows_smem(int H, int RBP) { return sizeof(cplx<T>) * (size_t)(H + 1) * RBP; }

template <class T>
static void pick_rows_tiling(long total_rows, int H, int* RB, int* RBP, int* nthreads) {
    int rb = 8;
    while (rb > 1 && (rows_smem<T>(H, rb + 1) > 96 * 1024 || total_rows < (long)rb * 148)) rb >>= 1;
    if (rows_smem<T>(H, rb + 1) > HIPGP_ROW_SMEM_MAX) throw Error("row axis too long for the shared-memory FFT (L = " + std::to_string(2 * H) + ")");
    *RB = rb; *RBP = rb == 1 ? 1 : rb + 1;
    long work = (long)H * rb / 8;
    *nthreads = work >= 256 ? 256 : (work >= 128 ? 128 : (work >= 64 ? 64 : 32));
}

// Does the row pass take a row of H complex bins in rows of up to n_real samples?  The specialised kernels need their tile
// plus a side buffer of the real rows, the generic kernel two padded rows (pick_rows_tiling).
template <class T>
static bool row_pass_fits(int H, long n_real) {
    switch (H) {
#define X(LEN, ...) case LEN: return rows_fast_fits_len<T, LEN>(n_real);
        HIPGP_FAST_LIST(X)
#undef X
        default: return rows_smem<T>(H, 2) <= HIPGP_ROW_SMEM_MAX;
    }
}
// ... for every pass of a 1-D embedding of length L: the matvecs (rows of up to n_max samples, plan dtype) and the fp64
// set-up forward of the whole embedding (build_spectrum)
template <class T>
static bool row_embedding_fits(int L, long n_max) { return row_pass_fits<T>(L / 2, n_max) && row_pass_fits<double>(L / 2, L); }

// the four-step path of long last axes (long1d_api.inl)
template <class T> static LongGeom<T>& long_geom(hipgp_plan* pl, int which);
template <class T> static void long_conv(hipgp_plan* pl, LongGeom<T>& g, Geom<T>& cg, const T* in, const int* n_in, T* out, const int* n_out,
                                         const void* spec, int kind, long B, const int* done, cudaStream_t s);
static void long_dct1(hipgp_plan* pl, const double* in, double* out, bool normalise, cudaStream_t s);
template <class T> static void long_pcg_begin(hipgp_plan* pl, const PcgDev& st, long B, bool precond, cudaStream_t s);
template <class T> static void long_pcg_iterate(hipgp_plan* pl, const PcgDev& st, int niter, cudaStream_t s);
// what the entry points that need the row-pass layout (gradients, slab decomposition) say when they refuse such a plan
static std::string four_step_plans(const hipgp_plan* pl) {
    return pl->D == 1 ? "long 1-D plans (grids too long for the one-block row pass)"
                      : "grids whose last axis is too long for the one-block row pass (four-step path)";
}

template <class T> static bool aligned2(const void* p) { return ((uintptr_t)p % (2 * sizeof(T))) == 0; }

template <class T>
static bool launch_rows_fast(hipgp_plan* pl, bool inverse, RowsParams<T>& P, cudaStream_t st) {
    switch (P.H) {
#define X(LEN, ...) case LEN: launch_rows_fast_len<T, LEN>(pl, inverse, P, st); return true;
        HIPGP_FAST_LIST(X)
#undef X
        default: return false;
    }
}

template <class T>
static void launch_rows(hipgp_plan* pl, const Geom<T>& g, bool inverse, RowsParams<T>& P, cudaStream_t st) {
    P.vec_ok = (aligned2<T>(P.in) && aligned2<T>(P.out) && aligned2<T>(P.v0) && aligned2<T>(P.v1) && aligned2<T>(P.v2)) ? 1 : 0;
    {
        auto a16 = [](const void* q) { return ((uintptr_t)q % 16) == 0; };
        P.vec16_ok = (a16(P.in) && a16(P.out) && a16(P.v0) && a16(P.v1) && a16(P.v2)) ? 1 : 0;
    }
    if (g.fast && launch_rows_fast<T>(pl, inverse, P, st)) return;
    int nth;
    pick_rows_tiling<T>(P.total_rows, P.H, &P.RB, &P.RBP, &nth);
    const size_t smem = rows_smem<T>(P.H, P.RBP);
    dim3 grid((unsigned)((P.total_rows + P.RB - 1) / P.RB));
    PROF_BEGIN(pl, inverse ? 2 : 0, st);
    if (inverse) {
        auto k = rows_inv_kernel<T>;
        if (smem > 48 * 1024) HIPGP_SET_MAX_SMEM(k, smem);
        HIPGP_LAUNCH(k, grid, dim3(nth), smem, st, P);
    } else {
        auto k = rows_fwd_kernel<T>;
        if (smem > 48 * 1024) HIPGP_SET_MAX_SMEM(k, smem);
        HIPGP_LAUNCH(k, grid, dim3(nth), smem, st, P);
    }
    PROF_END(pl, st);
    CK_LAUNCH();
    pl->launches++;
}

template <class T>
static bool launch_cols_fast(hipgp_plan* pl, ColsParams<T>& P, long n_outer, long B, cudaStream_t st) {
    switch (P.f.Ln) {
#define X(LEN, ...) case LEN: launch_cols_fast_len<T, LEN>(pl, P, n_outer, B, st); return true;
        HIPGP_FAST_LIST(X)
#undef X
        default: return false;
    }
}

template <class T>
static void launch_cols(hipgp_plan* pl, const Geom<T>& g, ColsParams<T>& P, long n_outer, long B, cudaStream_t st) {
    if (g.fast && launch_cols_fast<T>(pl, P, n_outer, B, st)) return;
    const int L = P.f.Ln;
    int tb = sizeof(T) == 4 ? 16 : 8;
    while (tb > 1 && sizeof(cplx<T>) * (size_t)L * (tb + 1) > 100 * 1024) tb >>= 1;
    while (tb > 1 && (long)tb > P.inner) tb >>= 1;
    const int tbp = tb == 1 ? 1 : tb + 1;
    const size_t smem = sizeof(cplx<T>) * (size_t)L * tbp;
    if (smem > 220 * 1024) throw Error("grid axis too long for the shared-memory FFT (L = " + std::to_string(L) + ")");
    P.TB = tb; P.TBP = tbp;
    long work = (long)L * tb / 8;
    int nth = work >= 512 ? 512 : (work >= 256 ? 256 : (work >= 128 ? 128 : (work >= 64 ? 64 : 32)));
    dim3 grid((unsigned)((P.inner + tb - 1) / tb), (unsigned)n_outer, (unsigned)B);
    auto k = cols_pass_kernel<T>;
    if (smem > 48 * 1024) HIPGP_SET_MAX_SMEM(k, smem);
    PROF_BEGIN(pl, 1, st);
    HIPGP_LAUNCH(k, grid, dim3(nth), smem, st, P);
    PROF_END(pl, st);
    CK_LAUNCH();
    pl->launches++;
}

static PcgDev null_state() { PcgDev st{}; return st; }
static RowsFusion plain_in(const void* in) { RowsFusion f; f.mode = RF_PLAIN; f.in = in; return f; }
static RowsFusion plain_out(void* out) { RowsFusion f; f.mode = RI_PLAIN; f.out = out; return f; }

// One row pass over B batch entries of `nrows` rows each.  Forward: real rows of n_real samples (f.in, or the operands of
// the fused update f) -> half spectra in W.  Inverse: W -> real rows of n_real samples (f.out, f.v0), after applying the
// 1-D spectrum `spec` when there is one.  Batch entry b owns W_rows >= nrows rows of W, g.P complex elements each.
template <class T>
static void run_rows(hipgp_plan* pl, Geom<T>& g, bool inverse, long nrows, cplx<T>* W, long W_rows, long B, int n_real,
                     const RowsFusion& f, const PcgDev& st, cudaStream_t s, const void* spec = nullptr, int spec_kind = SPEC_NONE) {
    RowsParams<T> R{};
    R.L = g.L[g.D - 1]; R.H = g.H; R.W_pitch = g.P;
    R.f = g.frow.dev; R.twL = g.twL.template as<cplx<T>>(); R.twLp = g.twLp.template as<cplx<T>>();
    R.part = g.part.template as<int>(); R.pairq = g.pairq.template as<int>();
    R.pairs = g.pairs.template as<int>(); R.pairw = g.pairw.template as<cplx<T>>(); R.npair0 = g.npair0;
    R.quadq = g.quadq.template as<int>(); R.quadw = g.quadw.template as<cplx<T>>(); R.nquad = g.nquad;
    R.in = (const T*)f.in; R.out = (T*)f.out; R.v0 = (T*)f.v0; R.v1 = (T*)f.v1; R.v2 = (const T*)f.v2;
    R.mode = f.mode; R.dot_kind = f.dot_kind; R.do_fft = 1; R.st = st; R.spec = spec; R.spec_kind = spec_kind;
    R.W = W; R.W_rows = (int)W_rows; R.total_rows = B * nrows; R.nrows = (int)nrows; R.n_real = n_real;
    launch_rows<T>(pl, g, inverse, R, s);
}

// A buffer of the column passes: batch entries `bstride` complex elements apart, each holding n[0] (x n[1]) rows along
// the leading axes, row-major.
template <class T> struct ColBuf { cplx<T>* p; long bstride; const int* n; };

// The column passes of the leading D - 1 axes from src to dst, over B batch entries of rows of `pitch` complex elements
// whose first `bins` are transformed.  chain CM_FWD: forward, src zero-padded to L, dst holds all L[0] (x L[1]) rows;
// CM_INV: inverse, src holds all L rows (and is overwritten), dst gets its own extents; CM_FUSED: forward, times `spec` on
// axis 0, inverse (3-D: through W2[b][max n0][L1][pitch]).  done: optional PCG early-exit flag.
template <class T>
static void run_cols(hipgp_plan* pl, Geom<T>& g, int chain, const ColBuf<T>& src, const ColBuf<T>& dst, long pitch, long bins,
                     long B, const void* spec, int spec_kind, const int* done, cudaStream_t s) {
    if (g.D == 1) return;
    const long plane = (long)g.L[1] * pitch;      // 3-D: an [L1][pitch] plane, the lines of the axis-0 pass
    auto pass = [&](int axis, int mode, const ColBuf<T>& in, const ColBuf<T>& out) {
        const bool rows = axis == g.D - 2;
        ColsParams<T> C{};
        C.in = in.p; C.out = out.p; C.f = g.fcol[axis].dev; C.mode = mode; C.done_flag = done;
        C.n_in = (mode == CM_INV ? dst : src).n[axis]; C.n_out = (mode == CM_FWD ? src : dst).n[axis];
        C.inner = rows ? bins : plane; C.pitch = rows ? pitch : plane;
        C.in_bstride = in.bstride; C.out_bstride = out.bstride;
        if (axis == 1) { C.in_ostride = in.n[1] * pitch; C.out_ostride = out.n[1] * pitch; }
        if (mode == CM_FUSED) { C.spec = spec; C.spec_kind = spec_kind; }
        launch_cols<T>(pl, g, C, axis == 1 ? (mode == CM_FWD ? src : dst).n[0] : 1, B, s);
    };
    if (g.D == 2) { pass(0, chain, src, dst); return; }
    // 3-D: axis 1 forward into a buffer of L1 rows per plane, axis 0 in place on it, axis 1 inverse out of it
    ColBuf<T> mid = chain == CM_FWD ? dst : src;
    const int mid_n[2] = {std::max(src.n[0], dst.n[0]), g.L[1]};
    if (chain == CM_FUSED) {
        pl->W2.ensure(sizeof(cplx<T>) * (size_t)(B * mid_n[0] * plane), &pl->dev_bytes);
        mid = {pl->W2.as<cplx<T>>(), mid_n[0] * plane, mid_n};
    }
    if (chain != CM_INV) pass(1, CM_FWD, src, mid);
    pass(0, chain, mid, mid);
    if (chain != CM_FWD) pass(1, CM_INV, mid, dst);
}

// The pruned D-dimensional circular convolution:  out = crop_{n_out} IFFT( spec * FFT pad_{n_in} in ).
template <class T>
static void run_pipeline(hipgp_plan* pl, Geom<T>& g, const int* n_in, const int* n_out, const void* spec, int spec_kind,
                         long B, const RowsFusion& ff, const RowsFusion& fi, const PcgDev& st, bool gated, cudaStream_t s) {
    const int D = g.D;
    long rows_in = 1, rows_out = 1;
    for (int d = 0; d + 1 < D; ++d) { rows_in *= n_in[d]; rows_out *= n_out[d]; }
    const long Wrows = std::max(rows_in, rows_out);
    pl->W1.ensure(sizeof(cplx<T>) * (size_t)(B * Wrows * g.P), &pl->dev_bytes);
    cplx<T>* W1 = pl->W1.as<cplx<T>>();
    run_rows<T>(pl, g, false, rows_in, W1, Wrows, B, n_in[D - 1], ff, st, s);
    run_cols<T>(pl, g, CM_FUSED, {W1, Wrows * g.P, n_in}, {W1, Wrows * g.P, n_out}, g.P, g.H + 1, B, spec, spec_kind,
                gated ? st.flags : nullptr, s);
    // the inverse pass's alignment flags (vec_ok, vec16_ok) cover the forward pass's operands too
    RowsFusion fo = fi;
    fo.in = ff.in; fo.v1 = ff.v1; fo.v2 = ff.v2;
    run_rows<T>(pl, g, true, rows_out, W1, Wrows, B, n_out[D - 1], fo, st, s, D == 1 ? spec : nullptr, D == 1 ? spec_kind : SPEC_NONE);
}

// cos(pi t / (m-1)), t in [0, 2(m-1)), per active axis: built once per plan (the grid never changes), no per-call copies
static const double* axis_costab(hipgp_plan* pl, int d) {
    DevBuf& b = pl->costabs[d];
    if (!b.p) {
        const int md = pl->m[d];
        const int Nn = md > 1 ? 2 * (md - 1) : 1;
        std::vector<double> tab(Nn);
        for (int t = 0; t < Nn; ++t) tab[t] = md > 1 ? std::cos(M_PI * (double)t / (double)(md - 1)) : 1.0;
        b.ensure(sizeof(double) * Nn, &pl->dev_bytes);
        CK(cudaMemcpy(b.p, tab.data(), sizeof(double) * Nn, cudaMemcpyHostToDevice));
    }
    return b.as<double>();
}

// the parity-split weighted cosine matrix of an axis (m <= 2048: at most 16 MB), built once per plan on the caller's stream
static const double* axis_cosmat(hipgp_plan* pl, int d, cudaStream_t s) {
    const int md = pl->m[d];
    if (md > 2048) return nullptr;
    DevBuf& b = pl->cosmats[d];
    if (!b.p) {
        const double* tab = axis_costab(pl, d);
        const size_t h = (size_t)(md + 1) / 2;
        b.ensure(sizeof(double) * 2 * h * h, &pl->dev_bytes);              // parity-split: Cw2[p][j < h][k' < h]
        auto k = dct1_cosmat_sym_kernel;
        HIPGP_LAUNCH(k, dim3((unsigned)std::min<size_t>(148 * 4, (2 * h * h + 255) / 256)), dim3(256), 0, s, tab, b.as<double>(), md);
        CK_LAUNCH(); pl->launches++;
    }
    return b.as<double>();
}

// dct1_tile_kernel forms the cosine index (j k) mod N in 32-bit unsigned arithmetic
static void dct1_tile_check(int md) {
    if (md > 65536) throw Error("DCT-I set-up: an axis of " + std::to_string(md) + " points is beyond the tiled kernel (at most 65536)");
}

static void dct_all_axes(hipgp_plan* pl, const double* in, double* out, double* tmp, bool normalise, cudaStream_t s) {
    // separable DCT-I over the active axes; result always lands in `out`
    const double* src = in;
    const int D = pl->D;
    double* bufs[2] = {out, tmp};
    int which = (D % 2 == 1) ? 0 : 1;   // so that the last axis writes `out`
    for (int d = 0; d < D; ++d) {
        const int md = pl->m[d];
        long inner = 1, outer = 1;
        for (int e = d + 1; e < D; ++e) inner *= pl->m[e];
        for (int e = 0; e < d; ++e) outer *= pl->m[e];
        const double* tab = axis_costab(pl, d);
        const int Nn = md > 1 ? 2 * (md - 1) : 1;
        double* dst = bufs[which];
        const double scale = normalise ? 1.0 / (double)Nn : 1.0;
        if (inner == 1) {
            dim3 grid((unsigned)((md + 63) / 64), (unsigned)((outer + 127) / 128), 1);      // 128 x 64 output tile per block
            const double* cw = md > 2 ? axis_cosmat(pl, d, s) : nullptr;
            if (cw) {      // reflection symmetry folded in: two half-size products, one per output parity (grid.z)
                const int hk0 = (md + 1) / 2;
                dim3 gs((unsigned)((hk0 + 63) / 64), (unsigned)((outer + 127) / 128), 2);
                auto k = dct1_sym_kernel<true>; HIPGP_LAUNCH(k, gs, dim3(256), 0, s, src, dst, cw, md, inner, outer, scale, 0);
            } else { dct1_tile_check(md); auto k = dct1_tile_kernel<true>; HIPGP_LAUNCH(k, grid, dim3(256), 0, s, src, dst, tab, md, inner, outer, scale); }
        } else {
            // grid.z = outer index (<= 65535 for every supported grid: at most two leading axes of a 3-D grid)
            if (outer > 65535) throw Error("DCT set-up: more than 65535 outer slices");
            dim3 grid((unsigned)((inner + 63) / 64), (unsigned)((md + 127) / 128), (unsigned)outer);
            const double* cw = md > 2 ? axis_cosmat(pl, d, s) : nullptr;
            if (cw) {
                const int hk0 = (md + 1) / 2, nty = (hk0 + 127) / 128;
                dim3 gs((unsigned)((inner + 63) / 64), (unsigned)(2 * nty), (unsigned)outer);
                auto k = dct1_sym_kernel<false>; HIPGP_LAUNCH(k, gs, dim3(256), 0, s, src, dst, cw, md, inner, outer, scale, nty);
            } else { dct1_tile_check(md); auto k = dct1_tile_kernel<false>; HIPGP_LAUNCH(k, grid, dim3(256), 0, s, src, dst, tab, md, inner, outer, scale); }
        }
        CK_LAUNCH();
        pl->launches++;
        src = dst; which ^= 1;
    }
}

// the DCT-I of set_first_row / ensure_wide: Bluestein on long 1-D plans, the tiled kernels otherwise
static void dct1(hipgp_plan* pl, const double* in, double* out, double* tmp, bool normalise, cudaStream_t s) {
    if (pl->D == 1 && pl->long_n) long_dct1(pl, in, out, normalise, s);
    else dct_all_axes(pl, in, out, tmp, normalise, s);
}

// The spectrum of a re-embedded first column, from the fp64 forward passes of the matvecs, in the layout they leave: half
// spectra [L0]([L1])[P] on the row pass, full complex rows [L0]([L1])[L1 L2] in four-step order on the four-step path.
template <class T>
static void build_spectrum(hipgp_plan* pl, bool wide, const double* col, DevBuf& dst, bool complex_spec, cudaStream_t s) {
    const bool four = wide ? pl->long_w : pl->long_n;
    const int* Le = wide ? pl->Lw : pl->Ln;
    Geom<double>& g = wide ? pl->gw64 : pl->gn64;
    EmbedDims e{};
    e.D = pl->D;
    long total = 1;
    for (int d = 0; d < 3; ++d) { e.m[d] = 1; e.N[d] = 1; e.L[d] = 1; e.wide[d] = 0; }
    // right-align the D active axes into the 3 slots of EmbedDims
    for (int d = 0; d < pl->D; ++d) {
        const int slot = 3 - pl->D + d;
        e.m[slot] = pl->m[d]; e.N[slot] = pl->N[d]; e.L[slot] = Le[d]; e.wide[slot] = wide ? (pl->wide_real ? 2 : 1) : 0;
        total *= Le[d];
    }
    pl->tmpB.ensure(sizeof(double) * (size_t)total, &pl->dev_bytes);
    {
        auto k = embed_kernel;
        const int nb = (int)std::min<long>((total + 255) / 256, 148 * 8);
        HIPGP_LAUNCH(k, dim3(nb), dim3(256), 0, s, col, pl->tmpB.as<double>(), e);
        CK_LAUNCH(); pl->launches++;
    }
    // forward transform of the embedded column into W1 (raw spectrum, pipeline layout)
    long n;
    double scale;
    if (four) {
        long_conv<double>(pl, long_geom<double>(pl, wide ? 1 : 0), g, pl->tmpB.as<double>(), Le, nullptr, nullptr, nullptr, SPEC_NONE, 1, nullptr, s);
        n = total; scale = 1.0 / (double)total;
    } else {
        n = g.spec_elems();
        pl->W1.ensure(sizeof(cplx<double>) * (size_t)n, &pl->dev_bytes);
        cplx<double>* W1 = pl->W1.as<cplx<double>>();
        run_rows<double>(pl, g, false, n / g.P, W1, n / g.P, 1, g.L[g.D - 1], plain_in(pl->tmpB.as<double>()), null_state(), s);
        run_cols<double>(pl, g, CM_FWD, {W1, 0, g.L}, {W1, 0, g.L}, g.P, g.H + 1, 1, nullptr, SPEC_NONE, nullptr, s);
        scale = 0.25;
        for (int d = 0; d < g.D; ++d) scale /= (double)g.L[d];
    }
    cplx<double>* W1 = pl->W1.as<cplx<double>>();
    const unsigned nblk = (unsigned)((n + 255) / 256);
    if (complex_spec) {
        dst.ensure(sizeof(cplx<T>) * (size_t)n, &pl->dev_bytes);
        auto k = store_spec_cplx_kernel<T>; HIPGP_LAUNCH(k, dim3(nblk), dim3(256), 0, s, W1, dst.as<cplx<T>>(), n, scale);
    } else {
        dst.ensure(sizeof(T) * (size_t)n, &pl->dev_bytes);
        auto k = store_spec_real_kernel<T>; HIPGP_LAUNCH(k, dim3(nblk), dim3(256), 0, s, W1, dst.as<T>(), n, scale);
    }
    CK_LAUNCH(); pl->launches++;
}

// (a four-step last axis builds its own geometry on first use; its geometry here holds the leading axes' column passes)
template <class T>
static void ensure_geoms(hipgp_plan* pl, bool wide) {
    const bool four = wide ? pl->long_w : pl->long_n;
    if (four && pl->D == 1) return;
    Geom<double>& g64 = wide ? pl->gw64 : pl->gn64;
    const int* L = wide ? pl->Lw : pl->Ln;
    if (!g64.built) g64.build(pl->D, L, &pl->dev_bytes, !four);
    if (sizeof(T) == 4) {
        Geom<float>& g32 = wide ? pl->gw32 : pl->gn32;
        if (!g32.built) g32.build(pl->D, L, &pl->dev_bytes, !four);
    }
}

template <class T>
static void set_first_row(hipgp_plan* pl, const void* column, double clampv, cudaStream_t s) {
    const long M = pl->M;
    pl->clampv = clampv;
    ensure_geoms<T>(pl, false);
    for (DevBuf* b : {&pl->Dm, &pl->Dinv, &pl->Dsqrt, &pl->colK, &pl->colG, &pl->colS, &pl->tmpA})
        b->ensure(sizeof(double) * (size_t)M, &pl->dev_bytes);
    pl->tmpB.ensure(sizeof(double) * (size_t)M, &pl->dev_bytes);
    pl->counts.ensure(sizeof(unsigned) * 4, &pl->dev_bytes);
    CK(cudaMemsetAsync(pl->counts.p, 0, sizeof(unsigned) * 4, s));
    const unsigned nb = (unsigned)((M + 255) / 256);
    {
        auto k = to_double_kernel<T>;
        HIPGP_LAUNCH(k, dim3(nb), dim3(256), 0, s, (const T*)column, pl->colK.as<double>(), M);
        CK_LAUNCH(); pl->launches++;
    }
    // D = DCT-I(column), clamp, derive
    dct1(pl, pl->colK.as<double>(), pl->tmpA.as<double>(), pl->tmpB.as<double>(), false, s);
    {
        auto k = clamp_derive_kernel<T>;
        HIPGP_LAUNCH(k, dim3(nb), dim3(256), 0, s, pl->tmpA.as<double>(), pl->Dm.as<double>(), pl->Dinv.as<double>(),
                     pl->Dsqrt.as<double>(), M, clampv, pl->counts.as<unsigned>());
        CK_LAUNCH(); pl->launches++;
    }
    unsigned hc[4] = {0, 0, 0, 0};
    CK(cudaMemcpyAsync(hc, pl->counts.p, sizeof(hc), cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    pl->nclamped = hc[0];
    // first columns of C' (only when something was clamped or rounded: otherwise the column itself), C'^-1, C'^1/2
    if (pl->nclamped != 0 || sizeof(T) == 4)
        dct1(pl, pl->Dm.as<double>(), pl->colK.as<double>(), pl->tmpB.as<double>(), true, s);
    dct1(pl, pl->Dinv.as<double>(), pl->colG.as<double>(), pl->tmpB.as<double>(), true, s);
    // (the first column of C'^1/2 belongs to the wide embedding: ensure_wide builds it on the first R^T / R)
    build_spectrum<T>(pl, false, pl->colK.as<double>(), pl->specK, false, s);
    build_spectrum<T>(pl, false, pl->colG.as<double>(), pl->specCinv, false, s);
    pl->have_spec = true; pl->have_wide = false; pl->have_slabK = pl->have_slabCinv = false;
}

template <class T>
static void ensure_wide(hipgp_plan* pl, cudaStream_t s) {
    if (pl->have_wide) return;
    ensure_geoms<T>(pl, true);
    // Where every axis of the wide embedding is at least 2N - 1 long (config 2: 4096 >= 3995, the length the cost model picks
    // anyway) the taps are extended symmetrically and the spectrum of C^(1/2) is REAL: R^T and R then take the same staged
    // real-spectrum column pass as K instead of reading a complex spectrum from global memory.
    bool real_ok = true;
    for (int d = 0; d < pl->D; ++d) if (pl->Lw[d] < 2 * pl->N[d] - 1) real_ok = false;
    pl->wide_real = real_ok;
    dct1(pl, pl->Dsqrt.as<double>(), pl->colS.as<double>(), pl->tmpB.as<double>(), true, s);
    build_spectrum<T>(pl, true, pl->colS.as<double>(), pl->specW, !real_ok, s);
    pl->have_wide = true;
}

template <class T>
static void matvec(hipgp_plan* pl, int mode, const void* in, void* out, long B, cudaStream_t s) {
    if (!pl->have_spec) throw Error("plan has no spectrum: call hipgp_plan_set_first_row first");
    if (B < 0) throw Error("negative number of right-hand sides");
    if (B == 0) return;
    if (!in || !out) throw Error("null vector pointer");
    const bool wide = (mode == HIPGP_MV_RT || mode == HIPGP_MV_R);
    if (wide) ensure_wide<T>(pl, s);
    int n_in[3], n_out[3];
    for (int d = 0; d < pl->D; ++d) {
        n_in[d] = mode == HIPGP_MV_R ? pl->N[d] : pl->m[d];
        n_out[d] = mode == HIPGP_MV_RT ? pl->N[d] : pl->m[d];
    }
    const void* spec; int kind;
    switch (mode) {
        case HIPGP_MV_K: spec = pl->specK.p; kind = SPEC_REAL; break;
        case HIPGP_MV_CINV: spec = pl->specCinv.p; kind = SPEC_REAL; break;
        case HIPGP_MV_RT: spec = pl->specW.p; kind = pl->wide_real ? SPEC_REAL : SPEC_CPLX; break;
        case HIPGP_MV_R: spec = pl->specW.p; kind = pl->wide_real ? SPEC_REAL : SPEC_CPLX_CONJ; break;
        default: throw Error("unknown matvec mode");
    }
    if (wide ? pl->long_w : pl->long_n) {
        long_conv<T>(pl, long_geom<T>(pl, wide ? 1 : 0), geom(pl, wide, Tag<T>()), (const T*)in, n_in, (T*)out, n_out, spec, kind, B, nullptr, s);
        return;
    }
    run_pipeline<T>(pl, geom(pl, wide, Tag<T>()), n_in, n_out, spec, kind, B, plain_in(in), plain_out(out), null_state(), false, s);
}

template <class T>
static PcgDev pcg_state(hipgp_plan* pl, long B, double tol, bool cg_mode) {
    const long M = pl->M;
    long nrows = 1;
    for (int d = 0; d + 1 < pl->D; ++d) nrows *= pl->m[d];
    for (DevBuf* b : {&pl->vr, &pl->vp, &pl->vz, &pl->vAp}) b->ensure(sizeof(T) * (size_t)(B * M), &pl->dev_bytes);
    pl->partial.ensure(sizeof(double) * (size_t)(B * nrows), &pl->dev_bytes);
    pl->scal.ensure(sizeof(double) * (size_t)(4 * B), &pl->dev_bytes);
    const bool fresh = pl->cnt.bytes < sizeof(unsigned) * (size_t)(B + 1);
    pl->cnt.ensure(sizeof(unsigned) * (size_t)(B + 1), &pl->dev_bytes);
    pl->flags.ensure(sizeof(int) * 4, &pl->dev_bytes);
    if (fresh) CK(cudaMemset(pl->cnt.p, 0, pl->cnt.bytes));
    PcgDev st{};
    double* sc = pl->scal.as<double>();
    st.zr = sc; st.zr_prev = sc + B; st.pAp = sc + 2 * B; st.rr = sc + 3 * B;
    st.partial = pl->partial.as<double>();
    st.row_cnt = pl->cnt.as<unsigned>(); st.rhs_cnt = pl->cnt.as<unsigned>() + B;
    st.flags = pl->flags.as<int>();
    st.tol = tol; st.B = (int)B; st.cg_mode = cg_mode ? 1 : 0;
    return st;
}

// plain (no FFT) fused vector kernels reuse rows_fwd_kernel with do_fft = 0
template <class T>
static void launch_vec(hipgp_plan* pl, int mode, const PcgDev& st, long B, const void* in, void* v0, void* v1, const void* v2,
                       cudaStream_t s) {
    long nrows = 1;
    for (int d = 0; d + 1 < pl->D; ++d) nrows *= pl->m[d];
    RowsParams<T> R{};
    R.in = (const T*)in; R.v0 = (T*)v0; R.v1 = (T*)v1; R.v2 = (const T*)v2;
    R.mode = mode; R.do_fft = 0; R.total_rows = B * nrows; R.nrows = (int)nrows; R.n_real = pl->m[pl->D - 1];
    R.H = (R.n_real + 1) / 2; R.L = 2 * R.H; R.st = st;
    R.RB = 8; R.RBP = 9;
    dim3 grid((unsigned)((R.total_rows + R.RB - 1) / R.RB));
    auto k = rows_fwd_kernel<T>;
    PROF_BEGIN(pl, 3, s);
    HIPGP_LAUNCH(k, grid, dim3(256), 0, s, R);
    PROF_END(pl, s);
    CK_LAUNCH(); pl->launches++;
}

// x = 0 ; r = b ; z = P r (or r) ; r.z  -- everything before the first iteration of cg.py:58-62
template <class T>
static void pcg_begin(hipgp_plan* pl, const void* b, void* x, long B, double tol, bool precond, cudaStream_t s) {
    if (!pl->have_spec) throw Error("plan has no spectrum: call hipgp_plan_set_first_row first");
    if (B <= 0) throw Error("pcg needs at least one right-hand side");
    if (!b || !x) throw Error("null vector pointer");
    const long M = pl->M;
    PcgDev st = pcg_state<T>(pl, B, tol, !precond);
    if (!pl->pinned) CK(cudaMallocHost(&pl->pinned, 64));
    T* r = pl->vr.as<T>(); T* z = precond ? pl->vz.as<T>() : r;
    // x = 0 ; r = b - A(0) = b   (cg.py:58-59; the reference spends a matvec on the zero vector)
    CK(cudaMemsetAsync(x, 0, sizeof(T) * (size_t)(B * M), s));
    CK(cudaMemcpyAsync(r, b, sizeof(T) * (size_t)(B * M), cudaMemcpyDeviceToDevice, s));
    // flags = {0, 0, 1, 0} without a pageable host copy (which would synchronise the stream): clear, then one byte
    CK(cudaMemsetAsync(st.flags, 0, sizeof(int) * 4, s));
    CK(cudaMemsetAsync(reinterpret_cast<char*>(st.flags) + 2 * sizeof(int), 1, 1, s));
    RowsFusion ff, fi;
    if (pl->long_n) {
        long_pcg_begin<T>(pl, st, B, precond, s);
    } else if (precond) {   // z = P r ; zr = z.r
        int nn[3];
        for (int d = 0; d < pl->D; ++d) nn[d] = pl->m[d];
        ff.mode = RF_PLAIN; ff.in = r; fi.mode = RI_DOT; fi.dot_kind = DOT_ZR; fi.out = z; fi.v0 = r;
        run_pipeline<T>(pl, geom(pl, false, Tag<T>()), nn, nn, pl->specCinv.p, SPEC_REAL, B, ff, fi, st, false, s);
    } else {         // z = r ; zr = r.r
        launch_vec<T>(pl, RF_SELFDOT, st, B, r, nullptr, nullptr, nullptr, s);
    }
    pl->run_x = x; pl->run_B = B; pl->run_precond = precond; pl->run_tol = tol; pl->run_active = true;
}

// `niter` more iterations of the loop body cg.py:64-78 (kernels of a locally converged solve are no-ops)
template <class T>
static void pcg_iterate(hipgp_plan* pl, int niter, cudaStream_t s) {
    if (!pl->run_active) throw Error("hipgp_pcg_step without hipgp_pcg_begin");
    const long B = pl->run_B;
    const bool precond = pl->run_precond;
    PcgDev st = pcg_state<T>(pl, B, pl->run_tol, !precond);
    if (pl->long_n) { long_pcg_iterate<T>(pl, st, niter, s); return; }
    Geom<T>& g = geom(pl, false, Tag<T>());
    int nn[3];
    for (int d = 0; d < pl->D; ++d) nn[d] = pl->m[d];
    T* r = pl->vr.as<T>(); T* p = pl->vp.as<T>(); T* z = precond ? pl->vz.as<T>() : r; T* Ap = pl->vAp.as<T>();
    void* x = pl->run_x;
    RowsFusion ff, fi;
    for (int c = 0; c < niter; ++c) {
        // p = z + beta p ; Ap = K p ; pAp
        ff = RowsFusion(); fi = RowsFusion();
        ff.mode = RF_PUPDATE; ff.in = z; ff.v0 = p;
        fi.mode = RI_DOT; fi.dot_kind = DOT_PAP; fi.out = Ap; fi.v0 = p;
        run_pipeline<T>(pl, g, nn, nn, pl->specK.p, SPEC_REAL, B, ff, fi, st, true, s);
        if (precond) {   // x += a p ; r -= a Ap ; rr ; stop test ; z = P r ; zr
            ff = RowsFusion(); fi = RowsFusion();
            ff.mode = RF_XRUPDATE; ff.in = Ap; ff.v0 = r; ff.v1 = x; ff.v2 = p;
            fi.mode = RI_DOT; fi.dot_kind = DOT_ZR; fi.out = z; fi.v0 = r;
            run_pipeline<T>(pl, g, nn, nn, pl->specCinv.p, SPEC_REAL, B, ff, fi, st, true, s);
        } else {
            launch_vec<T>(pl, RF_XRUPDATE, st, B, Ap, r, x, p, s);
        }
    }
}

// flags + residuals to the host (synchronises the stream)
static void pcg_poll(hipgp_plan* pl, int* done, int* iters, double* max_resid, double* resid_out, cudaStream_t s) {
    int* hflags = reinterpret_cast<int*>(pl->pinned);
    CK(cudaMemcpyAsync(hflags, pl->flags.p, sizeof(int) * 4, cudaMemcpyDeviceToHost, s));
    std::vector<double> rr;
    if (max_resid || resid_out) {
        rr.resize(pl->run_B);
        CK(cudaMemcpyAsync(rr.data(), pl->scal.as<double>() + 3 * pl->run_B, sizeof(double) * pl->run_B, cudaMemcpyDeviceToHost, s));
    }
    CK(cudaStreamSynchronize(s));
    if (done) *done = hflags[0];
    if (iters) *iters = hflags[1];
    if (max_resid) {
        double mx = 0.0; bool nan = false;
        for (double v : rr) { const double q = std::sqrt(v); if (q != q) nan = true; else if (q > mx) mx = q; }
        *max_resid = nan ? NAN : mx;
    }
    if (resid_out) for (long i = 0; i < pl->run_B; ++i) resid_out[i] = std::sqrt(rr[i]);
}

template <class T>
static void pcg(hipgp_plan* pl, const void* b, void* x, long B, int maxiter, double tol, bool precond, int* iters_out,
                int* callbacks_out, double* resid_out, hipgp_iter_cb cb, void* user, cudaStream_t s) {
    if (iters_out) *iters_out = 0;
    if (callbacks_out) *callbacks_out = 0;
    if (B < 0) throw Error("negative number of right-hand sides");
    if (B == 0) return;
    pcg_begin<T>(pl, b, x, B, tol, precond, s);
    const int check_every = cb ? 1 : 8;
    int done = 0, iters = 0, n = 0;
    while (n < maxiter && !done) {
        const int chunk = std::min(check_every, maxiter - n);
        pcg_iterate<T>(pl, chunk, s);
        pcg_poll(pl, &done, &iters, nullptr, nullptr, s);
        n += chunk;
        if (cb && !done) cb(n - 1, x, user);
    }
    if (iters_out) *iters_out = iters;
    if (callbacks_out) *callbacks_out = done ? iters - 1 : iters;
    if (resid_out) pcg_poll(pl, nullptr, nullptr, nullptr, resid_out, s);
    pl->run_active = false;
}

}  // namespace hipgp

// ---------------------------------------------------------------------------------------------
// C ABI
#define API_BEGIN try {
#define API_END                                                                          \
    } catch (const std::exception& e) { hipgp::g_err = e.what(); return -1; }            \
      catch (...) { hipgp::g_err = "unknown error"; return -2; }                         \
    return 0;

#define DISPATCH(pl, call_f32, call_f64) do { if ((pl)->dtype == HIPGP_F32) { call_f32; } else { call_f64; } } while (0)

static void need_plan(const hipgp_plan* pl) { if (!pl) throw Error("null plan handle"); }
static void set_device(const hipgp_plan* pl) { need_plan(pl); CK(cudaSetDevice(pl->device)); }

static void slab_peer_close(hipgp_plan* pl) {
#ifndef HIPGP_EMU
    for (int i = 0; i < pl->n_ipc_opened; ++i) if (pl->ipc_opened[i]) cudaIpcCloseMemHandle(pl->ipc_opened[i]);
#endif
    pl->n_ipc_opened = 0; pl->peers_ready = false;
}

extern "C" {

const char* hipgp_last_error(void) { return hipgp::g_err.c_str(); }
int hipgp_version(void) { return 100; }

int hipgp_plan_create(int ndim, const int64_t* m, int dtype, int device, hipgp_plan** out) {
    API_BEGIN
    if (!out || !m || ndim < 1) throw Error("bad arguments");
    if (dtype != HIPGP_F32 && dtype != HIPGP_F64) throw Error("dtype must be HIPGP_F32 or HIPGP_F64");
    hipgp_plan* pl = new hipgp_plan();
    pl->dtype = dtype; pl->device = device; pl->ndim_user = ndim;
    int D = 0;
    for (int d = 0; d < ndim; ++d) {
        if (m[d] < 1) { delete pl; throw Error("grid extents must be >= 1"); }
        pl->m_user.push_back((long)m[d]);
        pl->M *= m[d];
        if (m[d] > 1) {
            if (D == 3) { delete pl; throw Error("at most 3 grid axes of extent > 1 are supported"); }
            pl->m[D] = (int)m[d]; pl->N[D] = 2 * (int)m[d] - 2; pl->E *= pl->N[D]; ++D;
        }
    }
    if (D == 0) { D = 1; pl->m[0] = 1; pl->N[0] = 1; }
    pl->D = D;
    try {
        for (int d = 0; d < D; ++d) {
            const bool row = (d == D - 1);
            pl->Ln[d] = choose_length(2L * pl->m[d] - 1, row);
            pl->Lw[d] = choose_length((long)pl->N[d] + pl->m[d] - 1, row);
        }
        // an embedding whose last-axis row pass would not fit shared memory takes the four-step path along that axis, at a
        // length L1 * L2 (the other axes keep theirs)
        {
            const int a = D - 1;
            const long ma = pl->m[a], Na = pl->N[a];
            auto fits = [&](int L, long n_max) { return dtype == HIPGP_F32 ? row_embedding_fits<float>(L, n_max) : row_embedding_fits<double>(L, n_max); };
            auto split = [&](long n, int which, int* L) {
                int* f = pl->lsplit[which];
                if (!long_split(n, &f[0], &f[1]))
                    throw Error((D == 1 ? "1-D grid of " : "last grid axis of ") + std::to_string(ma) + " points is too long: the four-step path reaches " +
                                std::to_string((long)kLongMaxFactor * kLongMaxFactor) + "-point transforms (m <= " +
                                std::to_string(((long)kLongMaxFactor * kLongMaxFactor + 5) / 4) + ")");
                if (L) *L = f[0] * f[1];
            };
            pl->long_n = !fits(pl->Ln[a], ma);
            pl->long_w = pl->long_n || !fits(pl->Lw[a], Na);
            if (pl->long_n) { split(2 * ma - 1, 0, &pl->Ln[a]); if (D == 1) split(2 * Na - 1, 2, nullptr); }
            if (pl->long_w) split(Na + ma - 1, 1, &pl->Lw[a]);
        }
    } catch (...) { delete pl; throw; }
    *out = pl;
    API_END
}

int hipgp_plan_destroy(hipgp_plan* pl) {
    API_BEGIN
    if (!pl) return 0;
    size_t* t = &pl->dev_bytes;
    pl->gn32.release(t); pl->gw32.release(t); pl->gn64.release(t); pl->gw64.release(t);
    pl->ln32.release(t); pl->lw32.release(t); pl->ln64.release(t); pl->lw64.release(t); pl->lb64.release(t);
    pl->bluA.release(t); pl->bluSpec.release(t);
    for (DevBuf* b : {&pl->specK, &pl->specCinv, &pl->specW, &pl->Dm, &pl->Dinv, &pl->Dsqrt, &pl->colK, &pl->colG, &pl->colS,
                      &pl->tmpA, &pl->tmpB, &pl->counts, &pl->W1, &pl->W2, &pl->vr, &pl->vp, &pl->vz, &pl->vAp,
                      &pl->partial, &pl->scal, &pl->cnt, &pl->flags, &pl->stage_in, &pl->stage_out, &pl->corrU, &pl->corrV, &pl->corrS,
                      &pl->corrLag, &pl->gradA, &pl->slabSpecK, &pl->slabSpecCinv, &pl->slabR1, &pl->slabR2, &pl->slot_in[0], &pl->slot_in[1], &pl->slot_out[0], &pl->slot_out[1], &pl->costabs[0], &pl->costabs[1], &pl->costabs[2], &pl->cosmats[0], &pl->cosmats[1], &pl->cosmats[2]})
        b->release(t);
    slab_peer_close(pl);
#ifndef HIPGP_EMU
    for (auto& se : pl->slot_ev) for (auto& e : se) if (e) cudaEventDestroy(e);
    if (pl->slot_flags) cudaFreeHost(pl->slot_flags);
#else
    delete[] pl->slot_flags;
#endif
    if (pl->pinned) cudaFreeHost(pl->pinned);
#ifndef HIPGP_EMU
    for (auto& cs : pl->copy_streams) if (cs) cudaStreamDestroy(cs);
#endif
    delete pl;
    API_END
}

int hipgp_plan_sizes(const hipgp_plan* pl, int64_t* M, int64_t* Mprime) {
    API_BEGIN
    need_plan(pl);
    if (M) *M = pl->M;
    if (Mprime) *Mprime = pl->E;
    API_END
}

int hipgp_plan_embedding(const hipgp_plan* pl, int64_t* Ln, int64_t* Lw) {
    API_BEGIN
    need_plan(pl);
    int a = 0;
    for (int d = 0; d < pl->ndim_user; ++d) {
        const bool active = pl->m_user[d] > 1 || (pl->D == 1 && pl->M == 1 && d == 0);
        if (Ln) Ln[d] = active ? pl->Ln[a] : 1;
        if (Lw) Lw[d] = active ? pl->Lw[a] : 1;
        if (active) ++a;
    }
    API_END
}

int hipgp_plan_set_first_row(hipgp_plan* pl, const void* column, double clampv, int64_t* clamped_out, void* stream) {
    API_BEGIN
    set_device(pl);
    DISPATCH(pl, set_first_row<float>(pl, column, clampv, (cudaStream_t)stream), set_first_row<double>(pl, column, clampv, (cudaStream_t)stream));
    if (clamped_out) *clamped_out = pl->nclamped;
    API_END
}

int hipgp_plan_spectrum(hipgp_plan* pl, int which, void* out, void* stream) {
    API_BEGIN
    set_device(pl);
    if (!pl->have_spec) throw Error("plan has no spectrum");
    if (which < 0 || which > 3) throw Error("bad spectrum selector");
    EmbedDims e{};
    for (int d = 0; d < 3; ++d) { e.m[d] = 1; e.N[d] = 1; e.L[d] = 1; e.wide[d] = 0; }
    for (int d = 0; d < pl->D; ++d) { const int slot = 3 - pl->D + d; e.m[slot] = pl->m[d]; e.N[slot] = pl->N[d]; }
    const int nb = (int)std::min<long>((pl->E + 255) / 256, 148 * 8);
    cudaStream_t s = (cudaStream_t)stream;
    if (pl->dtype == HIPGP_F32) { auto k = expand_even_kernel<float>; HIPGP_LAUNCH(k, dim3(nb), dim3(256), 0, s, pl->Dm.as<double>(), (float*)out, e, which); }
    else { auto k = expand_even_kernel<double>; HIPGP_LAUNCH(k, dim3(nb), dim3(256), 0, s, pl->Dm.as<double>(), (double*)out, e, which); }
    CK_LAUNCH(); pl->launches++;
    API_END
}

int hipgp_matvec(hipgp_plan* pl, int mode, const void* in, void* out, int64_t B, void* stream) {
    API_BEGIN
    set_device(pl);
    DISPATCH(pl, matvec<float>(pl, mode, in, out, (long)B, (cudaStream_t)stream), matvec<double>(pl, mode, in, out, (long)B, (cudaStream_t)stream));
    API_END
}

static size_t elem_size(const hipgp_plan* pl) { return pl->dtype == HIPGP_F32 ? 4 : 8; }

int hipgp_matvec_host(hipgp_plan* pl, int mode, const void* in_host, void* out_host, int64_t B, void* stream) {
    API_BEGIN
    set_device(pl);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t nin = (size_t)B * (mode == HIPGP_MV_R ? pl->E : pl->M) * elem_size(pl);
    const size_t nout = (size_t)B * (mode == HIPGP_MV_RT ? pl->E : pl->M) * elem_size(pl);
    pl->stage_in.ensure(nin, &pl->dev_bytes); pl->stage_out.ensure(nout, &pl->dev_bytes);
    CK(cudaMemcpyAsync(pl->stage_in.p, in_host, nin, cudaMemcpyHostToDevice, s));
    DISPATCH(pl, matvec<float>(pl, mode, pl->stage_in.p, pl->stage_out.p, (long)B, s), matvec<double>(pl, mode, pl->stage_in.p, pl->stage_out.p, (long)B, s));
    CK(cudaMemcpyAsync(out_host, pl->stage_out.p, nout, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    API_END
}

int hipgp_pcg(hipgp_plan* pl, const void* b, void* x, int64_t B, int maxiter, double tol, int precond, int* iters_out,
              int* callbacks_out, double* resid_out, hipgp_iter_cb cb, void* user, void* stream) {
    API_BEGIN
    set_device(pl);
    cudaStream_t s = (cudaStream_t)stream;
    DISPATCH(pl, pcg<float>(pl, b, x, (long)B, maxiter, tol, precond != 0, iters_out, callbacks_out, resid_out, cb, user, s),
             pcg<double>(pl, b, x, (long)B, maxiter, tol, precond != 0, iters_out, callbacks_out, resid_out, cb, user, s));
    API_END
}

int hipgp_pcg_begin(hipgp_plan* pl, const void* b, void* x, int64_t B, double tol, int precond, void* stream) {
    API_BEGIN
    set_device(pl);
    cudaStream_t s = (cudaStream_t)stream;
    DISPATCH(pl, pcg_begin<float>(pl, b, x, (long)B, tol, precond != 0, s), pcg_begin<double>(pl, b, x, (long)B, tol, precond != 0, s));
    API_END
}

int hipgp_pcg_step(hipgp_plan* pl, int niter, int* done_out, int* iters_out, double* max_resid_out, void* stream) {
    API_BEGIN
    set_device(pl);
    cudaStream_t s = (cudaStream_t)stream;
    DISPATCH(pl, pcg_iterate<float>(pl, niter, s), pcg_iterate<double>(pl, niter, s));
    if (done_out || iters_out || max_resid_out) pcg_poll(pl, done_out, iters_out, max_resid_out, nullptr, s);
    API_END
}

int hipgp_pcg_host(hipgp_plan* pl, const void* b_host, void* x_host, int64_t B, int maxiter, double tol, int precond,
                   int* iters_out, int* callbacks_out, double* resid_out, void* stream) {
    API_BEGIN
    set_device(pl);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)B * pl->M * elem_size(pl);
    pl->stage_in.ensure(n, &pl->dev_bytes); pl->stage_out.ensure(n, &pl->dev_bytes);
    CK(cudaMemcpyAsync(pl->stage_in.p, b_host, n, cudaMemcpyHostToDevice, s));
    DISPATCH(pl, pcg<float>(pl, pl->stage_in.p, pl->stage_out.p, (long)B, maxiter, tol, precond != 0, iters_out, callbacks_out, resid_out, nullptr, nullptr, s),
             pcg<double>(pl, pl->stage_in.p, pl->stage_out.p, (long)B, maxiter, tol, precond != 0, iters_out, callbacks_out, resid_out, nullptr, nullptr, s));
    CK(cudaMemcpyAsync(x_host, pl->stage_out.p, n, cudaMemcpyDeviceToHost, s));
    CK(cudaStreamSynchronize(s));
    API_END
}

// The same solve with the transfers hidden: the right-hand sides are processed in groups (`group` at both ends, the rest in
// the middle; uniform groups of `group` when B < 4 group); the host-to-device copy of group g+1 and the device-to-host copy
// of group g-1 run on the plan's two copy streams while group g is solved on the caller's stream (events order them).  Every group is an independent batched solve: the stopping rule
// all_b sqrt(r_b.r_b) < tol (cg.py:70) is evaluated over the right-hand sides of ONE group, so a group may stop before
// another one does; iters_out receives the maximum over the groups.  Host buffers should be pinned.
int hipgp_pcg_host_pipelined(hipgp_plan* pl, const void* b_host, void* x_host, int64_t B, int maxiter, double tol, int precond,
                             int64_t group, int* iters_out, void* stream) {
    API_BEGIN
    set_device(pl);
    if (iters_out) *iters_out = 0;
    if (B < 0) throw Error("negative number of right-hand sides");
    if (B == 0) return 0;
    if (!b_host || !x_host) throw Error("null vector pointer");
    if (group <= 0 || group > B) group = B;
    cudaStream_t s = (cudaStream_t)stream;
#ifndef HIPGP_EMU
    if (!pl->copy_streams[0]) {
        CK(cudaStreamCreateWithFlags(&pl->copy_streams[0], cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&pl->copy_streams[1], cudaStreamNonBlocking));
    }
#endif
    const size_t row = (size_t)pl->M * elem_size(pl);
    pl->stage_in.ensure((size_t)B * row, &pl->dev_bytes); pl->stage_out.ensure((size_t)B * row, &pl->dev_bytes);
    // group sizes: a SMALL first and last group of `group` right-hand sides and everything else in one solve.  The first upload
    // and the last download are the only copies nothing can hide, so they are small; the bulk stays one big batch because the
    // solver is ~10 % more efficient per right-hand side at 48 than at 16 (measured: uniform groups of 16 cost more in solver
    // efficiency than they hide in copies).
    std::vector<long> gs;
    if (B >= 4 * group) { gs.push_back(group); gs.push_back(B - 2 * group); gs.push_back(group); }
    else for (long b0 = 0; b0 < B; b0 += group) gs.push_back(std::min<long>(group, B - b0));
    const long ng = (long)gs.size();
    std::vector<long> gb0(ng);
    { long acc = 0; for (long g = 0; g < ng; ++g) { gb0[g] = acc; acc += gs[g]; } }
    std::vector<cudaEvent_t> in_ready(ng), solved(ng);
#ifndef HIPGP_EMU
    for (long g = 0; g < ng; ++g) { CK(cudaEventCreateWithFlags(&in_ready[g], cudaEventDisableTiming)); CK(cudaEventCreateWithFlags(&solved[g], cudaEventDisableTiming)); }
    cudaStream_t cin = pl->copy_streams[0], cout = pl->copy_streams[1];
    // the copy streams start after whatever the caller has queued on its stream (the staging buffers may still be in use)
    cudaEvent_t start; CK(cudaEventCreateWithFlags(&start, cudaEventDisableTiming));
    CK(cudaEventRecord(start, s)); CK(cudaStreamWaitEvent(cin, start, 0)); CK(cudaStreamWaitEvent(cout, start, 0));
#else
    cudaStream_t cin = s, cout = s;
#endif
    for (long g = 0; g < ng; ++g) {       // all uploads are queued up front: they run ahead of the solves on their own stream
        const long b0 = gb0[g], nb = gs[g];
        CK(cudaMemcpyAsync((char*)pl->stage_in.p + b0 * row, (const char*)b_host + b0 * row, nb * row, cudaMemcpyHostToDevice, cin));
#ifndef HIPGP_EMU
        CK(cudaEventRecord(in_ready[g], cin));
#endif
    }
    int iters_max = 0;
    for (long g = 0; g < ng; ++g) {
        const long b0 = gb0[g], nb = gs[g];
#ifndef HIPGP_EMU
        CK(cudaStreamWaitEvent(s, in_ready[g], 0));
#endif
        int it = 0;
        void* bg = (char*)pl->stage_in.p + b0 * row; void* xg = (char*)pl->stage_out.p + b0 * row;
        DISPATCH(pl, pcg<float>(pl, bg, xg, nb, maxiter, tol, precond != 0, &it, nullptr, nullptr, nullptr, nullptr, s),
                 pcg<double>(pl, bg, xg, nb, maxiter, tol, precond != 0, &it, nullptr, nullptr, nullptr, nullptr, s));
        iters_max = std::max(iters_max, it);
#ifndef HIPGP_EMU
        CK(cudaEventRecord(solved[g], s));
        CK(cudaStreamWaitEvent(cout, solved[g], 0));
#endif
        CK(cudaMemcpyAsync((char*)x_host + b0 * row, xg, nb * row, cudaMemcpyDeviceToHost, cout));
    }
#ifndef HIPGP_EMU
    CK(cudaStreamSynchronize(cout));
    CK(cudaStreamSynchronize(s));
    for (long g = 0; g < ng; ++g) { cudaEventDestroy(in_ready[g]); cudaEventDestroy(solved[g]); }
    cudaEventDestroy(start);
#endif
    if (iters_out) *iters_out = iters_max;
    API_END
}

// Asynchronous host-buffer solves for a STREAM of batches: submit returns as soon as the work is queued -- upload on the plan's
// H2D stream, the whole solve (begin + maxiter iterations; kernels of a converged solve exit at their first instruction, so the
// reference's stopping rule holds without the host looking) on the caller's stream, download on the D2H stream -- and wait blocks
// until the slot's result is in x_host.  With two slots in flight the upload of batch k+1 and the download of batch k-1 run under
// the solve of batch k.  Solves of one plan are ordered on the caller's stream (they share the solver's work vectors).
int hipgp_pcg_host_submit(hipgp_plan* pl, const void* b_host, void* x_host, int64_t B, int maxiter, double tol, int precond, int slot,
                          void* stream) {
    API_BEGIN
    set_device(pl);
    if (slot < 0 || slot > 1) throw Error("slot must be 0 or 1");
    if (B <= 0) throw Error("hipgp_pcg_host_submit needs at least one right-hand side");
    if (!b_host || !x_host) throw Error("null vector pointer");
    if (maxiter < 0) throw Error("negative maxiter");
    cudaStream_t s = (cudaStream_t)stream;
#ifndef HIPGP_EMU
    if (!pl->copy_streams[0]) {
        CK(cudaStreamCreateWithFlags(&pl->copy_streams[0], cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&pl->copy_streams[1], cudaStreamNonBlocking));
    }
    for (int e = 0; e < 3; ++e) if (!pl->slot_ev[slot][e]) CK(cudaEventCreateWithFlags(&pl->slot_ev[slot][e], cudaEventDisableTiming));
    if (!pl->slot_flags) CK(cudaMallocHost((void**)&pl->slot_flags, sizeof(int) * 8));
    if (pl->slot_busy[slot]) { CK(cudaEventSynchronize(pl->slot_ev[slot][2])); pl->slot_busy[slot] = false; }   // the slot's previous batch
    cudaStream_t cin = pl->copy_streams[0], cout = pl->copy_streams[1];
#else
    if (!pl->slot_flags) pl->slot_flags = new int[8];
    cudaStream_t cin = s, cout = s;
#endif
    const size_t n = (size_t)B * pl->M * elem_size(pl);
    pl->slot_in[slot].ensure(n, &pl->dev_bytes); pl->slot_out[slot].ensure(n, &pl->dev_bytes);
    CK(cudaMemcpyAsync(pl->slot_in[slot].p, b_host, n, cudaMemcpyHostToDevice, cin));
#ifndef HIPGP_EMU
    CK(cudaEventRecord(pl->slot_ev[slot][0], cin));
    CK(cudaStreamWaitEvent(s, pl->slot_ev[slot][0], 0));
#endif
    if (pl->dtype == HIPGP_F32) { pcg_begin<float>(pl, pl->slot_in[slot].p, pl->slot_out[slot].p, (long)B, tol, precond != 0, s); pcg_iterate<float>(pl, maxiter, s); }
    else { pcg_begin<double>(pl, pl->slot_in[slot].p, pl->slot_out[slot].p, (long)B, tol, precond != 0, s); pcg_iterate<double>(pl, maxiter, s); }
    pl->run_active = false;
    CK(cudaMemcpyAsync(pl->slot_flags + 4 * slot, pl->flags.p, sizeof(int) * 4, cudaMemcpyDeviceToHost, s));
#ifndef HIPGP_EMU
    CK(cudaEventRecord(pl->slot_ev[slot][1], s));
    CK(cudaStreamWaitEvent(cout, pl->slot_ev[slot][1], 0));
#endif
    CK(cudaMemcpyAsync(x_host, pl->slot_out[slot].p, n, cudaMemcpyDeviceToHost, cout));
#ifndef HIPGP_EMU
    CK(cudaEventRecord(pl->slot_ev[slot][2], cout));
#endif
    pl->slot_busy[slot] = true;
    API_END
}
int hipgp_pcg_host_wait(hipgp_plan* pl, int slot, int* iters_out) {
    API_BEGIN
    set_device(pl);
    if (slot < 0 || slot > 1) throw Error("slot must be 0 or 1");
    if (!pl->slot_busy[slot]) throw Error("hipgp_pcg_host_wait: nothing was submitted on this slot");
#ifndef HIPGP_EMU
    CK(cudaEventSynchronize(pl->slot_ev[slot][2]));
#endif
    pl->slot_busy[slot] = false;
    if (iters_out) *iters_out = pl->slot_flags[4 * slot + 1];
    API_END
}

int hipgp_compute_kn(hipgp_plan* pl, const void* Knm, void* kn, int64_t B, int maxiter, double tol, int* iters_out, void* stream) {
    API_BEGIN
    set_device(pl);
    cudaStream_t s = (cudaStream_t)stream;
    const size_t n = (size_t)B * pl->M * elem_size(pl);
    pl->stage_out.ensure(n, &pl->dev_bytes);
    void* d0 = pl->stage_out.p;
    DISPATCH(pl, pcg<float>(pl, Knm, d0, (long)B, maxiter, tol, true, iters_out, nullptr, nullptr, nullptr, nullptr, s),
             pcg<double>(pl, Knm, d0, (long)B, maxiter, tol, true, iters_out, nullptr, nullptr, nullptr, nullptr, s));
    DISPATCH(pl, matvec<float>(pl, HIPGP_MV_RT, d0, kn, (long)B, s), matvec<double>(pl, HIPGP_MV_RT, d0, kn, (long)B, s));
    API_END
}

int hipgp_plan_profile(hipgp_plan* pl, int enable) {
    API_BEGIN
    need_plan(pl);
    pl->profiling = enable != 0;
    API_END
}
int hipgp_plan_profile_read(hipgp_plan* pl, int kernel_class, double* ms_total, int64_t* launches, int reset) {
    API_BEGIN
    need_plan(pl);
    if (kernel_class < 0 || kernel_class > 3) throw Error("kernel_class must be 0..3");
#ifndef HIPGP_EMU
    set_device(pl);
    CK(cudaDeviceSynchronize());
    for (auto& r : pl->prof) {
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, r.e0, r.e1));
        pl->prof_ms[r.cls] += ms; pl->prof_n[r.cls] += 1;
        cudaEventDestroy(r.e0); cudaEventDestroy(r.e1);
    }
    pl->prof.clear();
#endif
    if (ms_total) *ms_total = pl->prof_ms[kernel_class];
    if (launches) *launches = pl->prof_n[kernel_class];
    if (reset) for (int i = 0; i < 4; ++i) { pl->prof_ms[i] = 0; pl->prof_n[i] = 0; }
    API_END
}
int hipgp_plan_device_bytes(const hipgp_plan* pl, size_t* bytes) { API_BEGIN need_plan(pl); if (bytes) *bytes = pl->dev_bytes; API_END }
int hipgp_plan_launch_count(const hipgp_plan* pl, int64_t* launches) { API_BEGIN need_plan(pl); if (launches) *launches = pl->launches; API_END }

}  // extern "C"

#include "vec_api.inl"
#include "long1d_api.inl"
#include "kxu_api.inl"
#include "corr_api.inl"
#include "block_api.inl"
#include "slab_api.inl"

#ifdef HIPGP_EMU
namespace emu {
thread_local dim3 t_threadIdx, t_blockIdx;
dim3 g_blockDim, g_gridDim;
Barrier g_block_barrier;
Barrier g_warp_barrier[64];
NamedBarrier g_named_barrier[16];
unsigned char* g_dyn_smem = nullptr;
double g_shfl_scratch[64][32][2];
}
#endif
