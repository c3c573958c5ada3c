// plan_types.cuh -- host-side types shared by plan.cu and the per-length kernel instantiation units (fast_inst.cu).
#pragma once
#include "../../include/hipgp_b200.h"
#include "conv_kernels.cuh"

#include <string>
#include <stdexcept>

namespace hipgp {

extern thread_local std::string g_err;
struct Error : std::runtime_error { using std::runtime_error::runtime_error; };

#define CK(expr)                                                                                     \
    do {                                                                                             \
        cudaError_t e__ = (expr);                                                                    \
        if (e__ != cudaSuccess)                                                                      \
            throw Error(std::string(#expr) + ": " + cudaGetErrorString(e__));                        \
    } while (0)
#define CK_LAUNCH() CK(cudaGetLastError())

// ---------------------------------------------------------------------------------------------
struct DevBuf {
    void* p = nullptr; size_t bytes = 0;
    void ensure(size_t n, size_t* total) {
        if (n <= bytes) return;
        if (p) { cudaFree(p); *total -= bytes; }
        p = nullptr; bytes = 0;
        if (cudaMalloc(&p, n) != cudaSuccess) { p = nullptr; throw Error("cudaMalloc of " + std::to_string(n) + " bytes failed"); }
        bytes = n; *total += n;
    }
    void release(size_t* total) { if (p) { cudaFree(p); *total -= bytes; } p = nullptr; bytes = 0; }
    template <class U> U* as() const { return reinterpret_cast<U*>(p); }
};

// ---------------------------------------------------------------------------------------------
// line FFT descriptors
// Lengths with a compile-time specialised kernel family (fast_kernels.cuh) and their DIF radix lists.
// X(length, radices...)
#ifdef HIPGP_DEV_SMALL   /* quick developer / emulation builds: a handful of lengths, the rest takes the generic kernels */
#if defined(HIPGP_EXP) && HIPGP_EXP == 1
#define HIPGP_EXP_R2048 8, 8, 8, 4
#define HIPGP_EXP_R1024 8, 8, 4, 4
#elif defined(HIPGP_EXP) && HIPGP_EXP == 2
#define HIPGP_EXP_R2048 8, 16, 16
#define HIPGP_EXP_R1024 8, 8, 16
#else
#define HIPGP_EXP_R2048 16, 8, 16
#define HIPGP_EXP_R1024 8, 8, 16
#endif
#define HIPGP_FAST_LIST_G0(X) X(2048, HIPGP_EXP_R2048)
#define HIPGP_FAST_LIST_G1(X) X(16, 16)
#define HIPGP_FAST_LIST_G2(X) X(1024, HIPGP_EXP_R1024) X(128, 8, 16)
#define HIPGP_FAST_LIST_G3(X) X(64, 4, 16) X(32, 8, 4)
#define HIPGP_FAST_LIST_G4(X)
#else
#define HIPGP_FAST_LIST_G0(X) X(2048, 16, 8, 16) X(8192, 16, 8, 8, 8)
#define HIPGP_FAST_LIST_G1(X) X(4096, 16, 16, 16) X(16, 16) X(8, 8) X(4, 4)
#define HIPGP_FAST_LIST_G2(X) X(1024, 8, 8, 16) X(512, 4, 8, 16) X(256, 16, 16) X(128, 8, 16)
#define HIPGP_FAST_LIST_G3(X) X(3072, 3, 16, 8, 8) X(1536, 3, 8, 8, 8) X(768, 3, 16, 16) X(64, 4, 16) X(32, 8, 4)
#define HIPGP_FAST_LIST_G4(X) X(640, 5, 8, 16) X(320, 5, 4, 16) X(384, 3, 8, 16) X(192, 3, 4, 16) X(96, 3, 8, 4)
#endif
#define HIPGP_FAST_LIST(X) HIPGP_FAST_LIST_G0(X) HIPGP_FAST_LIST_G1(X) HIPGP_FAST_LIST_G2(X) HIPGP_FAST_LIST_G3(X) HIPGP_FAST_LIST_G4(X)

inline std::vector<int> fast_radices(int Ln) {
    switch (Ln) {
#define X(LEN, ...) case LEN: return std::vector<int>{__VA_ARGS__};
        HIPGP_FAST_LIST(X)
#undef X
        default: return {};
    }
}

inline std::vector<int> choose_radices(int Ln) {
    std::vector<int> r = fast_radices(Ln);
    if (!r.empty()) return r;
    int n = Ln;
    while (n % 5 == 0) { r.push_back(5); n /= 5; }
    while (n % 3 == 0) { r.push_back(3); n /= 3; }
    int e = 0;
    while (n % 2 == 0) { ++e; n /= 2; }
    if (n != 1) throw Error("FFT length " + std::to_string(Ln) + " is not 2^a 3^b 5^c");
    // radix-16 stages first, then one stage for the remainder
    while (e >= 4) { r.push_back(16); e -= 4; }
    if (e == 3) r.push_back(8); else if (e == 2) r.push_back(4); else if (e == 1) r.push_back(2);
    return r;
}

inline double fft_cost(int Ln) {
    std::vector<int> r = choose_radices(Ln);
    double c = 0;
    for (int x : r) c += (x == 3 || x == 5) ? 1.3 : 1.0;
    const bool fast = !fast_radices(Ln).empty();
    return (double)Ln * (c + 0.5) * (fast ? 1.0 : 2.5);    // the generic runtime-radix kernels are ~2.5x slower
}

inline bool is_smooth(long n) {
    for (int p : {2, 3, 5}) while (n % p == 0) n /= p;
    return n == 1;
}

// Shared-memory budgets of the row passes: the generic kernel (pick_rows_tiling, two padded rows at least) and the
// specialised kernels (tile + side buffer).  An embedding whose last-axis row pass would exceed them takes the four-step
// path of long1d_api.inl along that axis instead.  The test-only emulation build lowers HIPGP_ROW_SMEM_MAX with -D to run that path at small sizes.
#ifndef HIPGP_ROW_SMEM_MAX
#define HIPGP_ROW_SMEM_MAX (200 * 1024)
#endif
constexpr size_t kRowsFastSmemMax = 227 * 1024;
// Four-step lengths L = L1 * L2: both factors from HIPGP_FAST_LIST and at most this long, so that one line (fp64: 64 KB)
// and its neighbours fit a CTA's shared memory.
constexpr int kLongMaxFactor = 4096;

// smallest L = L1 * L2 >= n with L1 <= L2 both in HIPGP_FAST_LIST (<= kLongMaxFactor); among equal L the most balanced split
inline bool long_split(long n, int* L1, int* L2) {
    std::vector<int> f;
#define X(LEN, ...) if (LEN <= kLongMaxFactor) f.push_back(LEN);
    HIPGP_FAST_LIST(X)
#undef X
    long best = -1;
    for (int a : f)
        for (int b : f) {
            const long L = (long)a * b;
            if (a > b || L < n) continue;
            if (best < 0 || L < best || (L == best && a > *L1)) { best = L; *L1 = a; *L2 = b; }
        }
    return best > 0;
}

// smallest-cost 2^a 3^b 5^c length >= n (even when `even`), searched in [n, 2n]
inline int choose_length(long n, bool even) {
    if (n < 2) n = 2;
    long best = -1; double bc = 0;
    for (long L = n; L <= 2 * n + 2; ++L) {
        if (even && (L & 1)) continue;
        if (!is_smooth(L)) continue;
        const double c = even ? 2.0 * fft_cost((int)(L / 2)) : fft_cost((int)L);
        if (best < 0 || c < bc) { best = L; bc = c; }
    }
    if (best < 0) throw Error("no embedding length found");
    return (int)best;
}

template <class T>
struct LineFftHost {
    LineFft<T> dev{};
    DevBuf tw, rev, pos, twst;
    std::vector<int> hrev_, hpos_;
    void build(int Ln, size_t* total) {
        std::vector<int> r = Ln > 1 ? choose_radices(Ln) : std::vector<int>();
        if ((int)r.size() > kMaxStages) throw Error("too many FFT stages");
        dev.Ln = Ln; dev.nst = (int)r.size();
        for (size_t i = 0; i < r.size(); ++i) dev.radix[i] = r[i];
        std::vector<cplx<T>> htw(Ln);
        for (int k = 0; k < Ln; ++k) {
            // exact argument reduction: angle = -2 pi k / Ln
            const double a = -2.0 * M_PI * (double)k / (double)Ln;
            htw[k].x = (T)std::cos(a); htw[k].y = (T)std::sin(a);
        }
        // position of frequency k after DIF with radices r[0..]: k = q0 + r0 (q1 + r1 (q2 + ...)),
        // p = q0 Ln/r0 + q1 Ln/(r0 r1) + ...
        std::vector<int> hrev(Ln), hpos(Ln);
        for (int k = 0; k < Ln; ++k) {
            int kk = k, p = 0, span = Ln;
            for (size_t i = 0; i < r.size(); ++i) { span /= r[i]; p += (kk % r[i]) * span; kk /= r[i]; }
            hpos[k] = p; hrev[p] = k;
        }
        tw.ensure(sizeof(cplx<T>) * Ln, total); rev.ensure(sizeof(int) * Ln, total); pos.ensure(sizeof(int) * Ln, total);
        CK(cudaMemcpy(tw.p, htw.data(), sizeof(cplx<T>) * Ln, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(rev.p, hrev.data(), sizeof(int) * Ln, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(pos.p, hpos.data(), sizeof(int) * Ln, cudaMemcpyHostToDevice));
        dev.tw = tw.as<cplx<T>>(); dev.rev = rev.as<int>(); dev.pos = pos.as<int>();
        hrev_ = hrev; hpos_ = hpos;
        // per-stage twiddle tables.  fp32, PAIRED: [(p * S + j) * 2 + e] = exp(-2 pi i j (2p + 1 + e) / Nt), p < R / 2 (unused half = 1);
        // fp64: [(r - 1) * S + j] = exp(-2 pi i j r / Nt)   (fft_engine.cuh: TwLayout)
        std::vector<cplx<T>> st;
        int Nt = Ln;
        auto tw_entry = [](int j, int rr, int Nt_) {
            const long num = ((long)j * rr) % Nt_;
            const double a = -2.0 * M_PI * (double)num / (double)Nt_;
            cplx<T> wv; wv.x = (T)std::cos(a); wv.y = (T)std::sin(a);
            return wv;
        };
        for (size_t i = 0; i < r.size(); ++i) {
            const int R = r[i], S = Nt / R;
            dev.twoff[i] = (int)st.size();
            if (TwLayout<T>::paired) {
                for (int p = 0; p < R / 2; ++p)
                    for (int j = 0; j < S; ++j)
                        for (int e = 0; e < 2; ++e) {
                            const int rr = 2 * p + 1 + e;
                            cplx<T> one; one.x = (T)1; one.y = (T)0;
                            st.push_back(rr < R ? tw_entry(j, rr, Nt) : one);
                        }
            } else {
                for (int rr = 1; rr < R; ++rr)
                    for (int j = 0; j < S; ++j) st.push_back(tw_entry(j, rr, Nt));
            }
            Nt = S;
        }
        if (st.empty()) st.resize(1);
        twst.ensure(sizeof(cplx<T>) * st.size(), total);
        CK(cudaMemcpy(twst.p, st.data(), sizeof(cplx<T>) * st.size(), cudaMemcpyHostToDevice));
        dev.twst = twst.as<cplx<T>>();
    }
    void release(size_t* total) { tw.release(total); rev.release(total); pos.release(total); twst.release(total); }
};

// geometry of one embedding: D active axes with lengths L[d]; the last axis is the real (row) axis
template <class T>
struct Geom {
    int D = 0;
    int L[3] = {1, 1, 1};
    int H = 1;          // L[D-1] / 2
    long P = 0;         // row pitch in complex elements (>= H + 1)
    LineFftHost<T> fcol[2];
    LineFftHost<T> frow;
    DevBuf twL, twLp, part, pairq, pairs, pairw, quadq, quadw;
    int npair0 = 0, nquad = 0;
    // Do the passes take the specialised kernel where their length has one?  fp32 pipelines keep the frequency workspace
    // in lane layout (lane_fft.cuh), which the generic kernels do not read, so an fp32 geometry takes them only when every
    // pass has one; fp64 lanes are plain interleaved complex numbers and the choice is made kernel by kernel (always true).
    bool fast = false;
    bool built = false;
    bool lane_layout() const { return sizeof(T) == 4 && fast; }
    // row_pass = false: a last axis on the four-step path (long1d_api.inl), which owns its own transforms; only the column
    // passes of the leading axes are built.  They run on rows of interleaved complex numbers, so fp32 takes the generic
    // column kernel throughout.
    void build(int D_, const int* L_, size_t* total, bool row_pass = true) {
        D = D_;
        for (int d = 0; d < D; ++d) L[d] = L_[d];
        H = L[D - 1] / 2;
        P = ((long)H + 1 + 7) / 8 * 8;
        bool all_listed = !fast_radices(H).empty();
        for (int d = 0; d + 1 < D; ++d) all_listed = all_listed && !fast_radices(L[d]).empty();
        fast = sizeof(T) == 8 || (row_pass && all_listed);
        for (int d = 0; d + 1 < D; ++d) fcol[d].build(L[d], total);
        if (!row_pass) { H = 0; P = L[D - 1]; built = true; return; }
        frow.build(H, total);
        std::vector<cplx<T>> w(H);
        for (int k = 0; k < H; ++k) {
            const double a = -2.0 * M_PI * (double)k / (double)L[D - 1];
            w[k].x = (T)std::cos(a); w[k].y = (T)std::sin(a);
        }
        twL.ensure(sizeof(cplx<T>) * H, total);
        CK(cudaMemcpy(twL.p, w.data(), sizeof(cplx<T>) * H, cudaMemcpyHostToDevice));
        std::vector<cplx<T>> wp(H); std::vector<int> pt(H);
        for (int q = 0; q < H; ++q) {
            const int k = frow.hrev_[q];
            wp[q] = w[k];
            pt[q] = k == 0 ? 0 : frow.hpos_[H - k];
        }
        std::vector<int> pq;
        for (int q = 0; q < H; ++q) if (q <= pt[q]) pq.push_back(q);
        if ((int)pq.size() != H / 2 + 1) throw Error("internal: r2c pair table has the wrong size");
        pairq.ensure(sizeof(int) * pq.size(), total);
        CK(cudaMemcpy(pairq.p, pq.data(), sizeof(int) * pq.size(), cudaMemcpyHostToDevice));
        // quads for the specialised row kernels: even positions a >= RL (RL = last radix) whose bins (a, a+1) mirror
        // onto (b+1, b) with b even: true for every digit group but group 0 when the list has more than one stage
        {
            const std::vector<int> rad = H > 1 ? choose_radices(H) : std::vector<int>();
            const int RL = rad.empty() ? 1 : rad.back();
            bool ok = rad.size() > 1 && RL % 2 == 0 && H % 2 == 0;
            std::vector<int> qd; std::vector<cplx<T>> qw;
            for (int qa = RL; ok && qa < H; qa += 2) {
                const int pa = pt[qa], pa1 = pt[qa + 1];
                if (pa != pa1 + 1 || (pa1 & 1) || pa1 < RL) { ok = false; break; }
                if (qa <= pa1) { qd.push_back(qa); qd.push_back(pa1); qw.push_back(wp[qa]); qw.push_back(wp[qa + 1]); }
            }
            if (!ok) { qd.clear(); qw.clear(); }
            nquad = (int)(qd.size() / 2);
            npair0 = 0;
            if (ok) { for (int q : pq) if (q < RL) ++npair0; } else npair0 = (int)pq.size();
            if (npair0 + 2 * nquad - (ok ? 0 : 0) < 0) throw Error("internal: quad table");
            std::vector<int> pr; std::vector<cplx<T>> pw;
            for (int q : pq) { pr.push_back(q); pr.push_back(q == 0 ? H : pt[q]); pw.push_back(wp[q]); }
            pairs.ensure(sizeof(int) * pr.size(), total); pairw.ensure(sizeof(cplx<T>) * pw.size(), total);
            CK(cudaMemcpy(pairs.p, pr.data(), sizeof(int) * pr.size(), cudaMemcpyHostToDevice));
            CK(cudaMemcpy(pairw.p, pw.data(), sizeof(cplx<T>) * pw.size(), cudaMemcpyHostToDevice));
            quadq.ensure(sizeof(int) * std::max<size_t>(qd.size(), 2), total); quadw.ensure(sizeof(cplx<T>) * std::max<size_t>(qw.size(), 2), total);
            if (!qd.empty()) {
                CK(cudaMemcpy(quadq.p, qd.data(), sizeof(int) * qd.size(), cudaMemcpyHostToDevice));
                CK(cudaMemcpy(quadw.p, qw.data(), sizeof(cplx<T>) * qw.size(), cudaMemcpyHostToDevice));
            }
        }
        twLp.ensure(sizeof(cplx<T>) * H, total); part.ensure(sizeof(int) * H, total);
        CK(cudaMemcpy(twLp.p, wp.data(), sizeof(cplx<T>) * H, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(part.p, pt.data(), sizeof(int) * H, cudaMemcpyHostToDevice));
        built = true;
    }
    long spec_elems() const { long n = P; for (int d = 0; d + 1 < D; ++d) n *= L[d]; return n; }
    void release(size_t* total) { for (auto& f : fcol) f.release(total); frow.release(total); twL.release(total); twLp.release(total); part.release(total); pairq.release(total); pairs.release(total); pairw.release(total); quadq.release(total); quadw.release(total); built = false; }
};

// four-step geometry of a long last axis (long1d_kernels.cuh): the two line FFTs and the twiddle tables, fp64-computed
template <class T>
struct LongGeom {
    int L1 = 0, L2 = 0;
    LineFftHost<T> f1, f2;
    DevBuf twh, twl;
    bool built = false;
    void build(int L1_, int L2_, size_t* total) {
        L1 = L1_; L2 = L2_;
        f1.build(L1, total); f2.build(L2, total);
        std::vector<cplx<T>> h(L1), l(L2);
        for (int j = 0; j < L1; ++j) { const double a = -2.0 * M_PI * (double)j / (double)L1; h[j].x = (T)std::cos(a); h[j].y = (T)std::sin(a); }
        for (int j = 0; j < L2; ++j) { const double a = -2.0 * M_PI * (double)j / ((double)L1 * L2); l[j].x = (T)std::cos(a); l[j].y = (T)std::sin(a); }
        twh.ensure(sizeof(cplx<T>) * L1, total); twl.ensure(sizeof(cplx<T>) * L2, total);
        CK(cudaMemcpy(twh.p, h.data(), sizeof(cplx<T>) * L1, cudaMemcpyHostToDevice));
        CK(cudaMemcpy(twl.p, l.data(), sizeof(cplx<T>) * L2, cudaMemcpyHostToDevice));
        built = true;
    }
    void release(size_t* total) { f1.release(total); f2.release(total); twh.release(total); twl.release(total); built = false; }
};

struct RowsFusion {
    int mode = 0, dot_kind = 0;
    const void* in = nullptr; void* out = nullptr; void* v0 = nullptr; void* v1 = nullptr; const void* v2 = nullptr;
};

}  // namespace hipgp

using namespace hipgp;

// ---------------------------------------------------------------------------------------------
struct hipgp_plan {
    int dtype = 0, device = 0;
    int ndim_user = 0;
    std::vector<long> m_user;
    int D = 0;                 // active axes (m > 1); at least 1
    int m[3] = {1, 1, 1}, N[3] = {1, 1, 1};
    long M = 1, E = 1;
    int Ln[3] = {1, 1, 1}, Lw[3] = {1, 1, 1};
    size_t dev_bytes = 0;
    long launches = 0;
    bool have_spec = false, have_wide = false;
    bool wide_real = false;    // wide embedding long enough for symmetric taps: real spectrum for R^T / R
    double clampv = 1e-6;
    long nclamped = 0;

    Geom<float> gn32, gw32;    // narrow (K, Cinv) / wide (RT, R) geometries in the plan dtype
    Geom<double> gn64, gw64;   // fp64 geometries (set-up always runs in fp64; also the fp64 plan's own)
    // embeddings whose last axis is too long for the row pass run that axis on the four-step path (long1d_api.inl): narrow /
    // wide, each decided on its own; lsplit = (L1, L2) of the narrow, wide and Bluestein (DCT-I set-up of a 1-D plan, only
    // when the narrow one is long) lengths.  gn / gw then hold the column passes of the leading axes only.
    bool long_n = false, long_w = false;
    int lsplit[3][2] = {{0, 0}, {0, 0}, {0, 0}};
    LongGeom<float> ln32, lw32;
    LongGeom<double> ln64, lw64, lb64;
    DevBuf bluA, bluSpec;                  // Bluestein work array and the chirp's spectrum (built once per plan)
    bool have_blu = false, long_first = false;
    DevBuf specK, specCinv, specW;         // stored spectra (plan dtype; specW complex)
    DevBuf Dm, Dinv, Dsqrt, colK, colG, colS, tmpA, tmpB, counts;   // fp64 set-up arrays (M each)
    DevBuf W1, W2;                         // frequency-domain workspace
    DevBuf vr, vp, vz, vAp, partial, scal, cnt, flags;   // PCG state
    DevBuf stage_in, stage_out;            // device staging for the *_host entry points
    DevBuf slabSpecK, slabSpecCinv;        // this rank's bins of the spectra, [L0][L1][Pq] (slab decomposition)
    bool have_slabK = false, have_slabCinv = false;
    DevBuf costabs[3], cosmats[3];                     // DCT-I cosine tables per active axis (built once per plan)
    DevBuf gradA;                          // R^T column gradient (corr_api.inl): one M-sized fp64 work array
    DevBuf corrU, corrV, corrS, corrLag;   // Toeplitz-column quadratic form (corr_api.inl): spectra of a chunk of pairs, their sum, lags
    void* pinned = nullptr;                // host flags mirror
    cudaStream_t copy_streams[2] = {nullptr, nullptr};   // H2D / D2H streams of hipgp_pcg_host_pipelined
    // asynchronous host solves (hipgp_pcg_host_submit / _wait): two slots, each with its own device staging and events
    DevBuf slot_in[2], slot_out[2];
    cudaEvent_t slot_ev[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};     // upload done, solved, download done
    bool slot_busy[2] = {false, false};
    int* slot_flags = nullptr;             // pinned: 4 ints per slot
    long pcg_B = 0;
    // peer-memory exchange (bins layout): R1 receives the way there, R2 the way back; peerR*[q] = rank q's buffers as mapped here
    DevBuf slabR1, slabR2;
    void* peerR1[16] = {}; void* peerR2[16] = {};
    void* ipc_opened[32] = {}; int n_ipc_opened = 0;
    bool peers_ready = false;
    int slab_chunks = 1;                     // bins layout: the exchange is cut into this many independent all-to-alls
    int slab_rank = 0, slab_nranks = 1;      // slab-decomposed grid (axis 0 split over ranks); 1 = not decomposed
    void* run_x = nullptr; long run_B = 0; bool run_precond = true; double run_tol = 0; bool run_active = false;   // begin/step state
    // optional per-kernel-class timing (bench.py roofline): CUDA events around every launch
    bool profiling = false;
    struct ProfRec { int cls; cudaEvent_t e0, e1; };
    std::vector<ProfRec> prof;
    double prof_ms[4] = {0, 0, 0, 0};
    long prof_n[4] = {0, 0, 0, 0};
};

#ifdef HIPGP_EMU
#define PROF_BEGIN(pl, cls, st) ((void)0)
#define PROF_END(pl, st) ((void)0)
#else
#define PROF_BEGIN(pl, cls_, st)                                                   \
    if ((pl)->profiling) {                                                         \
        hipgp_plan::ProfRec r__; r__.cls = (cls_);                                 \
        cudaEventCreate(&r__.e0); cudaEventCreate(&r__.e1);                        \
        cudaEventRecord(r__.e0, (st)); (pl)->prof.push_back(r__);                  \
    }
#define PROF_END(pl, st) if ((pl)->profiling) cudaEventRecord((pl)->prof.back().e1, (st));
#endif


// ---- per-length launchers of the specialised kernels.  Declared here, DEFINED in fast_launch.cuh and explicitly
// instantiated by fast_inst.cu (compiled once per length group so that the build runs in parallel). ----
namespace hipgp {
template <class T, int LEN> void launch_rows_fast_len(hipgp_plan* pl, bool inverse, RowsParams<T>& P, cudaStream_t st);
template <class T, int LEN> void launch_cols_fast_len(hipgp_plan* pl, ColsParams<T>& P, long n_outer, long B, cudaStream_t st);   // throws: lanes not 16-byte aligned
template <class T, int LEN> bool rows_fast_fits_len(long n_real);   // does the row pass of this length fit rows of n_real samples?
}
