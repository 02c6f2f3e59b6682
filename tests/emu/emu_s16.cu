// tests/emu/emu_s16.cu -- CPU emulation of the kernel bodies for 16-bit PCM inputs (TEST ONLY).
//
// Runs the kernel bodies like emu.cu, with runners that set the kernels' load flags the way the
// product does: one load of both elements of a packed point where the base is aligned to two elements
// (4 bytes for int16), two element loads otherwise; the fp32 / fp64 runners can force either.  Every
// runner is a template on the input type, so the int16_t instantiation and the double instantiation
// it is compared with run the same host code, and every runner returns the whole
// peak record (packed key, second-peak and seed order bits) next to the resolved index / peak /
// second peak.  Compiled by tests/test_pcm_s16_emu.py; never linked into the product.  It does not
// include emu.cu, whose other instantiations would double the compile time.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "fft_plan.h"
#include "gen_plan.h"

using namespace asc;

// the executor of emu.cu: every phase for all thread ids in turn, the same argmax merge rules
struct HostExec {
    int bx_, by_, bz_, nt;
    int bx() const { return bx_; }
    int by() const { return by_; }
    int bz() const { return bz_; }
    template <class F>
    void phase(F&& f) {
        for (int t = 0; t < nt; t++) f(t);
    }
    template <class F>
    void single(F&& f) { f(); }
    bool any(bool b) const { return b; }
    float warp_second(float /*best_mag*/, float second) const { return second; }
    unsigned long long peek_key(const unsigned long long* k) const { return *k; }
    unsigned int peek_bits(const unsigned int* k) const { return *k; }
    template <class F>
    void phase_argmax(F&& f, unsigned long long* dst, unsigned int* dst_second, void* /*scratch*/) {
        unsigned long long best = 0;
        float second = 0.0f;
        for (int t = 0; t < nt; t++) {
            const ArgmaxPair k = f(t);
            argmax_merge(best, second, k.best, k.second);
        }
        const unsigned long long old = *dst;
        if (best > old) *dst = best;
        if (old != best) argmax_merge(best, second, old, 0.0f);
        const unsigned int sb = float_order_bits(second);
        if (sb > *dst_second) *dst_second = sb;
    }
};

// one pair's record, as tests/test_pcm_s16_emu.py reads it
struct Rec {
    long long raw_index;
    double peak, second;
    unsigned long long key;
    unsigned second_bits, seed_bits;
};

namespace {

// the product's rule (static_plan_impl.cuh, run_small_wave, GenStage::col_fwd) for one packed pair:
// one load of two elements where the base is aligned to two elements and the pitch is even.  vec >= 0
// overrides it (the emulator reads any address, so both branches can run on the same arrays).
template <typename InT>
int vec_ok(const InT* p, long long pitch, int vec = -1) {
    if (vec >= 0) return vec;
    return reinterpret_cast<uintptr_t>(p) % (2 * sizeof(InT)) == 0 && pitch % 2 == 0;
}

void from_peak(const PairPeak& pk, double scale, Rec* r) {
    r->raw_index = (long long)argmax_key_index(pk.key);
    r->peak = (double)argmax_key_value(pk.key) * scale;
    r->second = (double)pair_second(pk) * scale;
    r->key = pk.key; r->second_bits = pk.second_bits; r->seed_bits = pk.seed_bits;
}

// static four-step plan: K_A through its register path, K_B, K_C
template <class P, typename InT>
void static_plan(const InT* source, const InT* sample, PairPeak* peak, int vec = -1) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    constexpr int M1 = Col::n, M2 = Row::n;
    const long long M = P::L;
    std::vector<cplx> planes(2 * M);
    std::vector<cplx> col_tw = build_pass_tables(radix_vector<Col>());
    std::vector<cplx> row_tw = build_pass_tables(radix_vector<Row>());
    std::vector<cplx> col_tc = build_col_tc(M, Col::weight(Col::count - 1));
    std::vector<cplx> row_rev = build_row_rev<Row>();
    std::vector<cplx> row_tab = build_row_tab<Row>(M, M1);
    std::vector<cplx> m_lo, m_hi;
    build_two_level(M, M - 1, m_lo, m_hi);
    peak->key = 12345ull; peak->second_bits = 777u; peak->seed_bits = 777u;   // garbage: K_A must clear them
    {
        using K = ColFwdKernel<Col, Row::n, P::NT_COL, InT, false>;
        typename K::Params p{source, sample, planes.data(), peak, col_tw.data(), col_tc.data(), m_lo.data(), m_hi.data(), M,
                             2 * M, M, vec_ok(source, 2 * M, vec), vec_ok(sample, M, vec)};
        std::vector<cplx> smem(K::SMEM / sizeof(cplx));
        for (int sig = 0; sig < 2; sig++)
            for (int tile = 0; tile < M2 / COL_T; tile++) {
                HostExec ex{tile, sig, 0, K::THREADS};
                K::run(ex, p, smem.data());
            }
    }
    {
        using K = RowFusedKernel<Row, Col::n, P::NT_ROW>;
        typename K::Params p{planes.data(), row_tw.data(), row_rev.data(), m_lo.data(), m_hi.data(), M, row_tab.data()};
        std::vector<cplx> smem(K::SMEM / sizeof(cplx));
        for (int r = 0; r <= M1 / 2; r++) {
            HostExec ex{r, 0, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    }
    {
        using K = ColInvKernel<Col, Row::n, P::NT_COL>;
        typename K::Params p{planes.data(), peak, col_tw.data(), M};
        std::vector<cplx> smem(K::SMEM / sizeof(cplx));
        for (int tile = 0; tile < M2 / COL_T; tile++) {
            HostExec ex{0, tile, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    }
}

template <typename InT, bool PHAT = false>
int small_plan(const InT* source, const InT* sample, long long L, PairPeak* peak, int vec = -1) {
    SmallPlan pl;
    if (!make_small_plan(L, &pl)) return -1;
    std::vector<cplx> wm = build_full_table(L, L), wn = build_full_table(2 * L, L);
    using K = SmallXcorrKernel<InT, PHAT>;
    typename K::Params p{source, sample, peak, wm.data(), wn.data(), pl, 2 * L, L, vec_ok(source, 2 * L, vec),
                         vec_ok(sample, L, vec)};
    std::vector<cplx> smem(K::smem_bytes((int)L) / sizeof(cplx));
    peak->key = 12345ull; peak->second_bits = 777u; peak->seed_bits = 777u;   // garbage: the kernel must clear them
    HostExec ex{0, 0, 0, K::THREADS};
    K::run(ex, p, smem.data());
    return 0;
}

// runtime-radix four-step kernels, T = arithmetic type
template <typename T, typename InT>
int generic_plan(const InT* source, const InT* sample, long long L, Rec* out) {
    typedef typename GenTraits<T>::C C;
    GenShape sh;
    if (!gen_make_shape(L, sizeof(T) == 8, &sh)) return -1;
    const GenTables<C> tb = gen_build_tables<C>(sh);
    std::vector<C> planes(2 * sh.M);
    PairPeak pk;
    memset(&pk, 0, sizeof(pk));
    pk.key = 12345ull; pk.second_bits = 777u; pk.seed_bits = 777u;   // garbage: G_A must clear them
    auto col_fwd = [&](auto KK) {
        using K = decltype(KK);
        typename K::Params p{source, sample, planes.data(), &pk, tb.wcol.data(), tb.m_lo.data(), tb.m_hi.data(),
                             tb.p2f_col.data(), sh, 2 * L, L, vec_ok(source, 2 * L), vec_ok(sample, L)};
        std::vector<C> smem(K::smem_bytes(sh) / sizeof(C) + 1);
        for (int sig = 0; sig < 2; sig++)
            for (int tile = 0; tile < (sh.M2 + K::CT - 1) / K::CT; tile++) {
                HostExec ex{tile, sig, 0, K::THREADS};
                K::run(ex, p, smem.data());
            }
    };
    if (sh.nt_col == GEN_THREADS) { if (sh.ct == 16) col_fwd(GenColFwdKernel<T, InT, 16, GEN_THREADS>{}); else col_fwd(GenColFwdKernel<T, InT, 8, GEN_THREADS>{}); }
    else { if (sh.ct == 16) col_fwd(GenColFwdKernel<T, InT, 16, GEN_THREADS_SMALL>{}); else col_fwd(GenColFwdKernel<T, InT, 8, GEN_THREADS_SMALL>{}); }
    auto rows = [&](auto KK) {
        using K = decltype(KK);
        typename K::Params p{planes.data(), tb.wrow.data(), tb.wpos.data(), tb.m_lo.data(), tb.m_hi.data(),
                             tb.f2p_row.data(), sh};
        std::vector<C> smem(K::smem_bytes(sh) / sizeof(C) + 1);
        for (int r = 0; r <= sh.M1 / 2; r++) {
            HostExec ex{r, 0, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    };
    if (sh.nt_row == GEN_THREADS) rows(GenRowFusedKernel<T, GEN_THREADS>{}); else rows(GenRowFusedKernel<T, GEN_THREADS_SMALL>{});
    auto col_inv = [&](auto KK) {
        using K = decltype(KK);
        typename K::Params p{planes.data(), &pk, tb.wcol.data(), tb.p2f_col.data(), sh, reinterpret_cast<T*>(planes.data())};
        std::vector<C> smem(K::smem_bytes(sh) / sizeof(C) + 1);
        for (int tile = 0; tile < (sh.M2 + K::CT - 1) / K::CT; tile++) {
            HostExec ex{0, tile, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    };
    if (sh.nt_col == GEN_THREADS) { if (sh.ct == 16) col_inv(GenColInvKernel<T, 16, GEN_THREADS>{}); else col_inv(GenColInvKernel<T, 8, GEN_THREADS>{}); }
    else { if (sh.ct == 16) col_inv(GenColInvKernel<T, 16, GEN_THREADS_SMALL>{}); else col_inv(GenColInvKernel<T, 8, GEN_THREADS_SMALL>{}); }
    const double scale = gen_peak_scale(sh);
    if (sizeof(T) == 4) {
        from_peak(pk, scale, out);
        return 0;
    }
    // fp64: r[0 .. 2L) sits in plane 1; resolved like argmax_f64_kernel (reference :52-67)
    const T* r = reinterpret_cast<const T*>(planes.data()) + 2 * sh.M;
    long long best = 0;
    double bv = (double)r[0];
    for (long long i = 1; i < 2 * L; i++)
        if (fabs((double)r[i]) > bv) { bv = fabs((double)r[i]); best = i; }
    double second = 0.0;
    for (long long i = 0; i < 2 * L; i++)
        if (i != best && fabs((double)r[i]) > second) second = fabs((double)r[i]);
    *out = Rec{best, (double)r[best] * scale, second * scale, 0ull, 0u, 0u};
    return 0;
}

// the product's AUTO / FFT choice of plan; the direct path has no transform to emulate (-2).  PHAT:
// the single-CTA kernel's PHAT twin (-3 for the four-step plans, whose PHAT rows are not emulated here)
template <typename InT, bool PHAT = false>
int xcorr(const InT* source, const InT* sample, long long L, int forced, Rec* out, int* path, int vec = -1) {
    const PathKind kind = choose_path(L, forced);
    *path = (int)kind;
    PairPeak pk;
    memset(&pk, 0, sizeof(pk));
    if (kind == PATH_STATIC_FFT) {
        int rc = -1;
        for_each_static_plan([&](auto P) {
            using PT = decltype(P);
            if (PT::L != L) return;
            if (PHAT) { rc = -3; return; }
            static_plan<PT, InT>(source, sample, &pk, vec);
            rc = 0;
        });
        if (rc != 0) return rc;
    } else if (kind == PATH_SMALL_FFT) {
        if (small_plan<InT, PHAT>(source, sample, L, &pk, vec) != 0) return -1;
    } else if (kind == PATH_GENERIC_FFT) {
        if (PHAT) return -3;
        return generic_plan<float, InT>(source, sample, L, out);
    } else {
        return -2;
    }
    from_peak(pk, 1.0, out);
    return 0;
}

}  // namespace

extern "C" {

// one pair through the plan the product picks (forced: AUTO / FFT)
int emu16_xcorr_s16(const int16_t* source, const int16_t* sample, long long L, int forced, Rec* out, int* path) {
    return xcorr<int16_t>(source, sample, L, forced, out, path);
}
int emu16_xcorr_f64(const double* source, const double* sample, long long L, int forced, Rec* out, int* path) {
    return xcorr<double>(source, sample, L, forced, out, path);
}
// the runtime-radix kernels; precise != 0: fp64 arithmetic
int emu16_generic_s16(const int16_t* source, const int16_t* sample, long long L, int precise, Rec* out) {
    return precise ? generic_plan<double, int16_t>(source, sample, L, out) : generic_plan<float, int16_t>(source, sample, L, out);
}
int emu16_generic_f64(const double* source, const double* sample, long long L, int precise, Rec* out) {
    return precise ? generic_plan<double, double>(source, sample, L, out) : generic_plan<float, double>(source, sample, L, out);
}
// fp32 / fp64 inputs through K_A's register path (static lengths) or the single-CTA kernel (phat != 0:
// its PHAT twin) with both load flags forced to `vec`: one load of two elements, or two element loads
int emu16_xcorr_vec_f32(const float* source, const float* sample, long long L, int phat, int vec, Rec* out, int* path) {
    return phat ? xcorr<float, true>(source, sample, L, 0, out, path, vec) : xcorr<float>(source, sample, L, 0, out, path, vec);
}
int emu16_xcorr_vec_f64(const double* source, const double* sample, long long L, int phat, int vec, Rec* out, int* path) {
    return phat ? xcorr<double, true>(source, sample, L, 0, out, path, vec) : xcorr<double>(source, sample, L, 0, out, path, vec);
}

}
