// tests/emu/emu_phat.cu -- CPU emulation of the PHAT-weighted kernel bodies (TEST ONLY).
//
// Runs the PHAT twins of the row kernels (static RowFusedKernel, the same kernel with a run-time row
// count as the rows of a runtime-radix fp32 plan, GenRowFusedKernel in fp32 and fp64 arithmetic) and
// of the single-CTA kernel, with the unweighted column kernels around them and the split tables the
// product builds, on f64 inputs (the F64 call).  Every runner returns the resolved index / peak /
// second peak at the reference's scale (x N) and the packed peak record of the fp32-argmax paths.
// Compiled by tests/test_phat_emu.py; never linked into the product.  The executor is emu_s16.cu's.
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "fft_plan.h"
#include "gen_plan.h"

using namespace asc;

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

struct Rec {
    long long raw_index;
    double peak, second;
    unsigned long long key;
    unsigned second_bits, seed_bits;
};

namespace {

void from_peak(const PairPeak& pk, double scale, Rec* r) {
    r->raw_index = (long long)argmax_key_index(pk.key);
    r->peak = (double)argmax_key_value(pk.key) * scale;
    r->second = (double)pair_second(pk) * scale;
    r->key = pk.key; r->second_bits = pk.second_bits; r->seed_bits = pk.seed_bits;
}

// static four-step plan: K_A (register path), the PHAT row kernel, K_C
template <class P>
void static_plan(const double* source, const double* sample, PairPeak* peak) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    constexpr int M1 = Col::n, M2 = Row::n;
    const long long M = P::L;
    std::vector<cplx> planes(2 * M);
    std::vector<cplx> col_tw = build_pass_tables(radix_vector<Col>());
    std::vector<cplx> row_tw = build_pass_tables(radix_vector<Row>());
    std::vector<cplx> col_tc = build_col_tc(M, Col::weight(Col::count - 1));
    std::vector<cplx> row_tab = build_row_tab<Row>(M, M1);
    std::vector<cplx> m_lo, m_hi, n_lo, n_hi;
    build_two_level(M, M - 1, m_lo, m_hi);
    build_two_level(2 * M, M1 / 2, n_lo, n_hi);             // as build_static_plan for PHAT
    std::vector<cplx> rev_h = build_row_rev_half<Row>();
    peak->key = 12345ull; peak->second_bits = 777u; peak->seed_bits = 777u;   // garbage: K_A must clear them
    {
        using K = ColFwdKernel<Col, Row::n, P::NT_COL, double, false>;
        typename K::Params p{source, sample, planes.data(), peak, col_tw.data(), col_tc.data(), m_lo.data(), m_hi.data(), M, 2 * M, M};
        std::vector<cplx> smem(K::SMEM / sizeof(cplx));
        for (int sig = 0; sig < 2; sig++)
            for (int tile = 0; tile < M2 / COL_T; tile++) {
                HostExec ex{tile, sig, 0, K::THREADS};
                K::run(ex, p, smem.data());
            }
    }
    {
        using K = RowFusedKernel<Row, Col::n, P::NT_ROW, true>;
        typename K::Params p{planes.data(), row_tw.data(), rev_h.data(), n_lo.data(), n_hi.data(), M, row_tab.data()};
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

int small_plan(const double* source, const double* sample, long long L, PairPeak* peak) {
    SmallPlan pl;
    if (!make_small_plan(L, &pl)) return -1;
    std::vector<cplx> wm = build_full_table(L, L), wn = build_full_table(2 * L, L);
    using K = SmallXcorrKernel<double, true>;
    typename K::Params p{source, sample, peak, wm.data(), wn.data(), pl, 2 * L, L, 1, 1};
    std::vector<cplx> smem(K::smem_bytes((int)L) / sizeof(cplx));
    peak->key = 12345ull; peak->second_bits = 777u; peak->seed_bits = 777u;
    HostExec ex{0, 0, 0, K::THREADS};
    K::run(ex, p, smem.data());
    return 0;
}

// the rows of a runtime-radix fp32 plan on the static row kernel's PHAT twin (static_rows.cu)
template <class RL, int NT>
void static_rows_phat(std::vector<cplx>& planes, const GenShape& sh) {
    using K = RowFusedKernel<RL, 0, NT, true>;
    std::vector<cplx> row_tw = build_pass_tables(radix_vector<RL>());
    std::vector<cplx> row_tab = build_row_tab<RL>(sh.M, sh.M1);
    std::vector<cplx> rev_h = build_row_rev_half<RL>(), n_lo, n_hi;
    build_two_level(2 * sh.M, sh.M1 / 2, n_lo, n_hi);
    typename K::Params p{planes.data(), row_tw.data(), rev_h.data(), n_lo.data(), n_hi.data(), sh.M, row_tab.data(), sh.M1};
    std::vector<cplx> smem(K::SMEM / sizeof(cplx));
    for (int r = 0; r <= sh.M1 / 2; r++) {
        HostExec ex{r, 0, 0, K::THREADS};
        K::run(ex, p, smem.data());
    }
}

// runtime-radix four-step kernels with the PHAT row kernel, T = arithmetic type.  static_rows: the
// product's choice for fp32 plans whose M2 has a static row kernel.
template <typename T>
int generic_plan(const double* source, const double* sample, long long L, Rec* out, int* static_rows_used) {
    typedef typename GenTraits<T>::C C;
    GenShape sh;
    if (!gen_make_shape(L, sizeof(T) == 8, &sh) || sh.M != L) return -1;
    const GenTables<C> tb = gen_build_tables<C>(sh);
    std::vector<C> planes(2 * sh.M);
    PairPeak pk;
    memset(&pk, 0, sizeof(pk));
    pk.key = 12345ull; pk.second_bits = 777u; pk.seed_bits = 777u;
    auto col_fwd = [&](auto KK) {
        using K = decltype(KK);
        typename K::Params p{source, sample, planes.data(), &pk, tb.wcol.data(), tb.m_lo.data(), tb.m_hi.data(),
                             tb.p2f_col.data(), sh, 2 * L, L, 1, 1};
        std::vector<C> smem(K::smem_bytes(sh) / sizeof(C) + 1);
        for (int sig = 0; sig < 2; sig++)
            for (int tile = 0; tile < (sh.M2 + K::CT - 1) / K::CT; tile++) {
                HostExec ex{tile, sig, 0, K::THREADS};
                K::run(ex, p, smem.data());
            }
    };
    if (sh.nt_col == GEN_THREADS) { if (sh.ct == 16) col_fwd(GenColFwdKernel<T, double, 16, GEN_THREADS>{}); else col_fwd(GenColFwdKernel<T, double, 8, GEN_THREADS>{}); }
    else { if (sh.ct == 16) col_fwd(GenColFwdKernel<T, double, 16, GEN_THREADS_SMALL>{}); else col_fwd(GenColFwdKernel<T, double, 8, GEN_THREADS_SMALL>{}); }
    double scale = gen_peak_scale(sh);
    *static_rows_used = 0;
    if constexpr (sizeof(T) == 4) {
        if (sh.static_rows) {
            *static_rows_used = 1;
            scale *= 2.0;                                   // the static row kernel applies the merge's 1/2
            switch (sh.M2) {
                case 480: static_rows_phat<Plan144k::Row, Plan144k::NT_ROW>(planes, sh); break;
                case 960: static_rows_phat<Plan288k::Row, Plan288k::NT_ROW>(planes, sh); break;
                case 1200: static_rows_phat<Plan720k::Row, Plan720k::NT_ROW>(planes, sh); break;
                default: static_rows_phat<Plan1440k::Row, Plan1440k::NT_ROW>(planes, sh); break;
            }
        }
    }
    if (!*static_rows_used) {
        auto rows = [&](auto KK) {
            using K = decltype(KK);
            typename K::Params p{planes.data(), tb.wrow.data(), tb.wpos.data(), tb.m_lo.data(), tb.m_hi.data(),
                                 tb.f2p_row.data(), sh, tb.phat_pos.data(), tb.phat_lo.data(), tb.phat_hi.data()};
            std::vector<C> smem(K::smem_bytes(sh) / sizeof(C) + 1);
            for (int r = 0; r <= sh.M1 / 2; r++) {
                HostExec ex{r, 0, 0, K::THREADS};
                K::run(ex, p, smem.data());
            }
        };
        if (sh.nt_row == GEN_THREADS) rows(GenRowFusedKernel<T, GEN_THREADS, true>{});
        else rows(GenRowFusedKernel<T, GEN_THREADS_SMALL, true>{});
    }
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

}  // namespace

extern "C" {

// one pair through the plan a PHAT context picks (AUTO, fp32); *path: PathKind, -1 when refused
int emuphat_xcorr(const double* source, const double* sample, long long L, Rec* out, int* path) {
    const char* why = nullptr;
    const PathKind kind = choose_path_phat(L, AUDIOSYNC_CUDA_PATH_AUTO, false, &why);
    *path = kind == PATH_NONE ? -1 : (int)kind;
    PairPeak pk;
    memset(&pk, 0, sizeof(pk));
    if (kind == PATH_STATIC_FFT) {
        for_each_static_plan([&](auto P) {
            if (decltype(P)::L == L) static_plan<decltype(P)>(source, sample, &pk);
        });
    } else if (kind == PATH_SMALL_FFT) {
        if (small_plan(source, sample, L, &pk) != 0) return -1;
    } else if (kind == PATH_GENERIC_FFT) {
        int sr = 0;
        return generic_plan<float>(source, sample, L, out, &sr);
    } else {
        return -1;
    }
    from_peak(pk, 1.0, out);
    return 0;
}
// the runtime-radix kernels; precise != 0: fp64 arithmetic.  *static_rows: the rows ran on the static
// row kernel's PHAT twin
int emuphat_generic(const double* source, const double* sample, long long L, int precise, Rec* out, int* static_rows) {
    return precise ? generic_plan<double>(source, sample, L, out, static_rows)
                   : generic_plan<float>(source, sample, L, out, static_rows);
}
// choose_path_phat: PathKind or -1 (refused) for (L, forced path, precise)
int emuphat_path(long long L, int forced, int precise) {
    const char* why = nullptr;
    const PathKind k = choose_path_phat(L, forced, precise != 0, &why);
    return k == PATH_NONE ? -1 : (int)k;
}

}
