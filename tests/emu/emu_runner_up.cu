// tests/emu/emu_runner_up.cu -- CPU emulation of the runner-up kernel bodies (TEST ONLY).
//
// Runs the runner-up twins of the static K_C (ColInvKernel<..., WIN, !OUT, RU>), of the runtime-radix
// fp32 inverse column kernel (GenColInvKernel<float, CT, NT, true, false, true>) and of the single-CTA
// kernel (SmallXcorrKernel<double, false, true, false, false, true>), with the unwindowed forward and
// row kernels before them, on f64 inputs.  The centre comes, as on the device, from a batch record
// (here one whose raw_index the caller sets).  fp64 runtime-radix plans search r in
// argmax_f64_runner_up_kernel, whose body needs warp shuffles: its rule is restated here.  Every
// runner returns the resolved index / peak / second peak at the reference's scale (x N).
// Compiled by tests/golden/emu_build.py for the tests; never linked into the product.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
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

template <class P>
void static_plan(const double* source, const double* sample, const RunnerUp& ru, PairPeak* peak) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    constexpr int M1 = Col::n, M2 = Row::n;
    const long long M = P::L;
    std::vector<cplx> planes(2 * M);
    std::vector<cplx> col_tw = build_pass_tables(radix_vector<Col>());
    std::vector<cplx> row_tw = build_pass_tables(radix_vector<Row>());
    std::vector<cplx> col_tc = build_col_tc(M, Col::weight(Col::count - 1));
    std::vector<cplx> row_tab = build_row_tab<Row>(M, M1);
    std::vector<cplx> row_rev = build_row_rev<Row>();
    std::vector<cplx> m_lo, m_hi;
    build_two_level(M, M - 1, m_lo, m_hi);
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
        using K = RowFusedKernel<Row, Col::n, P::NT_ROW>;
        typename K::Params p{planes.data(), row_tw.data(), row_rev.data(), m_lo.data(), m_hi.data(), M, row_tab.data()};
        std::vector<cplx> smem(K::SMEM / sizeof(cplx));
        for (int r = 0; r <= M1 / 2; r++) {
            HostExec ex{r, 0, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    }
    auto col_inv = [&](auto KK, auto fill) {
        using K = decltype(KK);
        typename K::Params p{};
        static_cast<typename K::PlainParams&>(p) = {planes.data(), peak, col_tw.data(), M, full_window(M)};
        fill(p);
        std::vector<cplx> smem(K::SMEM / sizeof(cplx));
        for (int tile = 0; tile < M2 / COL_T; tile++) {
            HostExec ex{0, tile, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    };
    peak->key = 0ull; peak->second_bits = 0u; peak->seed_bits = 0u;   // the library clears the second PairPeak array
    col_inv(ColInvKernel<Col, Row::n, P::NT_COL, true, true, false, true>{}, [&](auto& p) { p.ru = ru; });
}

int small_plan(const double* source, const double* sample, long long L, const RunnerUp& ru, PairPeak* peak) {
    SmallPlan pl;
    if (!make_small_plan(L, &pl)) return -1;
    std::vector<cplx> wm = build_full_table(L, L), wn = build_full_table(2 * L, L);
    peak->key = 12345ull; peak->second_bits = 777u; peak->seed_bits = 777u;
    auto go = [&](auto KK, auto fill) {
        using K = decltype(KK);
        typename K::Params p{};
        static_cast<typename K::PlainParams&>(p) = {source, sample, peak, wm.data(), wn.data(), pl, 2 * L, L, 1, 1, full_window(L)};
        fill(p);
        std::vector<cplx> smem(K::smem_bytes((int)L) / sizeof(cplx));
        HostExec ex{0, 0, 0, K::THREADS};
        K::run(ex, p, smem.data());
    };
    go(SmallXcorrKernel<double, false, true, false, false, true>{}, [&](auto& p) { p.ru = ru; });
    return 0;
}

// argmax_f64_runner_up_kernel's rule: allowed indices in ascending order, r[0] the signed seed when
// allowed, strict >, a NaN never wins (but beats the empty start on index order), second = largest
// non-NaN |r| over the other allowed indices; an empty set gives raw_index -1
template <typename T>
void argmax_window_f64(const T* r, long long N, const PairWindow* win, Rec* out, double scale) {
    long long best = -1;
    double bv = -INFINITY;
    bool seeded = false;
    for (long long i = 0; i < N; i++) {
        if (win && !win->allows((uint32_t)i)) continue;
        const double x = (double)r[i], a = std::fabs(x);
        double v;
        if (i == 0) { v = std::isnan(x) ? INFINITY : x; seeded = true; }
        else v = std::isnan(a) ? -INFINITY : a;
        if (best < 0 || v > bv) { best = i; bv = v; }
    }
    (void)seeded;
    if (best < 0) { *out = Rec{-1, 0.0, 0.0, 0ull, 0u, 0u}; return; }
    double second = 0.0;
    for (long long i = 0; i < N; i++) {
        if (i == best || (win && !win->allows((uint32_t)i))) continue;
        const double a = std::fabs((double)r[i]);
        if (a == a && a > second) second = a;
    }
    *out = Rec{best, (double)r[best] * scale, second * scale, 0ull, 0u, 0u};
}

// runtime-radix four-step kernels (unwindowed rows), T = arithmetic type.  *static_rows: the product
// ran the rows on a static row kernel (fp32 plans whose M2 has one); the emulation always uses the
// runtime-radix row kernel, whose peak_scale is gen_peak_scale.
template <typename T>
int generic_plan(const double* source, const double* sample, long long L, const RunnerUp& ru, Rec* out) {
    typedef typename GenTraits<T>::C C;
    GenShape sh;
    if (!gen_make_shape(L, sizeof(T) == 8, &sh)) return -1;
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
    const double scale = gen_peak_scale(sh);
    auto rows = [&](auto KK) {
        using K = decltype(KK);
        typename K::Params p{planes.data(), tb.wrow.data(), tb.wpos.data(), tb.m_lo.data(), tb.m_hi.data(),
                             tb.f2p_row.data(), sh, nullptr, nullptr, nullptr};
        std::vector<C> smem(K::smem_bytes(sh) / sizeof(C) + 1);
        for (int r = 0; r <= sh.M1 / 2; r++) {
            HostExec ex{r, 0, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    };
    if (sh.nt_row == GEN_THREADS) rows(GenRowFusedKernel<T, GEN_THREADS>{});
    else rows(GenRowFusedKernel<T, GEN_THREADS_SMALL>{});
    auto col_inv = [&](auto KK, auto fill) {
        using K = decltype(KK);
        typename K::Params p{};
        static_cast<typename K::PlainParams&>(p) = {planes.data(), &pk, tb.wcol.data(), tb.p2f_col.data(), sh,
                                                    reinterpret_cast<T*>(planes.data())};
        fill(p);
        std::vector<C> smem(K::smem_bytes(sh) / sizeof(C) + 1);
        for (int tile = 0; tile < (sh.M2 + K::CT - 1) / K::CT; tile++) {
            HostExec ex{0, tile, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    };
    auto pick = [&](auto CTC, auto NTC) {
        constexpr int CT = decltype(CTC)::value, NT = decltype(NTC)::value;
        if constexpr (sizeof(T) == 4) {
            pk.key = 0ull; pk.second_bits = 0u; pk.seed_bits = 0u;
            col_inv(GenColInvKernel<T, CT, NT, true, false, true>{}, [&](auto& p) { p.win = full_window(L); p.ru = ru; });
            return;
        }
        col_inv(GenColInvKernel<T, CT, NT>{}, [](auto&) {});
    };
    if (sh.nt_col == GEN_THREADS) { if (sh.ct == 16) pick(IC<16>{}, IC<GEN_THREADS>{}); else pick(IC<8>{}, IC<GEN_THREADS>{}); }
    else { if (sh.ct == 16) pick(IC<16>{}, IC<GEN_THREADS_SMALL>{}); else pick(IC<8>{}, IC<GEN_THREADS_SMALL>{}); }
    if (sizeof(T) == 4) {
        from_peak(pk, scale, out);
        return 0;
    }
    const T* r = reinterpret_cast<const T*>(planes.data()) + 2 * sh.M;
    const PairWindow win = ru.window(0);
    argmax_window_f64(r, 2 * L, &win, out, scale);
    return 0;
}

}  // namespace

extern "C" {

// the runner-up set of centre p at D in the effective window [lo, hi] at L: lo0 n0 lo1 n1 lo2 n2
void emuru_window(long long p, long long lo, long long hi, long long D, long long L, unsigned* out6) {
    const PairWindow w = runner_up_window(p, lo, hi, D, L);
    out6[0] = w.lo0; out6[1] = w.n0; out6[2] = w.lo1; out6[3] = w.n1; out6[4] = w.lo2; out6[5] = w.n2;
}

// kind: 0 static four-step (L one of the six), 1 single-CTA, 2 runtime-radix fp32, 3 runtime-radix fp64.
// [lo, hi]: the effective lag window; first_raw: the batch record's raw_index (the centre); D >= 1.
int emuru_run(int kind, const double* source, const double* sample, long long L, long long lo, long long hi,
              long long first_raw, long long D, Rec* out) {
    audiosync_cuda_result first;
    memset(&first, 0, sizeof(first));
    first.raw_index = first_raw;
    const RunnerUp ru{&first, lo, hi, D, L};
    PairPeak pk;
    memset(&pk, 0, sizeof(pk));
    if (kind == 0) {
        bool found = false;
        for_each_static_plan([&](auto P) {
            if (decltype(P)::L == L) { static_plan<decltype(P)>(source, sample, ru, &pk); found = true; }
        });
        if (!found) return -1;
    } else if (kind == 1) {
        if (small_plan(source, sample, L, ru, &pk) != 0) return -1;
    } else if (kind == 2) {
        return generic_plan<float>(source, sample, L, ru, out);
    } else if (kind == 3) {
        return generic_plan<double>(source, sample, L, ru, out);
    } else {
        return -1;
    }
    from_peak(pk, 1.0, out);
    return 0;
}

}
