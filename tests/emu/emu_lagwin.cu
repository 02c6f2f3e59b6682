// tests/emu/emu_lagwin.cu -- CPU emulation of the lag-windowed kernel bodies (TEST ONLY).
//
// Runs the windowed twins of the static K_C (ColInvKernel<..., WIN = true>), of the runtime-radix fp32
// inverse column kernel (GenColInvKernel<float, CT, NT, true>) and of the single-CTA kernel
// (SmallXcorrKernel<double, false, true>), with the unwindowed forward and row kernels before them, on
// f64 inputs (the F64 call); `windowed` = 0 runs the unwindowed kernels instead.  fp64 runtime-radix
// plans write r and resolve it with argmax_f64_window_kernel, whose body needs warp shuffles: it is
// restated here (the same candidates and order rule).  Every runner returns the resolved index / peak /
// second peak at the reference's scale (x N) and the packed peak record of the fp32-argmax paths.
// emulw_perturb changes one entry of a table the static plans build on the host before their kernels
// run (tests/test_xcorr_error_emu.py: a corrupted table must fail the per-lag error bound).
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

// what: 0 none, 1 col_tw[i] *= (1 + eps), 2 row_tab[i] conjugated, 3 row_tw[i] and row_tw[j] swapped
struct Perturb { int what; long long i, j; double eps; };
Perturb g_perturb{0, 0, 0, 0.0};

void apply_perturb(std::vector<cplx>& col_tw, std::vector<cplx>& row_tw, std::vector<cplx>& row_tab) {
    const Perturb& q = g_perturb;
    if (q.what == 1) col_tw.at(q.i) = cmake((float)(col_tw.at(q.i).x * (1.0 + q.eps)), (float)(col_tw.at(q.i).y * (1.0 + q.eps)));
    else if (q.what == 2) row_tab.at(q.i).y = -row_tab.at(q.i).y;
    else if (q.what == 3) std::swap(row_tw.at(q.i), row_tw.at(q.j));
}

void from_peak(const PairPeak& pk, double scale, Rec* r) {
    r->raw_index = (long long)argmax_key_index(pk.key);
    r->peak = (double)argmax_key_value(pk.key) * scale;
    r->second = (double)pair_second(pk) * scale;
    r->key = pk.key; r->second_bits = pk.second_bits; r->seed_bits = pk.seed_bits;
}

template <class P>
void static_plan(const double* source, const double* sample, const RawWindow& win, bool windowed, PairPeak* peak) {
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
    apply_perturb(col_tw, row_tw, row_tab);
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
        typename K::Params p{planes.data(), peak, col_tw.data(), M};
        fill(p);
        std::vector<cplx> smem(K::SMEM / sizeof(cplx));
        for (int tile = 0; tile < M2 / COL_T; tile++) {
            HostExec ex{0, tile, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    };
    if (windowed) col_inv(ColInvKernel<Col, Row::n, P::NT_COL, true, true>{}, [&](auto& p) { p.win = win; });
    else col_inv(ColInvKernel<Col, Row::n, P::NT_COL>{}, [](auto&) {});
}

int small_plan(const double* source, const double* sample, long long L, const RawWindow& win, bool windowed, PairPeak* peak) {
    SmallPlan pl;
    if (!make_small_plan(L, &pl)) return -1;
    std::vector<cplx> wm = build_full_table(L, L), wn = build_full_table(2 * L, L);
    peak->key = 12345ull; peak->second_bits = 777u; peak->seed_bits = 777u;
    auto go = [&](auto KK, auto fill) {
        using K = decltype(KK);
        typename K::Params p{source, sample, peak, wm.data(), wn.data(), pl, 2 * L, L, 1, 1};
        fill(p);
        std::vector<cplx> smem(K::smem_bytes((int)L) / sizeof(cplx));
        HostExec ex{0, 0, 0, K::THREADS};
        K::run(ex, p, smem.data());
    };
    if (windowed) go(SmallXcorrKernel<double, false, true>{}, [&](auto& p) { p.win = win; });
    else go(SmallXcorrKernel<double>{}, [](auto&) {});
    return 0;
}

// argmax_f64_window_kernel's rule: allowed indices in ascending order, r[0] the signed seed when
// allowed, strict >, a NaN never wins (but beats the empty start on index order), second = largest
// non-NaN |r| over the other allowed indices
template <typename T>
void argmax_window_f64(const T* r, long long N, const RawWindow* win, Rec* out, double scale) {
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
int generic_plan(const double* source, const double* sample, long long L, const RawWindow& win, bool windowed, Rec* out) {
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
        typename K::Params p{planes.data(), &pk, tb.wcol.data(), tb.p2f_col.data(), sh, reinterpret_cast<T*>(planes.data())};
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
            if (windowed) { col_inv(GenColInvKernel<T, CT, NT, true>{}, [&](auto& p) { p.win = win; }); return; }
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
    argmax_window_f64(r, 2 * L, windowed ? &win : nullptr, out, scale);
    return 0;
}

}  // namespace

extern "C" {

// the table entry the static plans change from now on (what = 0: none); not thread-safe against runs
void emulw_perturb(int what, long long i, long long j, double eps) { g_perturb = Perturb{what, i, j, eps}; }

// the library's description of the runtime-radix plan (kind 2 fp32, 3 fp64) at L: its length, -1 none
int emulw_describe(int kind, long long L, char* buf, int len) {
    GenShape sh;
    if ((kind != 2 && kind != 3) || !gen_make_shape(L, kind == 3, &sh)) return -1;
    const std::string d = gen_describe(sh, kind == 3);
    if ((int)d.size() + 1 > len) return -1;
    memcpy(buf, d.c_str(), d.size() + 1);
    return (int)d.size();
}

// sizes of the static plan's host tables at L: col_tw, row_tw, row_tab (-1: no static plan)
long long emulw_table_sizes(long long L, long long* out3) {
    long long rc = -1;
    for_each_static_plan([&](auto P) {
        using PP = decltype(P);
        if (PP::L != L) return;
        out3[0] = (long long)build_pass_tables(radix_vector<typename PP::Col>()).size();
        out3[1] = (long long)build_pass_tables(radix_vector<typename PP::Row>()).size();
        out3[2] = (long long)build_row_tab<typename PP::Row>(PP::L, PP::Col::n).size();
        rc = 0;
    });
    return rc;
}

// raw ranges of the lag window [lo, hi] at L: -1 empty, 0 all of [-L, L-1], 1 restrictive
int emulw_window(long long lo, long long hi, long long L, unsigned* out4) {
    RawWindow w{0u, 0u, 0u, 0u};
    const int rc = raw_window_of(lo, hi, L, &w);
    out4[0] = w.lo0; out4[1] = w.n0; out4[2] = w.lo1; out4[3] = w.n1;
    return rc;
}

// kind: 0 static four-step (L one of the six), 1 single-CTA, 2 runtime-radix fp32, 3 runtime-radix fp64
int emulw_run(int kind, const double* source, const double* sample, long long L, long long lo, long long hi,
              int windowed, Rec* out) {
    RawWindow win{0u, 0u, 0u, 0u};
    if (windowed && raw_window_of(lo, hi, L, &win) != 1) return -2;
    PairPeak pk;
    memset(&pk, 0, sizeof(pk));
    if (kind == 0) {
        bool found = false;
        for_each_static_plan([&](auto P) {
            if (decltype(P)::L == L) { static_plan<decltype(P)>(source, sample, win, windowed != 0, &pk); found = true; }
        });
        if (!found) return -1;
    } else if (kind == 1) {
        if (small_plan(source, sample, L, win, windowed != 0, &pk) != 0) return -1;
    } else if (kind == 2) {
        return generic_plan<float>(source, sample, L, win, windowed != 0, out);
    } else if (kind == 3) {
        return generic_plan<double>(source, sample, L, win, windowed != 0, out);
    } else {
        return -1;
    }
    from_peak(pk, 1.0, out);
    return 0;
}

}
