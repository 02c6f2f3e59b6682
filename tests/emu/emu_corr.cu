// tests/emu/emu_corr.cu -- CPU emulation of the correlation-exporting kernel bodies (TEST ONLY).
//
// Runs one pair through the static four-step plan at 144,000, the single-CTA kernel or the runtime-radix
// fp32 kernels (rows on the static row kernel where the plan's M2 has one, as the product does), on f64
// inputs, unweighted or PHAT, and ends it either with the non-exporting inverse kernel the library runs
// without export (unwindowed, or the windowed twin) or with the exporting twin (ColInvKernel<..., true,
// true, true>, GenColInvKernel<float, CT, NT, true, true>, SmallXcorrKernel<double, PHAT, true, false,
// true>), which gets the lag window or, when none is set, all of [0, 2L).  Returns the packed peak record
// and the exported row.  Compiled by tests/golden/emu_build.py for the tests; never linked into the product.
#include <cmath>
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
    double peak, second;      // as pearson_block forms them: the kernel's value times `scale`
    unsigned long long key;
    unsigned second_bits, seed_bits;
    double scale;             // the plan's peak_scale
};

namespace {

// How the inverse pass ends: the library's kernel without export, or the exporting twin.
struct Ending {
    bool out;                 // exporting twin
    const RawWindow* win;     // lag window (nullptr: none)
    CorrOut corr;             // out: the row
};

template <class K, class Fill>
void run_col_inv_static(const Fill& fill, int tiles) {
    typename K::Params p{};
    fill(p);
    std::vector<cplx> smem(K::SMEM / sizeof(cplx));
    for (int tile = 0; tile < tiles; tile++) {
        HostExec ex{0, tile, 0, K::THREADS};
        K::run(ex, p, smem.data());
    }
}

void static_144k(const double* source, const double* sample, bool phat, const Ending& e, PairPeak* peak) {
    using P = Plan144k;
    using Col = P::Col;
    using Row = P::Row;
    constexpr int M1 = Col::n, M2 = Row::n;
    const long long M = P::L;
    std::vector<cplx> planes(2 * M);
    std::vector<cplx> col_tw = build_pass_tables(radix_vector<Col>());
    std::vector<cplx> row_tw = build_pass_tables(radix_vector<Row>());
    std::vector<cplx> col_tc = build_col_tc(M, Col::weight(Col::count - 1));
    std::vector<cplx> row_tab = build_row_tab<Row>(M, M1);
    std::vector<cplx> row_rev = build_row_rev<Row>(), rev_h = build_row_rev_half<Row>();
    std::vector<cplx> m_lo, m_hi, n_lo, n_hi;
    build_two_level(M, M - 1, m_lo, m_hi);
    build_two_level(2 * M, M1 / 2, n_lo, n_hi);
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
    auto rows = [&](auto KK, const cplx* rev, const cplx* lo, const cplx* hi) {
        using K = decltype(KK);
        typename K::Params p{planes.data(), row_tw.data(), rev, lo, hi, M, row_tab.data()};
        std::vector<cplx> smem(K::SMEM / sizeof(cplx));
        for (int r = 0; r <= M1 / 2; r++) {
            HostExec ex{r, 0, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    };
    if (phat) rows(RowFusedKernel<Row, Col::n, P::NT_ROW, true>{}, rev_h.data(), n_lo.data(), n_hi.data());
    else rows(RowFusedKernel<Row, Col::n, P::NT_ROW>{}, row_rev.data(), m_lo.data(), m_hi.data());
    auto base = [&](auto& p) { p.planes = planes.data(); p.peaks = peak; p.tw = col_tw.data(); p.L = M; };
    if (e.out)
        run_col_inv_static<ColInvKernel<Col, Row::n, P::NT_COL, true, true, true>>([&](auto& p) {
            base(p); p.win = e.win ? *e.win : full_window(M); p.corr = e.corr;
        }, M2 / COL_T);
    else if (e.win)
        run_col_inv_static<ColInvKernel<Col, Row::n, P::NT_COL, true, true>>([&](auto& p) { base(p); p.win = *e.win; }, M2 / COL_T);
    else
        run_col_inv_static<ColInvKernel<Col, Row::n, P::NT_COL>>([&](auto& p) { base(p); }, M2 / COL_T);
}

int small_plan(const double* source, const double* sample, long long L, bool phat, const Ending& e, PairPeak* peak) {
    SmallPlan pl;
    if (!make_small_plan(L, &pl)) return -1;
    std::vector<cplx> wm = build_full_table(L, L), wn = build_full_table(2 * L, L);
    peak->key = 12345ull; peak->second_bits = 777u; peak->seed_bits = 777u;
    auto go = [&](auto KK, auto fill) {
        using K = decltype(KK);
        typename K::Params p{};
        p.sources = source; p.samples = sample; p.peaks = peak; p.wm = wm.data(); p.wn = wn.data(); p.plan = pl;
        p.src_pitch = 2 * L; p.smp_pitch = L; p.vec_src = 1; p.vec_smp = 1;
        fill(p);
        std::vector<cplx> smem(K::smem_bytes((int)L) / sizeof(cplx));
        HostExec ex{0, 0, 0, K::THREADS};
        K::run(ex, p, smem.data());
    };
    auto pick = [&](auto PHAT) {
        constexpr bool PH = decltype(PHAT)::value;
        if (e.out) go(SmallXcorrKernel<double, PH, true, false, true>{}, [&](auto& p) { p.win = e.win ? *e.win : full_window(L); p.corr = e.corr; });
        else if (e.win) go(SmallXcorrKernel<double, PH, true>{}, [&](auto& p) { p.win = *e.win; });
        else go(SmallXcorrKernel<double, PH>{}, [](auto&) {});
    };
    if (phat) pick(std::true_type{});
    else pick(std::false_type{});
    return 0;
}

// the rows of a runtime-radix fp32 plan on a static row kernel (static_rows.cu)
template <class RL, int NT>
void static_rows(std::vector<cplx>& planes, const GenShape& sh, bool phat) {
    std::vector<cplx> row_tw = build_pass_tables(radix_vector<RL>());
    std::vector<cplx> row_tab = build_row_tab<RL>(sh.M, sh.M1);
    std::vector<cplx> rev = build_row_rev<RL>(), rev_h = build_row_rev_half<RL>(), m_lo, m_hi, n_lo, n_hi;
    build_two_level(sh.M, sh.M - 1, m_lo, m_hi);
    build_two_level(2 * sh.M, sh.M1 / 2, n_lo, n_hi);
    auto go = [&](auto KK, const cplx* r, const cplx* lo, const cplx* hi) {
        using K = decltype(KK);
        typename K::Params p{planes.data(), row_tw.data(), r, lo, hi, sh.M, row_tab.data(), sh.M1};
        std::vector<cplx> smem(K::SMEM / sizeof(cplx));
        for (int rr = 0; rr <= sh.M1 / 2; rr++) {
            HostExec ex{rr, 0, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    };
    if (phat) go(RowFusedKernel<RL, 0, NT, true>{}, rev_h.data(), n_lo.data(), n_hi.data());
    else go(RowFusedKernel<RL, 0, NT>{}, rev.data(), m_lo.data(), m_hi.data());
}

// runtime-radix fp32 kernels; *scale: the plan's peak_scale, *static_rows_used as the product chooses
int generic_f32(const double* source, const double* sample, long long L, bool phat, const Ending& e, PairPeak* pk,
                double* scale, int* static_rows_used) {
    typedef cplx C;
    GenShape sh;
    if (!gen_make_shape(L, false, &sh)) return -1;
    if (phat && sh.M != L) return -1;                      // PHAT is not served on embedded lengths
    const GenTables<C> tb = gen_build_tables<C>(sh);
    std::vector<C> planes(2 * sh.M);
    pk->key = 12345ull; pk->second_bits = 777u; pk->seed_bits = 777u;
    auto col_fwd = [&](auto KK) {
        using K = decltype(KK);
        typename K::Params p{source, sample, planes.data(), pk, tb.wcol.data(), tb.m_lo.data(), tb.m_hi.data(),
                             tb.p2f_col.data(), sh, 2 * L, L, 1, 1};
        std::vector<C> smem(K::smem_bytes(sh) / sizeof(C) + 1);
        for (int sig = 0; sig < 2; sig++)
            for (int tile = 0; tile < (sh.M2 + K::CT - 1) / K::CT; tile++) {
                HostExec ex{tile, sig, 0, K::THREADS};
                K::run(ex, p, smem.data());
            }
    };
    if (sh.nt_col == GEN_THREADS) { if (sh.ct == 16) col_fwd(GenColFwdKernel<float, double, 16, GEN_THREADS>{}); else col_fwd(GenColFwdKernel<float, double, 8, GEN_THREADS>{}); }
    else { if (sh.ct == 16) col_fwd(GenColFwdKernel<float, double, 16, GEN_THREADS_SMALL>{}); else col_fwd(GenColFwdKernel<float, double, 8, GEN_THREADS_SMALL>{}); }
    *scale = gen_peak_scale(sh);
    *static_rows_used = sh.static_rows != 0;
    if (sh.static_rows) {
        *scale *= 2.0;                                      // the static row kernel applies the merge's 1/2
        switch (sh.M2) {
            case 480: static_rows<Plan144k::Row, Plan144k::NT_ROW>(planes, sh, phat); break;
            case 960: static_rows<Plan288k::Row, Plan288k::NT_ROW>(planes, sh, phat); break;
            case 1200: static_rows<Plan720k::Row, Plan720k::NT_ROW>(planes, sh, phat); break;
            default: static_rows<Plan1440k::Row, Plan1440k::NT_ROW>(planes, sh, phat); break;
        }
    } else {
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
        if (phat) { if (sh.nt_row == GEN_THREADS) rows(GenRowFusedKernel<float, GEN_THREADS, true>{}); else rows(GenRowFusedKernel<float, GEN_THREADS_SMALL, true>{}); }
        else { if (sh.nt_row == GEN_THREADS) rows(GenRowFusedKernel<float, GEN_THREADS>{}); else rows(GenRowFusedKernel<float, GEN_THREADS_SMALL>{}); }
    }
    CorrOut corr = e.corr;
    corr.scale = *scale;
    auto col_inv = [&](auto KK, auto fill) {
        using K = decltype(KK);
        typename K::Params p{};
        p.planes = planes.data(); p.peaks = pk; p.wcol = tb.wcol.data(); p.p2f_col = tb.p2f_col.data(); p.sh = sh;
        p.r_out = reinterpret_cast<float*>(planes.data());
        fill(p);
        std::vector<C> smem(K::smem_bytes(sh) / sizeof(C) + 1);
        for (int tile = 0; tile < (sh.M2 + K::CT - 1) / K::CT; tile++) {
            HostExec ex{0, tile, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    };
    auto pick = [&](auto CTC, auto NTC) {
        constexpr int CT = decltype(CTC)::value, NT = decltype(NTC)::value;
        if (e.out) col_inv(GenColInvKernel<float, CT, NT, true, true>{}, [&](auto& p) { p.win = e.win ? *e.win : full_window(L); p.corr = corr; });
        else if (e.win) col_inv(GenColInvKernel<float, CT, NT, true>{}, [&](auto& p) { p.win = *e.win; });
        else col_inv(GenColInvKernel<float, CT, NT>{}, [](auto&) {});
    };
    if (sh.nt_col == GEN_THREADS) { if (sh.ct == 16) pick(IC<16>{}, IC<GEN_THREADS>{}); else pick(IC<8>{}, IC<GEN_THREADS>{}); }
    else { if (sh.ct == 16) pick(IC<16>{}, IC<GEN_THREADS_SMALL>{}); else pick(IC<8>{}, IC<GEN_THREADS_SMALL>{}); }
    return 0;
}

}  // namespace

extern "C" {

// kind: 0 static four-step at 144,000, 1 single-CTA, 2 runtime-radix fp32.  out: 0 the library's kernel
// without export, 1 the exporting twin, writing lags [clo, chi] into corr (hi - lo + 1 doubles).
// windowed: the lag window [wlo, whi].  *info: runtime-radix plans: 1 when the rows ran on a static row
// kernel, 2 when the plan is embedded (M > L).  Returns 0, -1 (no such plan), -2 (empty window).
int emuc_run(int kind, int phat, const double* source, const double* sample, long long L, int out, int windowed,
             long long wlo, long long whi, long long clo, long long chi, double* corr, Rec* rec, int* info) {
    RawWindow win{0u, 0u, 0u, 0u};
    if (windowed && raw_window_of(wlo, whi, L, &win) != 1) return -2;
    Ending e{out != 0, windowed ? &win : nullptr, corr_out_of(clo, chi, L, corr, 1.0)};
    PairPeak pk;
    memset(&pk, 0, sizeof(pk));
    double scale = 1.0;
    *info = 0;
    if (kind == 0) {
        if (L != Plan144k::L) return -1;
        static_144k(source, sample, phat != 0, e, &pk);
    } else if (kind == 1) {
        if (small_plan(source, sample, L, phat != 0, e, &pk) != 0) return -1;
    } else if (kind == 2) {
        int sr = 0;
        if (generic_f32(source, sample, L, phat != 0, e, &pk, &scale, &sr) != 0) return -1;
        GenShape sh;
        gen_make_shape(L, false, &sh);
        *info = sr | (sh.M != L ? 2 : 0);
    } else {
        return -1;
    }
    rec->raw_index = (long long)argmax_key_index(pk.key);
    rec->peak = (double)argmax_key_value(pk.key) * scale;
    rec->second = (double)pair_second(pk) * scale;
    rec->key = pk.key; rec->second_bits = pk.second_bits; rec->seed_bits = pk.seed_bits;
    rec->scale = scale;
    return 0;
}

}
