// tests/emu/emu_shared.cu -- CPU emulation of the shared-source kernels (TEST ONLY).
//
// Runs one static plan two ways on a batch of pairs that share one source:
//   replicated  K_A on both signals of every pair, RowFusedKernel (ROWS_PAIR), K_C;
//   reuse       K_A on the source alone as one pair, the source-spectrum kernel (ROWS_SRC_SPECTRUM),
//               then per wave the sample-only K_A, the shared-source K_B (ROWS_SHARED_SRC), K_C;
// under NONE or PHAT weighting, on f64 inputs, and returns every pair's product plane (K_B's output,
// what K_C reads) and its packed peak record.  The reuse run fills plane 0 with NaN before its K_A, so
// that a K_B which read it would show.  Compiled by tests/test_shared_source_emu.py; never linked
// into the product.  The executor is emu_phat.cu's.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <vector>

#include "fft_plan.h"

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

namespace {

template <class P>
struct Tables {
    using Col = typename P::Col;
    using Row = typename P::Row;
    std::vector<cplx> col_tw = build_pass_tables(radix_vector<Col>());
    std::vector<cplx> row_tw = build_pass_tables(radix_vector<Row>());
    std::vector<cplx> col_tc = build_col_tc(P::L, Col::weight(Col::count - 1));
    std::vector<cplx> row_tab = build_row_tab<Row>(P::L, Col::n);
    std::vector<cplx> row_rev = build_row_rev<Row>();
    std::vector<cplx> rev_h = build_row_rev_half<Row>();
    std::vector<cplx> m_lo, m_hi, n_lo, n_hi;
    Tables() {
        build_two_level(P::L, P::L - 1, m_lo, m_hi);
        build_two_level(2 * P::L, Col::n / 2, n_lo, n_hi);    // as build_static_plan for PHAT
    }
};

// K_A over `pairs` pairs: SMP_ONLY, or `sigs` signals (1: the source alone)
template <class P, bool SMP_ONLY>
void col_fwd(const Tables<P>& t, const double* src, const double* smp, long long sp, long long mp, cplx* planes,
             PairPeak* peaks, int pairs, int sigs) {
    using K = ColFwdKernel<typename P::Col, P::Row::n, P::NT_COL, double, false, SMP_ONLY>;
    typename K::Params p{src, smp, planes, peaks, t.col_tw.data(), t.col_tc.data(), t.m_lo.data(), t.m_hi.data(), P::L, sp, mp, 1, 1};
    std::vector<cplx> smem(K::SMEM / sizeof(cplx));
    for (int pair = 0; pair < pairs; pair++)
        for (int sig = 0; sig < (SMP_ONLY ? 1 : sigs); sig++)
            for (int tile = 0; tile < P::Row::n / COL_T; tile++) {
                HostExec ex{tile, sig, pair, K::THREADS};
                K::run(ex, p, smem.data());
            }
}

template <class P, bool PHAT, int MODE>
void rows(const Tables<P>& t, cplx* planes, const cplx* spec, int pairs) {
    using K = RowFusedKernel<typename P::Row, P::Col::n, P::NT_ROW, PHAT, MODE>;
    const typename K::PairParams base{planes, t.row_tw.data(), PHAT ? t.rev_h.data() : t.row_rev.data(),
                                      PHAT ? t.n_lo.data() : t.m_lo.data(), PHAT ? t.n_hi.data() : t.m_hi.data(), P::L,
                                      t.row_tab.data()};
    typename K::Params p;
    if constexpr (MODE == ROWS_SHARED_SRC) p = {base, spec};
    else p = base;
    (void)spec;
    std::vector<cplx> smem(K::SMEM / sizeof(cplx));
    for (int pair = 0; pair < pairs; pair++)
        for (int r = 0; r <= P::Col::n / 2; r++) {
            HostExec ex{r, 0, pair, K::THREADS};
            K::run(ex, p, smem.data());
        }
}

template <class P>
void col_inv(const Tables<P>& t, const cplx* planes, PairPeak* peaks, int pairs) {
    using K = ColInvKernel<typename P::Col, P::Row::n, P::NT_COL>;
    std::vector<cplx> smem(K::SMEM / sizeof(cplx));
    for (int pair = 0; pair < pairs; pair++) {
        typename K::Params p{planes, peaks, t.col_tw.data(), P::L};
        for (int tile = 0; tile < P::Row::n / COL_T; tile++) {
            HostExec ex{pair, tile, 0, K::THREADS};
            K::run(ex, p, smem.data());
        }
    }
}

template <class P, bool PHAT>
void run(const double* source, const double* samples, int pairs, int shared, cplx* product, PairPeak* peaks) {
    const long long M = P::L;
    Tables<P> t;
    std::vector<cplx> planes(2 * M * pairs);
    for (int i = 0; i < pairs; i++) { peaks[i] = cleared_peak(); peaks[i].key = 12345ull; peaks[i].second_bits = 777u; }
    if (!shared) {
        std::vector<double> sources(2 * M * pairs);                  // the source replicated per pair
        for (int i = 0; i < pairs; i++) memcpy(sources.data() + 2 * M * i, source, sizeof(double) * 2 * M);
        col_fwd<P, false>(t, sources.data(), samples, 2 * M, M, planes.data(), peaks, pairs, 2);
        rows<P, PHAT, ROWS_PAIR>(t, planes.data(), nullptr, pairs);
    } else {
        std::vector<cplx> spec(M);
        PairPeak scratch;
        col_fwd<P, false>(t, source, source, 2 * M, 2 * M, spec.data(), &scratch, 1, 1);
        rows<P, false, ROWS_SRC_SPECTRUM>(t, spec.data(), nullptr, 1);
        const float nan = std::numeric_limits<float>::quiet_NaN();
        for (auto& z : planes) z = cmake(nan, nan);                   // plane 0 must never be read
        col_fwd<P, true>(t, nullptr, samples, 0, M, planes.data(), peaks, pairs, 1);
        rows<P, PHAT, ROWS_SHARED_SRC>(t, planes.data(), spec.data(), pairs);
    }
    for (int i = 0; i < pairs; i++) memcpy(product + M * i, planes.data() + 2 * M * i, sizeof(cplx) * M);
    col_inv<P>(t, planes.data(), peaks, pairs);
}

}  // namespace

extern "C" {

// source [2L], samples [pairs][L] -> product [pairs][L] complex fp32 (interleaved floats), and per pair
// the packed peak key, second_bits and seed_bits.  Returns -1 when L is not a static length.
int emushared_run(long long L, int phat, int shared, const double* source, const double* samples, int pairs,
                  float* product, unsigned long long* key, unsigned* second_bits, unsigned* seed_bits) {
    int rc = -1;
    std::vector<PairPeak> pk(pairs);
    for_each_static_plan([&](auto P) {
        using PT = decltype(P);
        if (PT::L != L) return;
        if (phat) run<PT, true>(source, samples, pairs, shared, reinterpret_cast<cplx*>(product), pk.data());
        else run<PT, false>(source, samples, pairs, shared, reinterpret_cast<cplx*>(product), pk.data());
        rc = 0;
    });
    for (int i = 0; rc == 0 && i < pairs; i++) {
        key[i] = pk[i].key; second_bits[i] = pk[i].second_bits; seed_bits[i] = pk[i].seed_bits;
    }
    return rc;
}

}
