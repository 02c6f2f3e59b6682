// tests/emu/emu_cross.cu -- CPU emulation of the cross-batch kernels (TEST ONLY).
//
// Runs one static plan two ways on every (source, sample) combination of a batch of sources and a
// batch of samples:
//   pair    per source: K_A on both signals of every pair (the source replicated), RowFusedKernel
//           (ROWS_PAIR), K_C;
//   cross   K_A on each source alone as one pair and the source-spectrum kernel (ROWS_SRC_SPECTRUM), once
//           per source; then per wave of samples the sample-only K_A and the source-spectrum kernel on
//           plane 1 (the samples' forward rows, in place), and per source K_B from both spectra
//           (ROWS_BOTH_SPECTRA) and K_C;
// under NONE or PHAT weighting, on f64 inputs, and returns every combination's product plane (K_B's
// output, what K_C reads) and its packed peak record.  The cross run leaves each wave's peak records as
// the previous source's K_C left them, fills plane 0 with NaN before every K_B and the row kernel's shared
// memory with NaN before every CTA, so that a K_B which did not clear a record, read plane 0 or a point of
// shared memory it did not stage would show.  Compiled by tests/test_cross_batch_emu.py; never linked into
// the product.  The executor is emu_shared.cu's.
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

const float NaN = std::numeric_limits<float>::quiet_NaN();

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
void rows(const Tables<P>& t, cplx* planes, const cplx* spec, PairPeak* peaks, int pairs) {
    using K = RowFusedKernel<typename P::Row, P::Col::n, P::NT_ROW, PHAT, MODE>;
    const typename K::PairParams base{planes, t.row_tw.data(), PHAT ? t.rev_h.data() : t.row_rev.data(),
                                      PHAT ? t.n_lo.data() : t.m_lo.data(), PHAT ? t.n_hi.data() : t.m_hi.data(), P::L,
                                      t.row_tab.data()};
    typename K::Params p;
    if constexpr (MODE == ROWS_BOTH_SPECTRA) p = {{base, spec}, peaks};
    else p = base;
    (void)spec; (void)peaks;
    std::vector<cplx> smem(K::SMEM / sizeof(cplx));
    for (int pair = 0; pair < pairs; pair++)
        for (int r = 0; r <= P::Col::n / 2; r++) {
            for (auto& z : smem) z = cmake(NaN, NaN);
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

// sources [S][2L], samples [n][L] -> product [S][n][L], peaks [S][n]
template <class P, bool PHAT>
void run(const double* sources, int S, const double* samples, int n, int wave, int cross, cplx* product, PairPeak* peaks) {
    const long long M = P::L;
    Tables<P> t;
    if (!cross) {
        std::vector<cplx> planes(2 * M * n);
        std::vector<double> rep(2 * M * n);
        for (int s = 0; s < S; s++) {
            for (int i = 0; i < n; i++) memcpy(rep.data() + 2 * M * i, sources + 2 * M * s, sizeof(double) * 2 * M);
            PairPeak* pk = peaks + (size_t)s * n;
            for (int i = 0; i < n; i++) { pk[i] = cleared_peak(); pk[i].key = 12345ull; pk[i].second_bits = 777u; }
            col_fwd<P, false>(t, rep.data(), samples, 2 * M, M, planes.data(), pk, n, 2);
            rows<P, PHAT, ROWS_PAIR>(t, planes.data(), nullptr, nullptr, n);
            for (int i = 0; i < n; i++) memcpy(product + M * ((size_t)s * n + i), planes.data() + 2 * M * i, sizeof(cplx) * M);
            col_inv<P>(t, planes.data(), pk, n);
        }
        return;
    }
    std::vector<cplx> spec(M * S);
    PairPeak scratch;
    for (int s = 0; s < S; s++) {
        col_fwd<P, false>(t, sources + 2 * M * s, sources + 2 * M * s, 2 * M, 2 * M, spec.data() + M * s, &scratch, 1, 1);
        rows<P, false, ROWS_SRC_SPECTRUM>(t, spec.data() + M * s, nullptr, nullptr, 1);
    }
    std::vector<cplx> planes(2 * M * wave);
    std::vector<PairPeak> wpk(wave);
    for (auto& z : planes) z = cmake(NaN, NaN);
    for (int p0 = 0; p0 < n; p0 += wave) {
        const int pairs = std::min(wave, n - p0);
        for (int i = 0; i < pairs; i++) { wpk[i] = cleared_peak(); wpk[i].key = 12345ull; wpk[i].second_bits = 777u; }
        col_fwd<P, true>(t, nullptr, samples + M * p0, 0, M, planes.data(), wpk.data(), pairs, 1);
        rows<P, false, ROWS_SRC_SPECTRUM>(t, planes.data() + M, nullptr, nullptr, pairs);   // plane 1, pair pitch 2M
        for (int s = 0; s < S; s++) {
            for (int i = 0; i < pairs; i++)                           // plane 0 must never be read
                for (long long k = 0; k < M; k++) planes[2 * M * i + k] = cmake(NaN, NaN);
            rows<P, PHAT, ROWS_BOTH_SPECTRA>(t, planes.data(), spec.data() + M * s, wpk.data(), pairs);
            for (int i = 0; i < pairs; i++)
                memcpy(product + M * ((size_t)s * n + p0 + i), planes.data() + 2 * M * i, sizeof(cplx) * M);
            col_inv<P>(t, planes.data(), wpk.data(), pairs);
            for (int i = 0; i < pairs; i++) peaks[(size_t)s * n + p0 + i] = wpk[i];   // wpk keeps them: K_B must clear
        }
    }
}

}  // namespace

extern "C" {

// sources [S][2L], samples [n][L] -> product [S][n][L] complex fp32 (interleaved floats), and per
// combination the packed peak key, second_bits and seed_bits.  cross: waves of `wave` samples.
// Returns -1 when L is not a static length.
int emucross_run(long long L, int phat, int cross, const double* sources, int S, const double* samples, int n,
                 int wave, float* product, unsigned long long* key, unsigned* second_bits, unsigned* seed_bits) {
    int rc = -1;
    std::vector<PairPeak> pk((size_t)S * n);
    for_each_static_plan([&](auto P) {
        using PT = decltype(P);
        if (PT::L != L) return;
        if (phat) run<PT, true>(sources, S, samples, n, wave, cross, reinterpret_cast<cplx*>(product), pk.data());
        else run<PT, false>(sources, S, samples, n, wave, cross, reinterpret_cast<cplx*>(product), pk.data());
        rc = 0;
    });
    for (size_t i = 0; rc == 0 && i < pk.size(); i++) {
        key[i] = pk[i].key; second_bits[i] = pk[i].second_bits; seed_bits[i] = pk[i].seed_bits;
    }
    return rc;
}

}
