// tests/emu/emu.cu -- CPU emulator of the transform kernels (TEST ONLY).
//
// Compiles the *same* kernel bodies the GPU runs (fft_kernels.cuh /
// fft_small.cuh are written against an executor) with a HostExec that runs
// every phase for all thread ids in turn.  It lets the CPU suite check the
// index maps, digit reversal, twiddle tables and the split/multiply/merge
// against the oracle without a GPU.  It is never linked into the product.
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
        // the CTA-level merge of (peak key, second peak) pairs, then the grid-level rule of
        // DeviceExec::phase_argmax (sequentially: max / max-of-min)
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

// TMA: K_A stages its tiles (fp32 only), otherwise its first pass loads through registers
template <class P, typename InT, bool TMA>
static int run_static(const InT* source, const InT* sample, PairPeak* peak, cplx* planes_out) {
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
        // TMA: host emulation copies the same boxes and leaves the last tile row unstaged
        using K = ColFwdKernel<Col, Row::n, P::NT_COL, InT, TMA>;
        typename K::Params p{source, sample, planes.data(), peak, col_tw.data(), col_tc.data(), m_lo.data(), m_hi.data(), M};
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
    if (planes_out) memcpy(planes_out, planes.data(), sizeof(cplx) * M);
    {
        using K = ColInvKernel<Col, Row::n, P::NT_COL>;
        typename K::Params p{planes.data(), peak, col_tw.data(), M};
        std::vector<cplx> smem(K::SMEM / sizeof(cplx));
        for (int tile = 0; tile < M2 / COL_T; tile++) {
            HostExec ex{0, tile, 0, K::THREADS};      // K_C grid = (pairs, tiles)
            K::run(ex, p, smem.data());
        }
    }
    return 0;
}

template <typename InT>
static int run_small(const InT* source, const InT* sample, long long L, PairPeak* peak) {
    SmallPlan pl;
    if (!make_small_plan(L, &pl)) return -1;
    std::vector<cplx> wm = build_full_table(L, L), wn = build_full_table(2 * L, L);
    using K = SmallXcorrKernel<InT>;
    typename K::Params p{source, sample, peak, wm.data(), wn.data(), pl};
    std::vector<cplx> smem(K::smem_bytes((int)L) / sizeof(cplx));
    peak->key = 12345ull; peak->second_bits = 777u; peak->seed_bits = 777u;   // garbage: the kernel must clear them
    HostExec ex{0, 0, 0, K::THREADS};
    K::run(ex, p, smem.data());
    return 0;
}

// ---- runtime-radix kernels (fft_generic.cuh): T = arithmetic type, InT = input type
template <typename T, typename InT>
static int run_generic(const InT* source, const InT* sample, long long L, long long* raw_index, double* peak_value,
                       double* second_value, char* desc, size_t desc_len) {
    typedef typename GenTraits<T>::C C;
    GenShape sh;
    if (!gen_make_shape(L, sizeof(T) == 8, &sh)) return -1;
    if (desc) snprintf(desc, desc_len, "%s", gen_describe(sh, sizeof(T) == 8).c_str());
    const GenTables<C> tb = gen_build_tables<C>(sh);
    std::vector<C> planes(2 * sh.M);
    PairPeak pk;
    memset(&pk, 0, sizeof(pk));
    pk.key = 12345ull; pk.second_bits = 777u; pk.seed_bits = 777u;   // garbage: G_A must clear them
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
        *raw_index = (long long)argmax_key_index(pk.key);
        *peak_value = (double)argmax_key_value(pk.key) * scale;
        *second_value = (double)pair_second(pk) * scale;
    } else {
        // fp64: r[0 .. 2L) sits in plane 1; resolve like argmax_f64_kernel (reference :52-67)
        const T* r = reinterpret_cast<const T*>(planes.data()) + 2 * sh.M;
        long long best = 0;
        double bv = (double)r[0];
        for (long long i = 1; i < 2 * L; i++)
            if (fabs((double)r[i]) > bv) { bv = fabs((double)r[i]); best = i; }
        double second = 0.0;
        for (long long i = 0; i < 2 * L; i++)
            if (i != best && fabs((double)r[i]) > second) second = fabs((double)r[i]);
        *raw_index = best;
        *peak_value = (double)r[best] * scale;
        *second_value = second * scale;
    }
    return 0;
}

static double g_last_second = 0.0;   // second peak of the last emu_any call

// ka_registers: static plans run K_A's register load even where the product stages fp32 tiles
template <typename InT>
static int emu_any(const InT* source, const InT* sample, long long L, int forced,
                   long long* raw_index, double* peak_value, int* path, bool ka_registers = false) {
    PairPeak pk;
    memset(&pk, 0, sizeof(pk));
    PathKind kind = choose_path(L, forced);
    *path = (int)kind;
    int rc = -1;
    if (kind == PATH_STATIC_FFT) {
        for_each_static_plan([&](auto P) {
            using PT = decltype(P);
            if (PT::L != L) return;
            if constexpr (sizeof(InT) == 4)
                rc = ka_registers ? run_static<PT, InT, false>(source, sample, &pk, nullptr)
                                  : run_static<PT, InT, true>(source, sample, &pk, nullptr);
            else
                rc = run_static<PT, InT, false>(source, sample, &pk, nullptr);
        });
    } else if (kind == PATH_SMALL_FFT) {
        rc = run_small<InT>(source, sample, L, &pk);
    } else if (kind == PATH_GENERIC_FFT) {
        double second = 0.0;
        rc = run_generic<float, InT>(source, sample, L, raw_index, peak_value, &second, nullptr, 0);
        g_last_second = second;
        return rc;
    } else {
        return -2;   // direct path has no transform to emulate
    }
    if (rc != 0) return rc;
    *raw_index = (long long)argmax_key_index(pk.key);
    *peak_value = (double)argmax_key_value(pk.key);
    g_last_second = (double)pair_second(pk);
    return 0;
}

extern "C" {

double emu_last_second(void) { return g_last_second; }

// runtime-radix four-step kernels; precise != 0: fp64 arithmetic.  desc receives the plan text.
int emu_generic_f32(const float* source, const float* sample, long long L, int precise, long long* raw_index,
                    double* peak_value, double* second_value, char* desc, size_t desc_len) {
    return precise ? run_generic<double, float>(source, sample, L, raw_index, peak_value, second_value, desc, desc_len)
                   : run_generic<float, float>(source, sample, L, raw_index, peak_value, second_value, desc, desc_len);
}
int emu_generic_f64(const double* source, const double* sample, long long L, int precise, long long* raw_index,
                    double* peak_value, double* second_value, char* desc, size_t desc_len) {
    return precise ? run_generic<double, double>(source, sample, L, raw_index, peak_value, second_value, desc, desc_len)
                   : run_generic<float, double>(source, sample, L, raw_index, peak_value, second_value, desc, desc_len);
}
// multiply-shift division of the runtime-radix kernels: first (n, d) with fast_div(n, d) != n / d, or 0
long long emu_fastdiv_first_error(unsigned d_max, unsigned n_max) {
    for (unsigned d = 1; d <= d_max; d++) {
        const FastDiv f = make_fastdiv(d);
        for (unsigned n = 0; n <= n_max; n = n < 70000 ? n + 1 : n + 997)
            if (fast_div(n, f) != n / d) return ((long long)d << 32) | n;
        for (unsigned n : {0x7fffffffu, 0x7ffffffeu, 0x40000000u})
            if (fast_div(n, f) != n / d) return ((long long)d << 32) | n;
    }
    return 0;
}
int emu_generic_describe(long long L, int precise, char* desc, size_t desc_len) {
    GenShape sh;
    if (!gen_make_shape(L, precise != 0, &sh)) return -1;
    snprintf(desc, desc_len, "%s", gen_describe(sh, precise != 0).c_str());
    return 0;
}

int emu_xcorr_f32(const float* source, const float* sample, long long L, int forced,
                  long long* raw_index, double* peak_value, int* path) {
    return emu_any<float>(source, sample, L, forced, raw_index, peak_value, path);
}

// the same with K_A's fp32 first pass through registers (the product's path for fp32 inputs
// that are not 16-byte aligned)
int emu_xcorr_f32_ka_registers(const float* source, const float* sample, long long L, int forced,
                               long long* raw_index, double* peak_value, int* path) {
    return emu_any<float>(source, sample, L, forced, raw_index, peak_value, path, true);
}

int emu_xcorr_f64(const double* source, const double* sample, long long L, int forced,
                  long long* raw_index, double* peak_value, int* path) {
    return emu_any<double>(source, sample, L, forced, raw_index, peak_value, path);
}

// fold of reference src/cross_correlation.c:256-271 as compiled into the product
void emu_fold(long long idx, long long L, long long* lag, long long* xoff, long long* yoff,
              long long* n) {
    Window w = fold_index(idx, L);
    *lag = w.lag; *xoff = w.xoff; *yoff = w.yoff; *n = w.n;
}

// argmax key helpers, for semantics tests
unsigned long long emu_key_abs(float v, unsigned idx) { return argmax_key_abs(v, idx); }
unsigned long long emu_key_seed(float v) { return argmax_key_seed(v); }
unsigned emu_key_index(unsigned long long k) { return argmax_key_index(k); }
float emu_key_value(unsigned long long k) { return argmax_key_value(k); }

int emu_path_for(long long L, int forced) { return (int)choose_path(L, forced); }
int emu_path_for_precise(long long L, int forced) { return (int)choose_path(L, forced, true); }

// box geometry of the TMA-staged column tiles (fft_kernels.cuh)
int emu_tile_boxes(int rows) { return tile_boxes(rows); }
int emu_tile_box_rows(int rows) { return tile_box_rows(rows); }
int emu_tile_box_start(int rows, int i) { return tile_box_start(rows, i); }
}
