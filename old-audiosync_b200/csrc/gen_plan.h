// gen_plan.h -- host-side planner of the runtime-radix four-step kernels (fft_generic.cuh):
// radix lists with the fewest passes, the M1 x M2 split, the embedding length for sample_len
// values that are not 2/3/5-smooth, and the tables.  Shared by the product library and the CPU
// emulator.  The reference plans per call for any length (src/cross_correlation.c:34, :237);
// this is the counterpart, cached per length by the caller.
#pragma once

#include <algorithm>
#include <cstdint>
#include <map>
#include <vector>

#include "fft_generic.cuh"
#include "fft_plan.h"

namespace asc {

// Shared memory one CTA of the generic kernels may use (227 KB opt-in per CTA on sm_100, some
// slack left for the driver's reservation).
constexpr size_t GEN_SMEM_MAX = 220 * 1024;
constexpr int GEN_RADICES[] = {16, 15, 12, 10, 9, 8, 6, 5, 4, 3, 2};

// Relative cost of one in-place pass per point: a fixed part (shared-memory round trip, index
// arithmetic, barrier) plus the butterfly's share -- measured on B200, a radix-5 pass costs about
// 1.6 x a radix-16 pass.
inline double gen_pass_cost(int r) { return 1.0 + 6.0 / (double)r; }

// Cheapest factorisation of n into supported radices: (cost, passes); cost < 0: impossible.
struct GenAxisCost { double cost; int passes; int first; };
inline GenAxisCost gen_axis_cost(int n, std::map<int, GenAxisCost>& memo) {
    if (n == 1) return GenAxisCost{0.0, 0, 1};
    auto it = memo.find(n);
    if (it != memo.end()) return it->second;
    GenAxisCost best{-1.0, 0, 0};
    for (int r : GEN_RADICES)
        if (n % r == 0) {
            const GenAxisCost sub = gen_axis_cost(n / r, memo);
            if (sub.cost < 0.0) continue;
            const double c = sub.cost + gen_pass_cost(r);
            if (best.cost < 0.0 || c < best.cost - 1e-12) best = GenAxisCost{c, sub.passes + 1, r};
        }
    memo[n] = best;
    return best;
}

inline bool gen_make_axis(int n, GenAxis* ax) {
    std::map<int, GenAxisCost> memo;
    const GenAxisCost top = gen_axis_cost(n, memo);
    if (n < 2 || top.cost < 0.0 || top.passes > GEN_MAX_PASSES) return false;
    ax->n = n;
    ax->npass = 0;
    std::vector<int> rs;
    for (int rest = n; rest > 1;) {
        const int r = gen_axis_cost(rest, memo).first;
        rs.push_back(r);
        rest /= r;
    }
    std::sort(rs.begin(), rs.end(), [](int a, int b) { return a > b; });   // the stride-1 pass gets the smallest radix
    for (int r : rs) ax->radix[ax->npass++] = r;
    long long prod = 1;
    for (int p = 0; p < ax->npass; p++) {
        prod *= ax->radix[p];
        ax->stride[p] = (int)(n / prod);
        ax->div_stride[p] = make_fastdiv((unsigned)ax->stride[p]);
        ax->div_items[p] = make_fastdiv((unsigned)(n / ax->radix[p]));
    }
    return true;
}

inline std::vector<int> gen_pos2freq(const GenAxis& ax) {
    std::vector<int> t(ax.n);
    for (int i = 0; i < ax.n; i++) {
        int rest = i, k = 0, weight = 1;
        for (int p = 0; p < ax.npass; p++) {
            const int d = rest / ax.stride[p];
            rest -= d * ax.stride[p];
            k += d * weight;
            weight *= ax.radix[p];
        }
        t[i] = k;
    }
    return t;
}
inline std::vector<int> gen_freq2pos(const GenAxis& ax) {
    const std::vector<int> p2f = gen_pos2freq(ax);
    std::vector<int> t(ax.n);
    for (int i = 0; i < ax.n; i++) t[p2f[i]] = i;
    return t;
}

// Row lengths for which a STATIC row kernel exists (RowFusedKernel<RL, 0, NT>: compile-time radices,
// strides and twiddle steps -- about half the time of the runtime-radix row kernel, which spends
// 45 % of its instructions on address and table arithmetic).  A runtime-radix plan whose M2 is one
// of them runs its rows there (fp32 arithmetic only); the planner prefers such splits -- every
// embedded length can choose one, and so can every length that is a multiple of 480.
inline bool gen_static_rows(long long M2) { return M2 == 480 || M2 == 960 || M2 == 1200 || M2 == 2400; }
constexpr double GEN_STATIC_ROWS_GAIN = 0.55;

// Relative cost of a split (lower is better), 0 = unusable.  elem = bytes per complex point,
// ct = columns per tile.
inline double gen_split_cost(long long M, int M1, int elem, int ct) {
    const long long M2 = M / M1;
    if (M1 < 2 || M2 < 2 || M2 > (1 << 20)) return 0.0;
    const size_t tile = (size_t)M1 * ct * elem, rows = (size_t)4 * (M2 + M2 / 8 + 1) * elem;
    if (tile > GEN_SMEM_MAX || rows > GEN_SMEM_MAX) return 0.0;
    std::map<int, GenAxisCost> memo;
    const GenAxisCost pc = gen_axis_cost(M1, memo), pr = gen_axis_cost((int)M2, memo);
    if (pc.cost < 0.0 || pr.cost < 0.0 || pc.passes > GEN_MAX_PASSES || pr.passes > GEN_MAX_PASSES) return 0.0;
    // a pass keeps a CTA's threads busy only if it has that many butterflies (radix ~10); the kernels
    // exist with 256 and with 64 threads per CTA
    auto util = [](double butterflies) { const double u = butterflies / GEN_THREADS_SMALL; return u > 1.0 ? 1.0 : (u < 0.25 ? 0.25 : u); };
    // resident CTAs per SM by shared memory (the kernels are compiled for three)
    auto occupancy_penalty = [](size_t bytes) { return bytes > 112 * 1024 ? 1.8 : (bytes > 74 * 1024 ? 1.25 : 1.0); };
    // column passes: forward on 1.5 signals + inverse on 1; row passes: forward on 2, inverse on 1
    double col = 2.5 * pc.cost / util((double)M1 * ct / 10.0) * occupancy_penalty(tile);
    if (ct * elem < 128) col *= 1.3;            // half cache lines per tile row (measured: K_A +27 % at M1 = 250)
    if (M2 % ct != 0) col *= 1.25;              // ragged last tile, rows not line-aligned
    double row = 3.0 * pr.cost / util(4.0 * (double)M2 / 10.0) * occupancy_penalty(rows);
    if (elem == 8 && gen_static_rows(M2))       // static row kernel: plain rows of exactly 4 * M2 points
        row = 3.0 * pr.cost / util(4.0 * (double)M2 / 10.0) * occupancy_penalty((size_t)4 * M2 * elem) * GEN_STATIC_ROWS_GAIN;
    return col + row;
}

inline bool gen_choose_split(long long M, int elem, bool is_double, int* M1_out, int* ct_out, double* cost_out) {
    double best = 0.0;
    int best_m1 = 0, best_ct = 0;
    for (long long d = 2; d <= 4096 && d <= M; d++) {
        if (M % d != 0) continue;
        for (int ct : {16, 8}) {
            if (is_double && ct != 8) continue;
            const double c = gen_split_cost(M, (int)d, elem, ct);
            if (c > 0.0 && (best == 0.0 || c < best)) { best = c; best_m1 = (int)d; best_ct = ct; }
        }
    }
    if (best == 0.0) return false;
    *M1_out = best_m1;
    *ct_out = best_ct;
    if (cost_out) *cost_out = best;
    return true;
}

// Shared-memory bank conflicts of the row kernel's passes for a row layout: per pass the worst
// number of lanes of one wavefront (128 bytes of lanes: 16 fp32 points, 8 fp64 points) that fall
// into the same bank group, averaged over the first butterflies and inputs; 1.0 = conflict-free.
inline double gen_row_conflicts(const GenAxis& row, int elem, bool padded) {
    const int lanes = 128 / elem, padsh = elem == 8 ? 4 : 3;
    auto phys = [&](int p) { return padded ? p + (p >> padsh) : p; };
    double total = 0.0;
    for (int ps = 0; ps < row.npass; ps++) {
        const int R = row.radix[ps], S = row.stride[ps], per_row = row.n / R;
        double worst_sum = 0.0;
        int cases = 0;
        for (int w0 = 0; w0 + lanes <= per_row && cases < 8; w0 += lanes)
            for (int q = 0; q < R && q < 4; q++) {
                int count[32] = {0};
                int worst = 0;
                for (int l = 0; l < lanes; l++) {
                    const int bf = w0 + l, blk = bf / S, j = bf - blk * S;
                    const int bank = phys(blk * S * R + j + q * S) % lanes;
                    worst = std::max(worst, ++count[bank]);
                }
                worst_sum += worst;
                cases++;
            }
        total += cases ? worst_sum / cases : 1.0;
    }
    return total / row.npass;
}

// The plan for a sample_len: the exact length when it is 2/3/5-smooth and splits, otherwise the
// cheapest embedding length M >= ceil(3L / 2) among the smooth numbers up to 15 % above the
// smallest one.  is_double: fp64 arithmetic (16-byte points, 8-column tiles).
inline bool gen_make_shape(long long L, bool is_double, GenShape* out) {
    const int elem = is_double ? 16 : 8;
    if (L < 1) return false;
    GenShape sh{};
    sh.L = L;
    int m1 = 0, ct = 0;
    double cost = 0.0;
    if (is_235_smooth(L) && gen_choose_split(L, elem, is_double, &m1, &ct, &cost)) {
        sh.M = L;
        sh.src_ext = 2 * L;
    } else {
        const long long lo = (3 * L + 1) / 2;
        std::vector<long long> cand;
        for (long long a = 1; a <= 4 * lo; a *= 2)
            for (long long b = a; b <= 4 * lo; b *= 3)
                for (long long c = b; c <= 4 * lo; c *= 5)
                    if (c >= lo) cand.push_back(c);
        std::sort(cand.begin(), cand.end());
        double best = 0.0;
        long long best_m = 0;
        int best_m1 = 0, best_ct = 0;
        long long first_ok = 0;
        for (long long m : cand) {
            if (first_ok && (double)m > 1.15 * (double)first_ok) break;
            int mm1, mct;
            double c;
            if (!gen_choose_split(m, elem, is_double, &mm1, &mct, &c)) continue;
            if (!first_ok) first_ok = m;
            const double total = c * (double)m;
            if (best == 0.0 || total < best) { best = total; best_m = m; best_m1 = mm1; best_ct = mct; }
        }
        if (best_m == 0) return false;
        sh.M = best_m;
        sh.src_ext = 3 * L;
        m1 = best_m1;
        ct = best_ct;
    }
    sh.M1 = m1;
    sh.ct = ct;
    sh.M2 = (int)(sh.M / m1);
    if (!gen_make_axis(sh.M1, &sh.col) || !gen_make_axis(sh.M2, &sh.row)) return false;
    // CTA size: the pass with the largest radix has the fewest butterflies per CTA (column tile:
    // M1 / R per column; rows: the inverse passes work on two rows)
    auto max_radix = [](const GenAxis& ax) { int m = 0; for (int p = 0; p < ax.npass; p++) m = std::max(m, ax.radix[p]); return m; };
    // rows: padded only where padding removes bank conflicts worth more than its address arithmetic
    sh.row_pad = gen_row_conflicts(sh.row, elem, true) < 0.8 * gen_row_conflicts(sh.row, elem, false) ? 1 : 0;
    // ... and only where the CTA's buffer is small enough that twelve 64-thread CTAs fit an SM
    const size_t tile_bytes = (size_t)sh.M1 * sh.ct * elem, rows_bytes = (size_t)4 * (sh.M2 + sh.M2 / 8 + 1) * elem;
    sh.nt_col = ((sh.M1 / max_radix(sh.col)) * sh.ct >= GEN_THREADS || tile_bytes > 18 * 1024) ? GEN_THREADS : GEN_THREADS_SMALL;
    sh.nt_row = ((sh.M2 / max_radix(sh.row)) * 2 >= GEN_THREADS || rows_bytes > 18 * 1024) ? GEN_THREADS : GEN_THREADS_SMALL;
    sh.static_rows = (!is_double && gen_static_rows(sh.M2)) ? 1 : 0;
    *out = sh;
    return true;
}

// r_reference = r_computed * gen_peak_scale: the split/merge leaves a factor 2 (its 1/2 is not
// applied in the generic kernels) and an embedded transform carries N' = 2M instead of N = 2L.
inline double gen_peak_scale(const GenShape& sh) { return 0.5 * (double)sh.L / (double)sh.M; }

template <class C>
struct GenTables {
    std::vector<C> wcol, wrow, wpos, m_lo, m_hi;
    std::vector<C> phat_pos, phat_lo, phat_hi;    // PHAT split: w = W_N^k1 * phat_pos[e], N = 2M
    std::vector<int> p2f_col, p2f_row, f2p_row;
};

template <class C>
inline GenTables<C> gen_build_tables(const GenShape& sh) {
    GenTables<C> t;
    t.wcol.resize(sh.M1);
    for (int a = 0; a < sh.M1; a++) t.wcol[a] = unit_root_as<C>(a, sh.M1);
    t.wrow.resize(sh.M2);
    for (int a = 0; a < sh.M2; a++) t.wrow[a] = unit_root_as<C>(a, sh.M2);
    t.m_lo.resize(1u << TW2_BITS);
    for (long long a = 0; a < (long long)t.m_lo.size(); a++) t.m_lo[a] = unit_root_as<C>(a, sh.M);
    const long long nh = ((sh.M - 1) >> TW2_BITS) + 1;
    t.m_hi.resize(nh);
    for (long long b = 0; b < nh; b++) t.m_hi[b] = unit_root_as<C>(b << TW2_BITS, sh.M);
    t.p2f_col = gen_pos2freq(sh.col);
    t.p2f_row = gen_pos2freq(sh.row);
    t.f2p_row = gen_freq2pos(sh.row);
    t.wpos.resize(sh.M2);
    for (int e = 0; e < sh.M2; e++) t.wpos[e] = t.wrow[t.p2f_row[e]];
    t.phat_pos.resize(sh.M2);
    for (int e = 0; e < sh.M2; e++) t.phat_pos[e] = unit_root_as<C>(t.p2f_row[e], 2LL * sh.M2);
    t.phat_lo.resize(1u << TW2_BITS);
    for (long long a = 0; a < (long long)t.phat_lo.size(); a++) t.phat_lo[a] = unit_root_as<C>(a, 2 * sh.M);
    t.phat_hi.resize(((sh.M1 / 2) >> TW2_BITS) + 1);      // k1 <= M1 / 2
    for (long long b = 0; b < (long long)t.phat_hi.size(); b++) t.phat_hi[b] = unit_root_as<C>(b << TW2_BITS, 2 * sh.M);
    return t;
}

inline std::string gen_describe(const GenShape& sh, bool is_double) {
    std::string d = "fft L=" + std::to_string(sh.L) + " M=" + std::to_string(sh.M) + " M1=" + std::to_string(sh.M1) +
                    " M2=" + std::to_string(sh.M2) + " col=";
    for (int i = 0; i < sh.col.npass; i++) d += (i ? "x" : "") + std::to_string(sh.col.radix[i]);
    d += " row=";
    for (int i = 0; i < sh.row.npass; i++) d += (i ? "x" : "") + std::to_string(sh.row.radix[i]);
    d += std::string(sh.row_pad ? " padded" : " plain") + " tile=" + std::to_string(sh.ct) + " threads=" + std::to_string(sh.nt_col) + "/" + std::to_string(sh.nt_row);
    if (sh.static_rows && !is_double) d += " static-rows";
    d += sh.M == sh.L ? " generic four-step" : " generic four-step, embedded (N'=2M>=3L)";
    d += is_double ? " fp64" : " fp32";
    return d;
}

// ------------------------------------------------------------- path choice
enum PathKind { PATH_STATIC_FFT, PATH_SMALL_FFT, PATH_DIRECT, PATH_GENERIC_FFT, PATH_NONE };

// Below this length AUTO prefers the fp64 time-domain kernel: it costs
// microseconds and keeps fp64 accuracy where the reference's own tests live
// (tests/test_cross_correlation.c T7: sin(i), L = 1000, has two peaks that
// differ by 1.2e-9 relative -- unresolvable by an fp32 transform).
constexpr long long DIRECT_AUTO_BELOW = 4096;
// The O(L^2) kernel is never chosen above this length (2 * L^2 = 8.6e9 fp64 FMAs, a millisecond
// on B200); longer inputs without a transform plan are refused, not ground through.
constexpr long long DIRECT_MAX_L = 65536;
// Shortest length the runtime-radix kernels are used for when a transform is asked for.
constexpr long long GEN_MIN_L = 256;

// precise: fp64 ARITHMETIC (validation mode).  The direct kernel is fp64 already; every
// transform then runs on the fp64 instantiation of the runtime-radix kernels.
inline PathKind choose_path(long long L, int forced, bool precise = false) {
    if (forced == AUDIOSYNC_CUDA_PATH_DIRECT) return L <= DIRECT_MAX_L ? PATH_DIRECT : PATH_NONE;
    GenShape gs;
    if (precise) {
        if (L >= (forced == AUDIOSYNC_CUDA_PATH_FFT ? GEN_MIN_L : DIRECT_AUTO_BELOW) && gen_make_shape(L, true, &gs))
            return PATH_GENERIC_FFT;
        return L <= DIRECT_MAX_L ? PATH_DIRECT : PATH_NONE;
    }
    if (has_static_plan(L)) return PATH_STATIC_FFT;
    if (forced != AUDIOSYNC_CUDA_PATH_FFT && L < DIRECT_AUTO_BELOW) return PATH_DIRECT;
    SmallPlan sp;
    if (make_small_plan(L, &sp)) return PATH_SMALL_FFT;
    if (L >= GEN_MIN_L && gen_make_shape(L, false, &gs)) return PATH_GENERIC_FFT;
    return L <= DIRECT_MAX_L ? PATH_DIRECT : PATH_NONE;   // short lengths without a plan (FFT forced on a tiny odd L)
}

// The path of a PHAT-weighted context.  PHAT is defined on the N = 2L spectrum, so only plans that
// transform at N = 2L serve it: the static plans, the single-CTA kernel (also below 4,096 frames)
// and the runtime-radix plans at the length's own size (precise: fp64 arithmetic).  Never the
// time-domain kernel, which has no spectrum, nor an embedded plan, whose weighted N'-point spectrum
// is a different function and would depend on the planner's choice of M.  PATH_NONE comes with the
// reason in *why.
inline PathKind choose_path_phat(long long L, int forced, bool precise, const char** why) {
    *why = nullptr;
    if (forced == AUDIOSYNC_CUDA_PATH_DIRECT) {
        *why = "PHAT weighting needs a transform; PATH_DIRECT has none";
        return PATH_NONE;
    }
    SmallPlan sp;
    if (!precise && has_static_plan(L)) return PATH_STATIC_FFT;
    if (!precise && make_small_plan(L, &sp)) return PATH_SMALL_FFT;
    GenShape gs;
    if (L >= GEN_MIN_L && gen_make_shape(L, precise, &gs)) {
        if (gs.M == L) return PATH_GENERIC_FFT;
        *why = "PHAT weighting is defined on the N = 2L spectrum; this length is not 2/3/5-smooth and would be embedded in N' = 2M >= 3L";
        return PATH_NONE;
    }
    *why = "no transform plan at N = 2L for PHAT weighting";
    return PATH_NONE;
}

}  // namespace asc
