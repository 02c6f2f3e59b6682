// fft_plan.h -- host-side planning shared by the product library and the CPU
// emulator: which path a sample_len takes, the static four-step plans for the
// reference's interval schedule, and the twiddle tables (computed in long
// double on the host, rounded once to fp32 -- never sincosf on the device).
#pragma once

#include <cmath>
#include <string>
#include <tuple>
#include <vector>

#include "fft_device.cuh"
#include "fft_small.cuh"

namespace asc {

// ------------------------------------------------------------ static plans
// One per entry of the reference's interval schedule (src/audiosync.c:50-57:
// sample_len = {3, 6, 10, 15, 20, 30} s x 48 kHz).  M = L = M1 * M2 with M2 a
// multiple of 16 (full 128-byte lines per tile row) and even.  Row radix lists
// are (a, b, 15): the stride-1 pass has an odd radix (free of bank conflicts)
// and the stride-15 pass runs with 16 thread slots per block (see
// RowFusedKernel::slots).
struct Plan144k {
    static constexpr long long L = 144000;
    using Col = RadixList<10, 6, 5>;     // M1 = 300
    using Row = RadixList<4, 8, 15>;     // M2 = 480
    static constexpr int NT_COL = 160, NT_ROW = 128;
};
struct Plan288k {
    static constexpr long long L = 288000;
    using Col = RadixList<10, 6, 5>;     // M1 = 300
    using Row = RadixList<4, 16, 15>;    // M2 = 960
    static constexpr int NT_COL = 160, NT_ROW = 256;
};
struct Plan480k {
    static constexpr long long L = 480000;
    using Col = RadixList<10, 10, 4>;    // M1 = 400
    using Row = RadixList<5, 16, 15>;    // M2 = 1200
    static constexpr int NT_COL = 320, NT_ROW = 320;
};
struct Plan720k {
    static constexpr long long L = 720000;
    using Col = RadixList<10, 10, 6>;    // M1 = 600
    using Row = RadixList<5, 16, 15>;    // M2 = 1200
    static constexpr int NT_COL = 320, NT_ROW = 320;
};
struct Plan960k {
    static constexpr long long L = 960000;
    using Col = RadixList<10, 10, 4>;    // M1 = 400
    using Row = RadixList<10, 16, 15>;   // M2 = 2400
    static constexpr int NT_COL = 320, NT_ROW = 320;
};
struct Plan1440k {
    static constexpr long long L = 1440000;
    using Col = RadixList<10, 10, 6>;    // M1 = 600
    using Row = RadixList<10, 16, 15>;   // M2 = 2400
    static constexpr int NT_COL = 320, NT_ROW = 320;
};

using StaticPlans = std::tuple<Plan144k, Plan288k, Plan480k, Plan720k, Plan960k, Plan1440k>;

template <class P>
constexpr bool plan_is_consistent() {
    return (long long)P::Col::n * P::Row::n == P::L && P::Row::n % COL_T == 0 && P::Row::n % 2 == 0;
}
static_assert(plan_is_consistent<Plan144k>() && plan_is_consistent<Plan288k>() &&
              plan_is_consistent<Plan480k>() && plan_is_consistent<Plan720k>() &&
              plan_is_consistent<Plan960k>() && plan_is_consistent<Plan1440k>(),
              "static plan: M1*M2 != L or M2 not a multiple of 16");

template <class RL>
inline std::vector<int> radix_vector() {
    std::vector<int> v;
    for (int i = 0; i < RL::count; i++) v.push_back(RL::r(i));
    return v;
}

template <class F, size_t... I>
inline void for_each_static_plan_impl(F&& f, std::index_sequence<I...>) {
    (f(std::tuple_element_t<I, StaticPlans>{}), ...);
}
template <class F>
inline void for_each_static_plan(F&& f) {
    for_each_static_plan_impl(static_cast<F&&>(f),
                              std::make_index_sequence<std::tuple_size<StaticPlans>::value>{});
}

inline bool has_static_plan(long long L) {
    bool found = false;
    for_each_static_plan([&](auto P) { if (decltype(P)::L == L) found = true; });
    return found;
}

// --------------------------------------------------------------- twiddles
// exp(-2*pi*i*a/base) as (cos, -sin) in long double
inline void unit_root_ld(long long a, long long base, long double* re, long double* im) {
    a %= base;
    const long double two_pi = 6.283185307179586476925286766559005768L;
    // reduce to the first octant so that sinl/cosl see a small argument
    long long q8 = (8 * a) / base;                      // octant 0..7
    long double c, s;
    auto cs = [&](long double num) {                    // angle = 2*pi*num/base
        long double th = two_pi * num / (long double)base;
        c = cosl(th); s = sinl(th);
    };
    switch (q8) {
        case 0: cs((long double)a); break;
        case 1: { cs((long double)(base / 4.0L - a)); long double t = c; c = s; s = t; } break;
        case 2: { cs((long double)(a - base / 4.0L)); long double t = c; c = -s; s = t; } break;
        case 3: { cs((long double)(base / 2.0L - a)); c = -c; } break;
        case 4: { cs((long double)(a - base / 2.0L)); c = -c; s = -s; } break;
        case 5: { cs((long double)(3.0L * base / 4.0L - a)); long double t = c; c = -s; s = -t; } break;
        case 6: { cs((long double)(a - 3.0L * base / 4.0L)); long double t = c; c = s; s = -t; } break;
        default: { cs((long double)(base - a)); s = -s; } break;
    }
    *re = c; *im = -s;
}
inline cplx unit_root(long long a, long long base) {   // rounded once to fp32
    long double re, im;
    unit_root_ld(a, base, &re, &im);
    return cmake((float)re, (float)im);
}
template <class C>
inline C unit_root_as(long long a, long long base) {    // fp32 or fp64
    long double re, im;
    unit_root_ld(a, base, &re, &im);
    typedef typename scalar_of<C>::type real;
    return cmake((real)re, (real)im);
}

// Pass tables for an in-place DIF radix list (layout: RadixList::tw_offset):
// per pass only the power-of-two multiples exp(-2*pi*i*j*2^i/(s*r)), 2^i < r.
inline std::vector<cplx> build_pass_tables(const std::vector<int>& radices) {
    long long n = 1;
    for (int r : radices) n *= r;
    std::vector<cplx> t;
    long long prod = 1;
    for (size_t p = 0; p < radices.size(); p++) {
        prod *= radices[p];
        const long long s = n / prod, m = s * radices[p];
        for (int k = 1; k < radices[p]; k *= 2)
            for (long long j = 0; j < s; j++) t.push_back(unit_root(j * k, m));
    }
    return t;
}

// K_A last-pass table: tc[f0][c] = exp(-2*pi*i*c*f0/M), f0 < wt, c < 16.
inline std::vector<cplx> build_col_tc(long long M, int wt) {
    std::vector<cplx> t((size_t)wt * COL_T);
    for (int f0 = 0; f0 < wt; f0++)
        for (int c = 0; c < COL_T; c++) t[(size_t)f0 * COL_T + c] = unit_root((long long)c * f0, M);
    return t;
}

// K_B split/merge table in POSITION order: rev[e] = exp(-2*pi*i*freq_of_pos(e)/M2)
// (the M1*k2 part of w^2 = exp(-2*pi*i*(k1 + M1*k2)/M), see split_mul_merge_w2).
template <class RL>
inline std::vector<cplx> build_row_rev() {
    std::vector<cplx> t(RL::n);
    for (int e = 0; e < RL::n; e++) t[e] = unit_root(RL::freq_of_pos(e), (long long)RL::n);
    return t;
}

// PHAT split tables (split_phat_merge needs w = exp(-2*pi*i*k/N), N = 2M, where the product needs
// w^2): in POSITION order exp(-2*pi*i*freq_of_pos(e)/(2*M2)), the half angles of build_row_rev; the
// W_N^k1 part comes from build_two_level(2M, M1 / 2).
template <class RL>
inline std::vector<cplx> build_row_rev_half() {
    std::vector<cplx> t(RL::n);
    for (int e = 0; e < RL::n; e++) t[e] = unit_root(RL::freq_of_pos(e), 2 * (long long)RL::n);
    return t;
}

// K_B final-pass tables, one row per k1 (layout: RowFusedKernel::TABP): S0 entries
// 0.5 * exp(-2*pi*i*j*k1/M), then R0 entries exp(-2*pi*i*k*S0*k1/M), zero padded to an even count.
template <class RL>
inline std::vector<cplx> build_row_tab(long long M, int M1) {
    constexpr int S0 = RL::stride(0), R0 = RL::r(0), TABP = (S0 + R0 + 1) & ~1;
    std::vector<cplx> t((size_t)M1 * TABP, cmake(0.f, 0.f));
    for (int k1 = 0; k1 < M1; k1++) {
        cplx* row = t.data() + (size_t)k1 * TABP;
        for (int j = 0; j < S0; j++) {
            const cplx u = unit_root((long long)j * k1, M);
            row[j] = cmake(0.5f * u.x, 0.5f * u.y);
        }
        for (int k = 0; k < R0; k++) row[S0 + k] = unit_root((long long)k * S0 * k1, M);
    }
    return t;
}

// Two-level tables for exp(-2*pi*i*a/base), a in [0, max_index].
inline void build_two_level(long long base, long long max_index, std::vector<cplx>& lo,
                            std::vector<cplx>& hi) {
    lo.resize(1u << TW2_BITS);
    for (long long a = 0; a < (long long)lo.size(); a++) lo[a] = unit_root(a, base);
    const long long nh = (max_index >> TW2_BITS) + 1;
    hi.resize(nh);
    for (long long b = 0; b < nh; b++) hi[b] = unit_root(b << TW2_BITS, base);
}

inline std::vector<cplx> build_full_table(long long base, long long count) {
    std::vector<cplx> t(count);
    for (long long a = 0; a < count; a++) t[a] = unit_root(a, base);
    return t;
}

// ------------------------------------------------------------- path choice
inline bool is_235_smooth(long long n) {
    if (n <= 0) return false;
    for (int p : {2, 3, 5}) while (n % p == 0) n /= p;
    return n == 1;
}

// Short-length plan: even, 2/3/5-smooth, M <= SMALL_MAX_M, at least 2 points.
inline bool make_small_plan(long long L, SmallPlan* out) {
    if (L < 2 || L % 2 != 0 || L > SMALL_MAX_M || !is_235_smooth(L)) return false;
    SmallPlan pl;
    pl.M = (int)L;
    pl.npass = 0;
    long long r = L;
    // radix order: 4s and 2 first, odd radices last (stride-1 pass conflict-free)
    auto push = [&](int f) { pl.radix[pl.npass++] = f; r /= f; };
    while (r % 4 == 0) push(4);
    while (r % 2 == 0) push(2);
    while (r % 3 == 0) push(3);
    while (r % 5 == 0) push(5);
    if (pl.npass > SMALL_MAX_PASSES) return false;
    long long prod = 1;
    for (int p = 0; p < pl.npass; p++) {
        prod *= pl.radix[p];
        pl.stride[p] = (int)(L / prod);
    }
    *out = pl;
    return true;
}

}  // namespace asc
