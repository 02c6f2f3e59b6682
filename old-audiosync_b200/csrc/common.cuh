// common.cuh -- shared device/host helpers for libaudiosync_cuda (sm_100a).
#pragma once

#include <cuda_runtime.h>
#include <stdint.h>
#include <stddef.h>
#include <math.h>
#include <type_traits>

#include "../../include/audiosync_cuda.h"

namespace asc {

// ---------------------------------------------------------------------------
// Argmax key.  The reference's max_abs_index (src/cross_correlation.c:52-67)
// keeps a running maximum seeded with the SIGNED r[0]; entries i >= 1 compete
// with |r[i]| under a strict '>' in ascending order.  As a commutative
// reduction that is the lexicographic maximum of (value, -index) with
//   value(0)   = r[0]            (NaN -> +inf: an incumbent NaN is never beaten)
//   value(i>0) = |r[i]|          (NaN -> lowest: a NaN never wins)
// For the fp32 transform path the pair is packed into one 64-bit word so a
// single atomicMax per CTA resolves it: high word = order-preserving image of
// the float, low word = ~index (smaller index => larger key).
// ---------------------------------------------------------------------------
__host__ __device__ __forceinline__ uint32_t float_order_bits(float v) {
#if defined(__CUDA_ARCH__)
    uint32_t u = __float_as_uint(v);
#else
    union { float f; uint32_t u; } c; c.f = v; uint32_t u = c.u;
#endif
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

__host__ __device__ __forceinline__ float float_from_order_bits(uint32_t k) {
    uint32_t u = (k & 0x80000000u) ? (k & 0x7fffffffu) : ~k;
#if defined(__CUDA_ARCH__)
    return __uint_as_float(u);
#else
    union { float f; uint32_t u; } c; c.u = u; return c.f;
#endif
}

// i >= 1 : magnitude key.  NaN maps to 0 (below every real key, incl. -inf's).
// Low word = (~index << 1) | sign(v): indices are < 2^31 so the dropped top bit
// of ~index is constant, order by index is preserved, and the sign of the
// winning entry travels with the key (needed to report the signed peak).
__host__ __device__ __forceinline__ uint64_t argmax_key_abs(float v, uint32_t index) {
    float a = fabsf(v);                       // clears the sign of -0.0 too
    uint32_t hi = (a != a) ? 0u : float_order_bits(a);
    uint32_t lo = ((~index) << 1) | ((v < 0.f) ? 1u : 0u);
    return ((uint64_t)hi << 32) | lo;
}

// i == 0 : signed seed.  NaN maps to the top key.
__host__ __device__ __forceinline__ uint64_t argmax_key_seed(float v) {
    v = v + 0.0f;                             // -0.0 -> +0.0 (compares equal to |0| in the reference)
    uint32_t hi = (v != v) ? 0xffffffffu : float_order_bits(v);
    return ((uint64_t)hi << 32) | 0xfffffffeu;
}

__host__ __device__ __forceinline__ uint32_t argmax_key_index(uint64_t key) {
    uint32_t lo = (uint32_t)(key & 0xffffffffu);
    return ~((lo >> 1) | 0x80000000u);
}

// the seed's key (index 0): abs keys carry an index >= 1 < 2^31, so their low word differs
__host__ __device__ __forceinline__ bool argmax_key_is_seed(uint64_t key) {
    return ((uint32_t)(key & 0xffffffffu) >> 1) == 0x7fffffffu;
}

// signed value of the winning entry
__host__ __device__ __forceinline__ float argmax_key_value(uint64_t key) {
    float m = float_from_order_bits((uint32_t)(key >> 32));
    return (key & 1ull) ? -m : m;
}

// Per-pair scratch record produced by the transform path, consumed by the
// Pearson kernels (device only).
struct PairPeak {
    unsigned long long key;   // packed argmax key (fp32 path) -- atomicMax target
    long long raw_index;      // resolved index (direct path writes it directly)
    double peak;              // r[raw_index]
    double second;            // resolved second peak (direct path)
    int resolved;             // 1 if raw_index/peak/second are already final
    unsigned int second_bits; // fp32 path: order bits of the largest |r[i]|, i >= 1, i != argmax (0: none yet)
    unsigned int seed_bits;   // fp32 path: order bits of |r[0]| (0: not written yet)
};

__host__ __device__ __forceinline__ PairPeak cleared_peak() {
    PairPeak z;
    z.key = 0ull; z.raw_index = 0; z.peak = 0.0; z.second = 0.0; z.resolved = 0; z.second_bits = 0u; z.seed_bits = 0u;
    return z;
}

// |value| carried by a packed key (abs keys hold |v|, the seed key holds the signed r[0]).
__host__ __device__ __forceinline__ float argmax_key_mag(uint64_t key) {
    return fabsf(float_from_order_bits((uint32_t)(key >> 32)));
}

// Second peak of the fp32 transform path: the largest |r[i]| over i >= 1 other than the peak
// (second_bits), joined by |r[0]| unless r[0] is the peak.  r[0] is kept out of second_bits
// because second_bits is also the threshold below which the kernels skip candidates, and a
// negative r[0] may lose while being the largest magnitude (see ArgmaxAcc).
__host__ __device__ __forceinline__ float pair_second(const PairPeak& p) {
    float s = p.second_bits != 0u ? float_from_order_bits(p.second_bits) : 0.0f;
    if (p.seed_bits != 0u && argmax_key_index(p.key) != 0u) s = fmaxf(s, float_from_order_bits(p.seed_bits));
    return s;
}

// Lag window of the batch calls (audiosync_cuda_set_lag_window) as the raw indices it allows:
// [lo0, lo0 + n0) and [lo1, lo1 + n1) of [0, 2L), lo0 the lowest allowed index (n1 = 0: one range).
struct RawWindow {
    uint32_t lo0, n0, lo1, n1;
    __host__ __device__ __forceinline__ bool allows(uint32_t i) const { return i - lo0 < n0 || i - lo1 < n1; }
};
// the unwindowed kernels' (empty) window parameter
struct NoWindow {};
// every raw index of [0, 2L): the windowed argmax then gives the unwindowed kernels' record
__host__ __device__ __forceinline__ RawWindow full_window(long long L) { return RawWindow{0u, (uint32_t)(2 * L), 0u, 0u}; }

// Correlation export of audiosync_cuda_xcorr_correlation: pair p's value at raw index i of range k
// of `range` is stored, as (double)value * scale, at out[p * W + off_k + (i - lo_k)].  `out` points
// at the wave's first row; offsets are 64-bit (pairs * W can exceed 2^31).
struct CorrOut {
    double* out;
    long long W;
    RawWindow range;
    uint32_t off0, off1;
    double scale;
    __host__ __device__ __forceinline__ void store(long long pair, uint32_t i, double v) const {
        if (i - range.lo0 < range.n0) out[pair * W + (long long)(off0 + (i - range.lo0))] = v * scale;
        else if (i - range.lo1 < range.n1) out[pair * W + (long long)(off1 + (i - range.lo1))] = v * scale;
    }
    // fp32 kernels: the value the peak search compared, as pearson_block scales the peak (-0 as +0,
    // as argmax_key_value returns it)
    __host__ __device__ __forceinline__ void store(long long pair, uint32_t i, float v) const {
        store(pair, i, (double)(v + 0.0f));
    }
};

// The export range [lo, hi] of folded lags (-L <= lo <= hi <= L - 1) as raw ranges and output offsets.
__host__ __device__ __forceinline__ CorrOut corr_out_of(long long lo, long long hi, long long L, double* out, double scale) {
    CorrOut c;
    c.out = out;
    c.W = hi - lo + 1;
    c.scale = scale;
    if (lo >= 0) { c.range = RawWindow{(uint32_t)lo, (uint32_t)c.W, 0u, 0u}; c.off0 = 0u; c.off1 = 0u; }
    else if (hi < 0) { c.range = RawWindow{(uint32_t)(lo + 2 * L), (uint32_t)c.W, 0u, 0u}; c.off0 = 0u; c.off1 = 0u; }
    else { c.range = RawWindow{0u, (uint32_t)(hi + 1), (uint32_t)(lo + 2 * L), (uint32_t)(-lo)}; c.off0 = (uint32_t)(-lo); c.off1 = 0u; }
    return c;
}

// Effective window [max(lo, -L), min(hi, L - 1)] of folded lags as raw ranges: raw = lag for lag >= 0,
// lag + 2L below.  Returns -1 when it is empty, 0 when it is all of [-L, L - 1] (the unwindowed call),
// 1 otherwise (*w filled, *elo / *ehi the effective lags).
__host__ __device__ __forceinline__ int raw_window_of(long long lo, long long hi, long long L, RawWindow* w,
                                                      long long* elo = nullptr, long long* ehi = nullptr) {
    if (lo < -L) lo = -L;
    if (hi > L - 1) hi = L - 1;
    if (lo > hi) return -1;
    if (elo) *elo = lo;
    if (ehi) *ehi = hi;
    if (lo == -L && hi == L - 1) return 0;
    if (lo >= 0) *w = RawWindow{(uint32_t)lo, (uint32_t)(hi - lo + 1), 0u, 0u};
    else if (hi < 0) *w = RawWindow{(uint32_t)(lo + 2 * L), (uint32_t)(hi - lo + 1), 0u, 0u};
    else *w = RawWindow{0u, (uint32_t)(hi + 1), (uint32_t)(lo + 2 * L), (uint32_t)(-lo)};
    return 1;
}

// Fold of src/cross_correlation.c:256-271.  Window = x[xoff .. xoff+n) of the
// source against y[yoff .. yoff+n) of the sample.
struct Window { long long lag; long long xoff; long long yoff; long long n; };

__host__ __device__ __forceinline__ Window fold_index(long long idx, long long L) {
    Window w;
    if (idx >= L) {
        w.lag = (idx % L) - L;
        w.xoff = 0;
        w.yoff = -w.lag;
        w.n = L + w.lag;
    } else {
        w.lag = idx;
        w.xoff = idx;
        w.yoff = 0;
        w.n = L;
    }
    return w;
}

// Runner-up search of audiosync_cuda_xcorr_runner_up: the raw indices pair i may pick from, as at most
// three ranges in ascending raw order (lo0 the lowest allowed index).  An empty set has n0 = n1 = n2 = 0
// and lo0 = 0xffffffff, which is no index.
struct PairWindow {
    uint32_t lo0, n0, lo1, n1, lo2, n2;
    __host__ __device__ __forceinline__ bool allows(uint32_t i) const {
        return i - lo0 < n0 || i - lo1 < n1 || i - lo2 < n2;
    }
    __host__ __device__ __forceinline__ bool empty() const { return n0 == 0u; }
};

// A(p) = { l in [lo, hi] : |l - p| >= D } ([lo, hi] the effective lag window, D >= 1) as raw ranges.
// Its two folded intervals [lo, p - D] and [p + D, hi] each have a part at lags >= 0 (raw = lag) and
// one below (raw = lag + 2L); only one interval can hold lag 0, so at most three parts are non-empty.
__host__ __device__ __forceinline__ PairWindow runner_up_window(long long p, long long lo, long long hi, long long D,
                                                                long long L) {
    if (D > 2 * L) D = 2 * L;                      // every pair of lags is closer than 2L
    const long long a0 = lo, b0 = p - D < hi ? p - D : hi;          // [lo, p - D]
    const long long a1 = p + D > lo ? p + D : lo, b1 = hi;          // [p + D, hi]
    PairWindow w{0xffffffffu, 0u, 0u, 0u, 0u, 0u};
    auto put = [&](long long s, long long n) {     // the next non-empty range, in ascending raw order
        if (n <= 0) return;
        if (w.n0 == 0u) { w.lo0 = (uint32_t)s; w.n0 = (uint32_t)n; }
        else if (w.n1 == 0u) { w.lo1 = (uint32_t)s; w.n1 = (uint32_t)n; }
        else { w.lo2 = (uint32_t)s; w.n2 = (uint32_t)n; }
    };
    // lags >= 0 (raw = lag), then lags < 0 (raw = lag + 2L, above every lag >= 0)
    put(a0 > 0 ? a0 : 0, b0 - (a0 > 0 ? a0 : 0) + 1);
    put(a1 > 0 ? a1 : 0, b1 - (a1 > 0 ? a1 : 0) + 1);
    put(a0 + 2 * L, (b0 < -1 ? b0 : -1) - a0 + 1);
    put(a1 + 2 * L, (b1 < -1 ? b1 : -1) - a1 + 1);
    return w;
}

// The runner-up twins' descriptor: pair i's centre p is the folded lag of first[i].raw_index, the wave's
// records of the batch call (written by the preceding Pearson step).
struct RunnerUp {
    const audiosync_cuda_result* first;
    long long lo, hi;               // the effective lag window
    long long D;                    // min_separation >= 1
    long long L;
    __host__ __device__ __forceinline__ PairWindow window(long long pair) const {
        return runner_up_window(fold_index(first[pair].raw_index, L).lag, lo, hi, D, L);
    }
};

// What a windowed kernel searches for `pair`: the call's lag window, or (RU: the runner-up twins, whose
// parameters add a RunnerUp `ru`) the pair's runner-up set.
template <bool RU, class Pm>
__host__ __device__ __forceinline__ decltype(auto) search_window(const Pm& p, long long pair) {
    if constexpr (RU) {
        return p.ru.window(pair);
    } else {
        (void)pair;
        return (p.win);
    }
}

// splitmix64 finaliser used by the seeded generator (oracle/xcorr_oracle.c).
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ULL;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ULL;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBULL;
    return z ^ (z >> 31);
}

}  // namespace asc
