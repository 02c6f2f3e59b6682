// reduce_kernels.cuh -- non-FFT kernels of the path: seeded generator, the
// universal time-domain (direct) correlation, argmax resolution, Pearson.
#pragma once

#include "common.cuh"
#include "fft_device.cuh"   // in_real: the input element as a real

namespace asc {

// ---------------------------------------------------------------------------
// Seeded synthetic pairs (SURVEY.md 8d; same integers as oracle/xcorr_oracle.c
// synth_pair_i32).  grid = (blocks, n_pairs); element e < 2L -> source[e],
// else sample[e - 2L].
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256)
synth_kernel(T* __restrict__ sources, T* __restrict__ samples, uint64_t seed,
             uint64_t first_pair, long long L)
{
    const uint64_t pair = first_pair + blockIdx.y;
    const uint64_t k0 = seed ^ (pair * 0xD1342543DE82EF95ULL);
    const uint64_t k1 = k0 ^ 0xA0761D6478BD642FULL;
    const uint64_t k2 = k0 ^ (2ULL * 0xA0761D6478BD642FULL);
    const long long tl = (long long)(splitmix64(k2) % (uint64_t)(L + 1)) - (L / 2);
    const long long amp = (pair % 4 == 3) ? 768 : 102;
    const long long half = L / 2;
    T* src = sources + (size_t)blockIdx.y * (size_t)(2 * L);
    T* smp = samples + (size_t)blockIdx.y * (size_t)L;
    const T scale = (T)(1.0 / 8388608.0);
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < 3 * L;
         e += (long long)gridDim.x * blockDim.x) {
        if (e < 2 * L) {
            long long q = (long long)(splitmix64(k0 + (uint64_t)(half + e)) >> 40) - (1LL << 23);
            src[e] = (T)q * scale;
        } else {
            long long j = e - 2 * L;
            long long b = (long long)(splitmix64(k0 + (uint64_t)(half + tl + j)) >> 40) - (1LL << 23);
            long long n = (long long)(splitmix64(k1 + (uint64_t)j) >> 40) - (1LL << 23);
            smp[j] = (T)(b + ((n * amp) >> 10)) * scale;
        }
    }
}

// f64le frames -> fp32 slot of a session pool (the wire-format conversion, on arrival).
static __global__ void __launch_bounds__(256)
convert_f64_to_f32_kernel(const double* __restrict__ in, float* __restrict__ out, long long n)
{
    for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
         i += (long long)gridDim.x * blockDim.x)
        out[i] = (float)in[i];
}

// ---------------------------------------------------------------------------
// Direct path: r[j] = N * sum_{n<L} source[(n + j) mod N] * sample[n], the
// quantity c2r(r2c(source) * conj(r2c(pad(sample)))) equals (reference
// src/cross_correlation.c:232-239, FFTW's unnormalised c2r).  fp64
// accumulation, any L.  grid = (ceil(N / 256), n_pairs), block = 256.
// ---------------------------------------------------------------------------
constexpr int DIRECT_TILE = 256;

template <typename T>
__global__ void __launch_bounds__(DIRECT_TILE)
direct_corr_kernel(const T* __restrict__ sources, const T* __restrict__ samples,
                   double* __restrict__ r_out, long long L, long long src_pitch, long long smp_pitch)
{
    __shared__ double s_smp[DIRECT_TILE];
    __shared__ double s_src[2 * DIRECT_TILE];
    const long long N = 2 * L;
    const T* src = sources + (size_t)blockIdx.y * (size_t)src_pitch;
    const T* smp = samples + (size_t)blockIdx.y * (size_t)smp_pitch;
    const long long j0 = (long long)blockIdx.x * DIRECT_TILE;
    const int t = threadIdx.x;
    double acc = 0.0;
    for (long long n0 = 0; n0 < L; n0 += DIRECT_TILE) {
        s_smp[t] = (n0 + t < L) ? in_real<double>(smp[n0 + t]) : 0.0;
        s_src[t] = in_real<double>(src[(j0 + n0 + t) % N]);
        s_src[t + DIRECT_TILE] = in_real<double>(src[(j0 + n0 + t + DIRECT_TILE) % N]);
        __syncthreads();
#pragma unroll 8
        for (int i = 0; i < DIRECT_TILE; i++) acc = fma(s_smp[i], s_src[t + i], acc);
        __syncthreads();
    }
    if (j0 + t < N) r_out[(size_t)blockIdx.y * (size_t)N + j0 + t] = acc * (double)N;
}

// Argmax over a double array with the reference's semantics, plus the second peak
// (largest |r[i]|, i != argmax; NaNs never count).  One CTA / pair.
struct KeyF64 {
    double v;       // compare value: signed r[0] for i == 0, |r[i]| otherwise (NaN handling below)
    long long i;
    double a;       // |r[i]| of this candidate (0 for NaN)
    double s;       // second peak of the set this candidate leads
};

__device__ __forceinline__ KeyF64 key_better(KeyF64 a, KeyF64 b) {
    // larger value wins; equal values -> smaller index wins; the loser's magnitude and both
    // sets' second peaks are second-peak candidates of the union
    const bool pick_b = b.v > a.v || (b.v == a.v && b.i < a.i);
    KeyF64 w = pick_b ? b : a;
    const KeyF64 l = pick_b ? a : b;
    double s = fmax(a.s, b.s);
    if (l.i != 0x7fffffffffffffffLL) s = fmax(s, l.a);
    w.s = s;
    return w;
}

__device__ __forceinline__ KeyF64 key_shfl_xor(KeyF64 k, int o) {
    KeyF64 c;
    c.v = __shfl_xor_sync(0xffffffffu, k.v, o);
    c.i = __shfl_xor_sync(0xffffffffu, k.i, o);
    c.a = __shfl_xor_sync(0xffffffffu, k.a, o);
    c.s = __shfl_xor_sync(0xffffffffu, k.s, o);
    return c;
}

// `pitch`: doubles between consecutive pairs' arrays (N when packed).
static __global__ void __launch_bounds__(1024)
argmax_f64_kernel(const double* __restrict__ r, long long N, long long pitch, PairPeak* __restrict__ peaks)
{
    __shared__ KeyF64 s_k[32];
    const double* rp = r + (size_t)blockIdx.x * (size_t)pitch;
    const double ninf = -INFINITY, pinf = INFINITY;
    KeyF64 best; best.v = ninf; best.i = 0x7fffffffffffffffLL; best.a = 0.0; best.s = 0.0;
    for (long long i = threadIdx.x; i < N; i += blockDim.x) {
        double x = rp[i];
        KeyF64 c;
        c.i = i;
        const double a = fabs(x);
        c.a = (a != a) ? 0.0 : a;
        c.s = 0.0;
        if (i == 0) c.v = (x != x) ? pinf : x;
        else c.v = (a != a) ? ninf : a;
        // a NaN candidate (ninf) must still lose to a real -inf seed on index order only
        best = key_better(best, c);
    }
    for (int o = 16; o > 0; o >>= 1) best = key_better(best, key_shfl_xor(best, o));
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) s_k[w] = best;
    __syncthreads();
    if (w == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        if (l < nw) best = s_k[l];
        else { best.v = ninf; best.i = 0x7fffffffffffffffLL; best.a = 0.0; best.s = 0.0; }
        for (int o = 16; o > 0; o >>= 1) best = key_better(best, key_shfl_xor(best, o));
        if (l == 0) {
            PairPeak p = cleared_peak();
            p.raw_index = best.i;
            p.peak = rp[best.i];
            p.second = best.s;
            p.resolved = 1;
            peaks[blockIdx.x] = p;
        }
    }
}

// The windowed twin (audiosync_cuda_set_lag_window): only the indices `win` allows are read, and
// i == 0 is the seed only when it is one of them.  A NaN candidate (ninf) still beats the sentinel
// on index order, so when no allowed value is a number the lowest allowed index is the answer with
// its NaN value, as a NaN seed is.  The rest is argmax_f64_kernel's (kept apart so that its code is
// unchanged).
static __global__ void __launch_bounds__(1024)
argmax_f64_window_kernel(const double* __restrict__ r, long long N, long long pitch, PairPeak* __restrict__ peaks,
                         RawWindow win)
{
    (void)N;
    __shared__ KeyF64 s_k[32];
    const double* rp = r + (size_t)blockIdx.x * (size_t)pitch;
    const double ninf = -INFINITY, pinf = INFINITY;
    KeyF64 best; best.v = ninf; best.i = 0x7fffffffffffffffLL; best.a = 0.0; best.s = 0.0;
    for (int g = 0; g < 2; g++) {
        const long long beg = g ? win.lo1 : win.lo0;
        const long long end = beg + (g ? win.n1 : win.n0);
        for (long long i = beg + threadIdx.x; i < end; i += blockDim.x) {
            const double x = rp[i];
            KeyF64 c;
            c.i = i;
            const double a = fabs(x);
            c.a = (a != a) ? 0.0 : a;
            c.s = 0.0;
            if (i == 0) c.v = (x != x) ? pinf : x;
            else c.v = (a != a) ? ninf : a;
            best = key_better(best, c);
        }
    }
    for (int o = 16; o > 0; o >>= 1) best = key_better(best, key_shfl_xor(best, o));
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) s_k[w] = best;
    __syncthreads();
    if (w == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        if (l < nw) best = s_k[l];
        else { best.v = ninf; best.i = 0x7fffffffffffffffLL; best.a = 0.0; best.s = 0.0; }
        for (int o = 16; o > 0; o >>= 1) best = key_better(best, key_shfl_xor(best, o));
        if (l == 0) {
            PairPeak p = cleared_peak();
            p.raw_index = best.i;
            p.peak = rp[best.i];
            p.second = best.s;
            p.resolved = 1;
            peaks[blockIdx.x] = p;
        }
    }
}

// The runner-up twin (audiosync_cuda_xcorr_runner_up): the window kernel's rule over pair i's runner-up
// set, at most three ranges; an empty set writes nothing (the runner-up Pearson step reports it).
static __global__ void __launch_bounds__(1024)
argmax_f64_runner_up_kernel(const double* __restrict__ r, long long pitch, PairPeak* __restrict__ peaks, RunnerUp ru)
{
    const PairWindow win = ru.window(blockIdx.x);
    if (win.empty()) return;
    __shared__ KeyF64 s_k[32];
    const double* rp = r + (size_t)blockIdx.x * (size_t)pitch;
    const double ninf = -INFINITY, pinf = INFINITY;
    KeyF64 best; best.v = ninf; best.i = 0x7fffffffffffffffLL; best.a = 0.0; best.s = 0.0;
    for (int g = 0; g < 3; g++) {
        const long long beg = g == 0 ? win.lo0 : g == 1 ? win.lo1 : win.lo2;
        const long long end = beg + (g == 0 ? win.n0 : g == 1 ? win.n1 : win.n2);
        for (long long i = beg + threadIdx.x; i < end; i += blockDim.x) {
            const double x = rp[i];
            KeyF64 c;
            c.i = i;
            const double a = fabs(x);
            c.a = (a != a) ? 0.0 : a;
            c.s = 0.0;
            if (i == 0) c.v = (x != x) ? pinf : x;
            else c.v = (a != a) ? ninf : a;
            best = key_better(best, c);
        }
    }
    for (int o = 16; o > 0; o >>= 1) best = key_better(best, key_shfl_xor(best, o));
    const int w = threadIdx.x >> 5, l = threadIdx.x & 31;
    if (l == 0) s_k[w] = best;
    __syncthreads();
    if (w == 0) {
        const int nw = (blockDim.x + 31) >> 5;
        if (l < nw) best = s_k[l];
        else { best.v = ninf; best.i = 0x7fffffffffffffffLL; best.a = 0.0; best.s = 0.0; }
        for (int o = 16; o > 0; o >>= 1) best = key_better(best, key_shfl_xor(best, o));
        if (l == 0) {
            PairPeak p = cleared_peak();
            p.raw_index = best.i;
            p.peak = rp[best.i];
            p.second = best.s;
            p.resolved = 1;
            peaks[blockIdx.x] = p;
        }
    }
}

// ---------------------------------------------------------------------------
// Pearson coefficient of the aligned windows (reference
// src/cross_correlation.c:74-116 on the windows of :256-271).
//
// One pass over the data with fp64 accumulators of the PIVOT-SHIFTED values
// dx = x - px, dy = y - py, where the pivots are the mean of 32 evenly spaced
// window samples (identical in every CTA of the pair): the shift removes the
// cancellation of the textbook one-pass formula without a second read of the
// window.  All five sums use one fixed reduction tree, so identical windows
// give cov == varx == vary bit for bit and the quotient is exactly +-1.0, as
// the reference's two-pass form does (tests/test_pearson_coefficient.c).
//
//   grid = (n_chunks, n_pairs), block = 256; chunk c covers window elements
//   [c * PEARSON_CHUNK, (c + 1) * PEARSON_CHUNK).
// ---------------------------------------------------------------------------
constexpr int PEARSON_THREADS = 256;
constexpr int PEARSON_PER_THREAD = 64;                       // window elements per thread and chunk
constexpr int PEARSON_CHUNK = PEARSON_THREADS * PEARSON_PER_THREAD;   // 16384 (stand-alone kernel)

struct PearsonPartial { double sx, sy, sxx, syy, sxy; };

// Shared scratch of one Pearson CTA.
template <int NTP>
struct PearsonShared {
    double piv[2];
    double red[NTP / 32][5];
    int last;
};

// Finishes one pair from the summed statistics (thread 0 of the finishing CTA).
// px, py: the pivots the sums were shifted by (sum x^2 = sxx + 2 px sx + n px^2).
// PHAT: the peak is that of the whitened correlation, and ncc = peak / N is its phase coherence
// (the window energies have no meaning under whitening).
template <bool PHAT>
__device__ __forceinline__ void pearson_finish(const PearsonPartial& s, const Window& w, long long raw,
                                               double peak, double second, double px, double py, long long L,
                                               audiosync_cuda_result* __restrict__ out)
{
    // n == 0 -> 0/0 = NaN, like the reference's empty pointer range.
    const double n = (double)w.n;
    const double cov = s.sxy - s.sx * s.sy / n;
    const double vx = s.sxx - s.sx * s.sx / n;
    const double vy = s.syy - s.sy * s.sy / n;
    const double coef = cov / sqrt(vx * vy);
    audiosync_cuda_result r;
    r.lag = w.lag;
    r.coef = coef;
    r.peak = peak;
    r.ret = (coef != coef) ? -1 : 0;                       // src/cross_correlation.c:276
    r.success = (r.ret == 0 && coef >= 0.95) ? 1 : 0;       // src/audiosync.c:254
    r.raw_index = raw;
    r.second = second;
    // peak quality (SURVEY 8f rank 4): margin of the peak over the second peak, and the peak
    // normalised by the energies of the two windows (unshifted sums of squares)
    const double ap = fabs(peak);
    r.margin = ap > 0.0 ? (ap - second) / ap : (ap == 0.0 ? 0.0 : peak);   // NaN peak -> NaN
    if constexpr (PHAT) {
        r.ncc = peak / (2.0 * (double)L);
    } else {
        const double ex = s.sxx + 2.0 * px * s.sx + n * px * px;
        const double ey = s.syy + 2.0 * py * s.sy + n * py * py;
        r.ncc = peak / (2.0 * (double)L * sqrt(ex * ey));
    }
    *out = r;
}

// One CTA of NTP threads: chunk `chunk` (NTP * 64 window elements) of pair `pair`.  The last
// CTA of a pair to finish (ticket counter, self-resetting) sums the chunk partials in a fixed
// order and writes the result record, so the whole Pearson step needs no second launch.
// Every thread of the CTA must call it (barriers inside).
// WIDE: fp64 arithmetic on the widened inputs (in_real) whatever T is.  T = float with WIDE is the
// path of host-narrowed batches whose floats are the exact images of the caller's doubles, T =
// int16_t that of 16-bit PCM (s * 2^-15, exact): element for element the same operations as
// T = double, so the record is the f64 call's on those doubles bit for bit.  Only fp32 inputs have
// the fp32 path.
template <typename T, int NTP, bool WIDE = !std::is_same<T, float>::value, bool PHAT = false>
__device__ __forceinline__ void pearson_block(
    const T* __restrict__ sources, const T* __restrict__ samples,
    long long src_pitch, long long smp_pitch, long long L,
    const PairPeak* __restrict__ peaks, long long explicit_n, double peak_scale,
    PearsonPartial* __restrict__ partials, unsigned int* __restrict__ tickets,
    int n_chunks, audiosync_cuda_result* __restrict__ results,
    int pair, int chunk, int t, PearsonShared<NTP>& sh)
{
    Window w;
    long long raw = 0;
    double peak = 0.0, second = 0.0;
    if (peaks == nullptr) {           // explicit window: whole arrays of length explicit_n
        w.lag = 0; w.xoff = 0; w.yoff = 0; w.n = explicit_n;
    } else {
        const PairPeak p = peaks[pair];
        raw = p.resolved ? p.raw_index : (long long)argmax_key_index(p.key);
        peak = p.resolved ? p.peak : (double)argmax_key_value(p.key);
        second = p.resolved ? p.second : (double)pair_second(p);
        // the transform's own scale -> the reference's (FFTW c2r: x N); powers of two for the static plans
        peak *= peak_scale;
        second *= peak_scale;
        w = fold_index(raw, L);
    }
    const T* __restrict__ x = sources + (size_t)pair * (size_t)src_pitch + w.xoff;
    const T* __restrict__ y = samples + (size_t)pair * (size_t)smp_pitch + w.yoff;

    PearsonPartial acc = {0.0, 0.0, 0.0, 0.0, 0.0};
    const long long lo = (long long)chunk * (NTP * PEARSON_PER_THREAD);
    if (lo < w.n) {
        if (t < 32) {
            long long k = ((long long)t * w.n) >> 5;
            double px = in_real<double>(x[k]), py = in_real<double>(y[k]);
            for (int o = 16; o > 0; o >>= 1) {
                px += __shfl_xor_sync(0xffffffffu, px, o);
                py += __shfl_xor_sync(0xffffffffu, py, o);
            }
            if (t == 0) { sh.piv[0] = px * (1.0 / 32.0); sh.piv[1] = py * (1.0 / 32.0); }
        }
        __syncthreads();
        const double px = sh.piv[0], py = sh.piv[1];
        long long hi = lo + (NTP * PEARSON_PER_THREAD);
        if (hi > w.n) hi = w.n;
        if constexpr (!WIDE) {
            // fp32 inputs: shifted values and products in fp32, 16 elements per thread and
            // iteration summed in fp32 (every term is < 4, so the partial is good to ~1e-7
            // relative), then folded into the fp64 accumulators -- 5 conversions per 16
            // elements instead of 2 per element.  The three product sums share one
            // instruction sequence, so identical windows still give cov == varx == vary.
            const float pxf = (float)px, pyf = (float)py;
            const bool xv = (reinterpret_cast<uintptr_t>(x + lo) & 15u) == 0;
            const bool yv = (reinterpret_cast<uintptr_t>(y + lo) & 15u) == 0;
            constexpr int VPT = 4;                                   // float4 groups per thread and iteration
            constexpr long long STEP = 4LL * NTP;        // elements per group row
            auto load4 = [](const float* __restrict__ p, bool vec) -> float4 {
                if (vec) return __ldg(reinterpret_cast<const float4*>(p));
                return make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
            };
            long long i = lo + 4LL * t;
            for (; i + (VPT - 1) * STEP + 3 < hi; i += VPT * STEP) {
                float4 xq[VPT], yq[VPT];
#pragma unroll
                for (int u = 0; u < VPT; u++) { xq[u] = load4(x + i + u * STEP, xv); yq[u] = load4(y + i + u * STEP, yv); }
                float fsx = 0.f, fsy = 0.f, fsxx = 0.f, fsyy = 0.f, fsxy = 0.f;
#pragma unroll
                for (int u = 0; u < VPT; u++) {
                    const float dx[4] = {xq[u].x - pxf, xq[u].y - pxf, xq[u].z - pxf, xq[u].w - pxf};
                    const float dy[4] = {yq[u].x - pyf, yq[u].y - pyf, yq[u].z - pyf, yq[u].w - pyf};
#pragma unroll
                    for (int e = 0; e < 4; e++) {
                        fsx += dx[e]; fsy += dy[e];
                        fsxx = fmaf(dx[e], dx[e], fsxx); fsyy = fmaf(dy[e], dy[e], fsyy); fsxy = fmaf(dx[e], dy[e], fsxy);
                    }
                }
                acc.sx += (double)fsx; acc.sy += (double)fsy;
                acc.sxx += (double)fsxx; acc.syy += (double)fsyy; acc.sxy += (double)fsxy;
            }
            // remainder of the chunk (window tail): element-wise, same fp32 shift
            for (long long k = i; k < hi; k += STEP) {
                for (int e = 0; e < 4 && k + e < hi; e++) {
                    const float dx = (float)x[k + e] - pxf, dy = (float)y[k + e] - pyf;
                    acc.sx += (double)dx; acc.sy += (double)dy;
                    acc.sxx += (double)(dx * dx); acc.syy += (double)(dy * dy); acc.sxy += (double)(dx * dy);
                }
            }
        } else {
            constexpr int UN = 8;
            long long i = lo + t;
            for (; i + (UN - 1) * NTP < hi; i += UN * NTP) {
                T xv[UN], yv[UN];
#pragma unroll
                for (int u = 0; u < UN; u++) { xv[u] = x[i + u * NTP]; yv[u] = y[i + u * NTP]; }
#pragma unroll
                for (int u = 0; u < UN; u++) {
                    const double dx = in_real<double>(xv[u]) - px, dy = in_real<double>(yv[u]) - py;
                    acc.sx += dx; acc.sy += dy;
                    acc.sxx = fma(dx, dx, acc.sxx); acc.syy = fma(dy, dy, acc.syy); acc.sxy = fma(dx, dy, acc.sxy);
                }
            }
            for (; i < hi; i += NTP) {
                const double dx = in_real<double>(x[i]) - px, dy = in_real<double>(y[i]) - py;
                acc.sx += dx; acc.sy += dy;
                acc.sxx = fma(dx, dx, acc.sxx); acc.syy = fma(dy, dy, acc.syy); acc.sxy = fma(dx, dy, acc.sxy);
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) {
        acc.sx += __shfl_xor_sync(0xffffffffu, acc.sx, o);
        acc.sy += __shfl_xor_sync(0xffffffffu, acc.sy, o);
        acc.sxx += __shfl_xor_sync(0xffffffffu, acc.sxx, o);
        acc.syy += __shfl_xor_sync(0xffffffffu, acc.syy, o);
        acc.sxy += __shfl_xor_sync(0xffffffffu, acc.sxy, o);
    }
    const int wid = t >> 5, lane = t & 31;
    if (lane == 0) {
        sh.red[wid][0] = acc.sx; sh.red[wid][1] = acc.sy; sh.red[wid][2] = acc.sxx;
        sh.red[wid][3] = acc.syy; sh.red[wid][4] = acc.sxy;
    }
    __syncthreads();
    if (t == 0) {
        PearsonPartial o = {0.0, 0.0, 0.0, 0.0, 0.0};
        for (int k = 0; k < NTP / 32; k++) {
            o.sx += sh.red[k][0]; o.sy += sh.red[k][1]; o.sxx += sh.red[k][2];
            o.syy += sh.red[k][3]; o.sxy += sh.red[k][4];
        }
        partials[(size_t)pair * n_chunks + chunk] = o;
        __threadfence();
        const unsigned int ticket = atomicAdd(&tickets[pair], 1u);
        sh.last = (ticket == (unsigned int)(n_chunks - 1)) ? 1 : 0;
    }
    __syncthreads();
    if (sh.last && t < 32) {
        __threadfence();
        // lane l sums chunks l, l+32, ... in ascending order; then a fixed xor tree
        PearsonPartial s = {0.0, 0.0, 0.0, 0.0, 0.0};
        const double* base = reinterpret_cast<const double*>(partials + (size_t)pair * n_chunks);
        for (int c = t; c < n_chunks; c += 32) {
            s.sx += __ldcg(base + 5 * c + 0); s.sy += __ldcg(base + 5 * c + 1);
            s.sxx += __ldcg(base + 5 * c + 2); s.syy += __ldcg(base + 5 * c + 3);
            s.sxy += __ldcg(base + 5 * c + 4);
        }
        for (int o = 16; o > 0; o >>= 1) {
            s.sx += __shfl_xor_sync(0xffffffffu, s.sx, o);
            s.sy += __shfl_xor_sync(0xffffffffu, s.sy, o);
            s.sxx += __shfl_xor_sync(0xffffffffu, s.sxx, o);
            s.syy += __shfl_xor_sync(0xffffffffu, s.syy, o);
            s.sxy += __shfl_xor_sync(0xffffffffu, s.sxy, o);
        }
        // the pivots again (this CTA's chunk may lie beyond the window and never have formed them);
        // fp32 inputs were shifted by the pivots rounded to fp32
        double px = 0.0, py = 0.0;
        if (w.n > 0) {
            const long long k = ((long long)t * w.n) >> 5;
            px = in_real<double>(x[k]); py = in_real<double>(y[k]);
            for (int o = 16; o > 0; o >>= 1) {
                px += __shfl_xor_sync(0xffffffffu, px, o);
                py += __shfl_xor_sync(0xffffffffu, py, o);
            }
            px *= (1.0 / 32.0); py *= (1.0 / 32.0);
            if constexpr (!WIDE) { px = (double)(float)px; py = (double)(float)py; }
        }
        if (t == 0) {
            pearson_finish<PHAT>(s, w, raw, peak, second, px, py, L, results + pair);
            tickets[pair] = 0u;       // ready for the next wave
        }
    }
}

// grid = (n_chunks, n_pairs), block = 256.  PHAT: records of a PHAT-weighted correlation (ncc rule).
template <typename T, bool WIDE = !std::is_same<T, float>::value, bool PHAT = false>
__global__ void __launch_bounds__(PEARSON_THREADS)
pearson_kernel(const T* __restrict__ sources, const T* __restrict__ samples,
               long long src_pitch, long long smp_pitch, long long L,
               const PairPeak* __restrict__ peaks, long long explicit_n, double peak_scale,
               PearsonPartial* __restrict__ partials, unsigned int* __restrict__ tickets,
               int n_chunks, audiosync_cuda_result* __restrict__ results)
{
    __shared__ PearsonShared<PEARSON_THREADS> sh;
    pdl_prologue();
    pearson_block<T, PEARSON_THREADS, WIDE, PHAT>(sources, samples, src_pitch, smp_pitch, L, peaks, explicit_n, peak_scale, partials,
                                      tickets, n_chunks, results, (int)blockIdx.y, (int)blockIdx.x,
                                      (int)threadIdx.x, sh);
}

// The record of a pair whose runner-up set is empty (audiosync_cuda_xcorr_runner_up).
__host__ __device__ __forceinline__ audiosync_cuda_result no_runner_up() {
    audiosync_cuda_result r;
    r.lag = 0; r.coef = NAN; r.peak = 0.0; r.ret = -1; r.success = 0;
    r.raw_index = -1; r.second = 0.0; r.margin = 0.0; r.ncc = NAN;
    return r;
}

// The runner-up twin of pearson_kernel: pair i's record from the second search's peaks, or
// no_runner_up() when its runner-up set is empty (every CTA of that pair returns at once, so its
// ticket counter is not touched).
template <typename T, bool WIDE = !std::is_same<T, float>::value, bool PHAT = false>
__global__ void __launch_bounds__(PEARSON_THREADS)
pearson_runner_up_kernel(const T* __restrict__ sources, const T* __restrict__ samples,
                         long long src_pitch, long long smp_pitch, long long L,
                         const PairPeak* __restrict__ peaks, RunnerUp ru, double peak_scale,
                         PearsonPartial* __restrict__ partials, unsigned int* __restrict__ tickets,
                         int n_chunks, audiosync_cuda_result* __restrict__ results)
{
    __shared__ PearsonShared<PEARSON_THREADS> sh;
    pdl_prologue();
    if (ru.window(blockIdx.y).empty()) {
        if (blockIdx.x == 0 && threadIdx.x == 0) results[blockIdx.y] = no_runner_up();
        return;
    }
    pearson_block<T, PEARSON_THREADS, WIDE, PHAT>(sources, samples, src_pitch, smp_pitch, L, peaks, 0LL, peak_scale, partials,
                                      tickets, n_chunks, results, (int)blockIdx.y, (int)blockIdx.x,
                                      (int)threadIdx.x, sh);
}

}  // namespace asc
