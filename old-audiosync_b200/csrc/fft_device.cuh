// fft_device.cuh -- building blocks of the sm_100a transform kernels:
// compile-time twiddle constants, in-register DFT butterflies (radix 2/3/4/5
// by hand, composites by prime-factor / Cooley-Tukey recursion with every
// index resolved at compile time), radix lists and digit-reversal maps.
//
// Everything here is __host__ __device__ so that tests/emu can execute the
// exact kernel bodies on the CPU (phase by phase) and compare them with the
// oracle before any GPU time is spent.
#pragma once

#include <cuda.h>            // CUtensorMap (the descriptor type only; no driver call is made from here)
#include <cuda_runtime.h>
#include <stdint.h>

#include <string.h>

#include <type_traits>
#include <utility>

#define ASC_HD __host__ __device__ __forceinline__

namespace asc {

typedef float2 cplx;

ASC_HD cplx cmake(float a, float b) { cplx r; r.x = a; r.y = b; return r; }

// Complex arithmetic.  On the device every operation is written with the
// sm_100 packed-fp32 instructions (FADD2 / FMUL2 / FFMA2: one issue slot for
// both halves of a float2 register pair).  ptxas folds the swaps and per-half
// sign flips below into operand modifiers (R.F32x2.LO_HI, .NP, scalar
// broadcast R.F32), so a complex add is one instruction and a complex multiply
// two.  The host versions (CPU emulator) compute the same values with scalar
// fmaf in the same association order.
#if defined(__CUDA_ARCH__)
#define ASC_PACKED 1
#else
#define ASC_PACKED 0
#endif
ASC_HD cplx cadd(cplx a, cplx b) {
#if ASC_PACKED
    return __fadd2_rn(a, b);
#else
    return cmake(a.x + b.x, a.y + b.y);
#endif
}
ASC_HD cplx csub(cplx a, cplx b) {
#if ASC_PACKED
    return __fadd2_rn(a, cmake(-b.x, -b.y));
#else
    return cmake(a.x - b.x, a.y - b.y);
#endif
}
ASC_HD cplx cscale(cplx a, float s) {
#if ASC_PACKED
    return __fmul2_rn(a, cmake(s, s));
#else
    return cmake(a.x * s, a.y * s);
#endif
}
// a + s * b
ASC_HD cplx caxpy(float s, cplx b, cplx a) {
#if ASC_PACKED
    return __ffma2_rn(b, cmake(s, s), a);
#else
    return cmake(fmaf(b.x, s, a.x), fmaf(b.y, s, a.y));
#endif
}
// a * b = a * b.x + (i a) * b.y, evaluated as fma(a, b.x, (-t.x, t.y)) with t = (a.y, a.x) * b.y
ASC_HD cplx cmul(cplx a, cplx b) {
#if ASC_PACKED
    const cplx t = __fmul2_rn(cmake(a.y, a.x), cmake(b.y, b.y));
    return __ffma2_rn(a, cmake(b.x, b.x), cmake(-t.x, t.y));
#else
    return cmake(fmaf(a.x, b.x, -(a.y * b.y)), fmaf(a.y, b.x, a.x * b.y));
#endif
}
// a * conj(b)
ASC_HD cplx cmulc(cplx a, cplx b) {
#if ASC_PACKED
    const cplx t = __fmul2_rn(cmake(a.y, a.x), cmake(b.y, b.y));
    return __ffma2_rn(a, cmake(b.x, b.x), cmake(t.x, -t.y));
#else
    return cmake(fmaf(a.x, b.x, a.y * b.y), fmaf(a.y, b.x, -(a.x * b.y)));
#endif
}
// a + i*b, a - i*b
ASC_HD cplx cadd_i(cplx a, cplx b) {
#if ASC_PACKED
    return __fadd2_rn(a, cmake(-b.y, b.x));
#else
    return cmake(a.x - b.y, a.y + b.x);
#endif
}
ASC_HD cplx csub_i(cplx a, cplx b) {
#if ASC_PACKED
    return __fadd2_rn(a, cmake(b.y, -b.x));
#else
    return cmake(a.x + b.y, a.y - b.x);
#endif
}
// a + s * (i*b), a - s * (i*b)
ASC_HD cplx caxpy_i(float s, cplx b, cplx a) {
#if ASC_PACKED
    return __ffma2_rn(cmake(-b.y, b.x), cmake(s, s), a);
#else
    return cmake(fmaf(-b.y, s, a.x), fmaf(b.x, s, a.y));
#endif
}
ASC_HD cplx caxmy_i(float s, cplx b, cplx a) {
#if ASC_PACKED
    return __ffma2_rn(cmake(b.y, -b.x), cmake(s, s), a);
#else
    return cmake(fmaf(b.y, s, a.x), fmaf(-b.x, s, a.y));
#endif
}
// v * (wr + i wi) with compile-time-known wr, wi (immediates in the SASS)
ASC_HD cplx cmul_const(cplx v, float wr, float wi) {
#if ASC_PACKED
    return __ffma2_rn(cmake(-v.y, v.x), cmake(wi, wi), __fmul2_rn(v, cmake(wr, wr)));
#else
    return cmake(fmaf(-v.y, wi, v.x * wr), fmaf(v.x, wi, v.y * wr));
#endif
}
// a + conj(b), a - conj(b)
ASC_HD cplx cconj_add(cplx a, cplx b) {
#if ASC_PACKED
    return __fadd2_rn(a, cmake(b.x, -b.y));
#else
    return cmake(a.x + b.x, a.y - b.y);
#endif
}
ASC_HD cplx cconj_sub(cplx a, cplx b) {
#if ASC_PACKED
    return __fadd2_rn(a, cmake(-b.x, b.y));
#else
    return cmake(a.x - b.x, a.y + b.y);
#endif
}
// acc + a * conj(b)
ASC_HD cplx cmulc_acc(cplx a, cplx b, cplx acc) {
#if ASC_PACKED
    const cplx t = __ffma2_rn(cmake(a.y, -a.x), cmake(b.y, b.y), acc);
    return __ffma2_rn(a, cmake(b.x, b.x), t);
#else
    return cmake(fmaf(a.x, b.x, fmaf(a.y, b.y, acc.x)), fmaf(a.y, b.x, fmaf(-a.x, b.y, acc.y)));
#endif
}
// acc - a * conj(b)
ASC_HD cplx cmulc_nacc(cplx a, cplx b, cplx acc) {
#if ASC_PACKED
    const cplx t = __ffma2_rn(cmake(-a.y, a.x), cmake(b.y, b.y), acc);
    return __ffma2_rn(a, cmake(-b.x, -b.x), t);
#else
    return cmake(fmaf(-a.x, b.x, fmaf(-a.y, b.y, acc.x)), fmaf(-a.y, b.x, fmaf(a.x, b.y, acc.y)));
#endif
}
// multiply by +i / -i
ASC_HD cplx cmul_pi(cplx a) { return cmake(-a.y, a.x); }
ASC_HD cplx cmul_ni(cplx a) { return cmake(a.y, -a.x); }

// ---- the same operations on double2 (fp64-arithmetic validation mode and nothing else: plain
// fma / add, no packed forms exist).  Selected by overload; scalar_of<C> names the real type.
typedef double2 cplxd;
ASC_HD cplxd cmake(double a, double b) { cplxd r; r.x = a; r.y = b; return r; }
ASC_HD cplxd cadd(cplxd a, cplxd b) { return cmake(a.x + b.x, a.y + b.y); }
ASC_HD cplxd csub(cplxd a, cplxd b) { return cmake(a.x - b.x, a.y - b.y); }
ASC_HD cplxd cscale(cplxd a, double s) { return cmake(a.x * s, a.y * s); }
ASC_HD cplxd caxpy(double s, cplxd b, cplxd a) { return cmake(fma(b.x, s, a.x), fma(b.y, s, a.y)); }
ASC_HD cplxd cmul(cplxd a, cplxd b) { return cmake(fma(a.x, b.x, -(a.y * b.y)), fma(a.y, b.x, a.x * b.y)); }
ASC_HD cplxd cmulc(cplxd a, cplxd b) { return cmake(fma(a.x, b.x, a.y * b.y), fma(a.y, b.x, -(a.x * b.y))); }
ASC_HD cplxd cadd_i(cplxd a, cplxd b) { return cmake(a.x - b.y, a.y + b.x); }
ASC_HD cplxd csub_i(cplxd a, cplxd b) { return cmake(a.x + b.y, a.y - b.x); }
ASC_HD cplxd caxpy_i(double s, cplxd b, cplxd a) { return cmake(fma(-b.y, s, a.x), fma(b.x, s, a.y)); }
ASC_HD cplxd caxmy_i(double s, cplxd b, cplxd a) { return cmake(fma(b.y, s, a.x), fma(-b.x, s, a.y)); }
ASC_HD cplxd cmul_const(cplxd v, double wr, double wi) { return cmake(fma(-v.y, wi, v.x * wr), fma(v.x, wi, v.y * wr)); }
ASC_HD cplxd cconj_add(cplxd a, cplxd b) { return cmake(a.x + b.x, a.y - b.y); }
ASC_HD cplxd cconj_sub(cplxd a, cplxd b) { return cmake(a.x - b.x, a.y + b.y); }
ASC_HD cplxd cmulc_acc(cplxd a, cplxd b, cplxd acc) {
    return cmake(fma(a.x, b.x, fma(a.y, b.y, acc.x)), fma(a.y, b.x, fma(-a.x, b.y, acc.y)));
}
ASC_HD cplxd cmulc_nacc(cplxd a, cplxd b, cplxd acc) {
    return cmake(fma(-a.x, b.x, fma(-a.y, b.y, acc.x)), fma(-a.y, b.x, fma(a.x, b.y, acc.y)));
}
ASC_HD cplxd cmul_pi(cplxd a) { return cmake(-a.y, a.x); }
ASC_HD cplxd cmul_ni(cplxd a) { return cmake(a.y, -a.x); }

template <class C> struct scalar_of;
template <> struct scalar_of<cplx> { typedef float type; };
template <> struct scalar_of<cplxd> { typedef double type; };

template <typename T>
ASC_HD T ldg(const T* p) {
#if defined(__CUDA_ARCH__)
    return __ldg(p);
#else
    return *p;
#endif
}

// ------------------------------------------------------- asynchronous staging
// Global -> shared copies that bypass the register file (LDGSTS / cp.async,
// 16 bytes per thread, L1 bypass) and the shared -> global bulk store of the
// TMA unit (cp.async.bulk, one instruction for a whole row).  The host versions
// (CPU emulator) are plain copies.
ASC_HD void cp_async16(void* smem_dst, const void* gmem_src) {
#if defined(__CUDA_ARCH__)
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(sa), "l"(gmem_src) : "memory");
#else
    memcpy(smem_dst, gmem_src, 16);
#endif
}
// the same for 8-byte elements (rows with an odd padding pitch are only 8-byte aligned)
ASC_HD void cp_async8(void* smem_dst, const void* gmem_src) {
#if defined(__CUDA_ARCH__)
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(sa), "l"(gmem_src) : "memory");
#else
    memcpy(smem_dst, gmem_src, 8);
#endif
}
ASC_HD void cp_async_wait_all() {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.wait_all;" ::: "memory");
#endif
}
// Makes this thread's earlier shared-memory writes visible to the async proxy
// (required between st.shared and a bulk store that reads the same bytes).
ASC_HD void fence_async_proxy() {
#if defined(__CUDA_ARCH__)
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
#endif
}
// One thread: shared -> global bulk copy, bytes % 16 == 0, both 16-byte aligned.
ASC_HD void bulk_store(void* gmem_dst, const void* smem_src, unsigned bytes) {
#if defined(__CUDA_ARCH__)
    const unsigned sa = (unsigned)__cvta_generic_to_shared(smem_src);
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(sa), "r"(bytes)
                 : "memory");
#else
    memcpy(gmem_dst, smem_src, bytes);
#endif
}
// Same thread: commit, then wait until the source bytes have been read out of
// shared memory (the CTA may exit / reuse the buffer; global visibility follows
// at kernel completion).
ASC_HD void bulk_store_commit_and_drain() {
#if defined(__CUDA_ARCH__)
    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
    asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
#endif
}

// Global -> shared bulk copies of the TMA unit, completion counted in bytes on an mbarrier
// (8 bytes of shared memory).  One thread: init, expect the byte total, issue the copies,
// wait, invalidate; the CTA barrier that follows publishes the data to the other threads.
// The copies do not pass through the LSU pipe (LDGSTS costs 4 issue + 4 shared-memory
// cycles per 512 bytes there).  Host versions (CPU emulator): plain copies.
ASC_HD void mbar_init(void* mbar, unsigned count) {
#if defined(__CUDA_ARCH__)
    const unsigned a = (unsigned)__cvta_generic_to_shared(mbar);
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(a), "r"(count) : "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // the async proxy sees the init
#else
    (void)mbar; (void)count;
#endif
}
ASC_HD void mbar_expect_tx(void* mbar, unsigned bytes) {
#if defined(__CUDA_ARCH__)
    const unsigned a = (unsigned)__cvta_generic_to_shared(mbar);
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(a), "r"(bytes) : "memory");
#else
    (void)mbar; (void)bytes;
#endif
}
// bytes % 16 == 0, both addresses 16-byte aligned
ASC_HD void bulk_load(void* smem_dst, const void* gmem_src, unsigned bytes, void* mbar) {
#if defined(__CUDA_ARCH__)
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    const unsigned a = (unsigned)__cvta_generic_to_shared(mbar);
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(d), "l"(gmem_src), "r"(bytes), "r"(a) : "memory");
#else
    (void)mbar;
    memcpy(smem_dst, gmem_src, bytes);
#endif
}
ASC_HD void mbar_wait(void* mbar, unsigned parity) {
#if defined(__CUDA_ARCH__)
    const unsigned a = (unsigned)__cvta_generic_to_shared(mbar);
    unsigned ok;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(ok) : "r"(a), "r"(parity) : "memory");
    } while (!ok);
#else
    (void)mbar; (void)parity;
#endif
}
// One box of a 3-D tiled tensor map (inner extent 128 bytes = one tile row, `rows` rows, one
// slice) into shared memory: [rows][128 bytes], the layout of the column tiles.  Coordinates
// are (float index in the row, row, slice).  Host version: the same rows copied from `raw`
// (pointer to the first row's 128 bytes) with `row_pitch_bytes` between rows.
ASC_HD void tma_load_rows(void* smem_dst, const CUtensorMap* tm, int c0, int c1, int c2, void* mbar,
                          const void* raw, size_t row_pitch_bytes, int rows) {
#if defined(__CUDA_ARCH__)
    (void)raw; (void)row_pitch_bytes; (void)rows;
    const unsigned d = (unsigned)__cvta_generic_to_shared(smem_dst);
    const unsigned a = (unsigned)__cvta_generic_to_shared(mbar);
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes "
                 "[%0], [%1, {%2, %3, %4}], [%5];"
                 ::"r"(d), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(a) : "memory");
#else
    (void)tm; (void)c0; (void)c1; (void)c2; (void)mbar;
    for (int i = 0; i < rows; i++)
        memcpy(static_cast<char*>(smem_dst) + (size_t)i * 128, static_cast<const char*>(raw) + (size_t)i * row_pitch_bytes, 128);
#endif
}
// required before the 8 bytes are used as ordinary shared memory again
ASC_HD void mbar_inval(void* mbar) {
#if defined(__CUDA_ARCH__)
    const unsigned a = (unsigned)__cvta_generic_to_shared(mbar);
    asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(a) : "memory");
#else
    (void)mbar;
#endif
}

// Programmatic dependent launch: the stages of a wave are launched with
// cudaLaunchAttributeProgrammaticStreamSerialization, so the next stage's CTAs are scheduled
// (and parked here) while the last CTAs of this one still run; `wait` returns when the
// preceding grid has completed and its memory is visible.  Without the attribute both are no-ops.
ASC_HD void pdl_prologue() {
#if defined(__CUDA_ARCH__)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    asm volatile("griddepcontrol.wait;" ::: "memory");
#endif
}

// --------------------------------------------------------------- static_for
template <int I>
using IC = std::integral_constant<int, I>;

template <int B, int E, class F>
ASC_HD void static_for(F&& f) {
    if constexpr (B < E) {
        f(IC<B>{});
        static_for<B + 1, E>(static_cast<F&&>(f));
    }
}

// ------------------------------------------------- compile-time trigonometry
// cos/sin of 2*pi*num/den evaluated in constant expressions only (the results
// become immediates in the SASS).  Range-reduced to [0, pi/4] with integer
// arithmetic, then a Taylor series in double: error < 1e-16.
namespace ct {
constexpr double PI = 3.14159265358979323846264338327950288;

constexpr double sin_small(double x) {  // |x| <= pi/4
    double x2 = x * x, term = x, sum = x;
    for (int k = 1; k < 12; k++) {
        term *= -x2 / (double)((2 * k) * (2 * k + 1));
        sum += term;
    }
    return sum;
}
constexpr double cos_small(double x) {
    double x2 = x * x, term = 1.0, sum = 1.0;
    for (int k = 1; k < 12; k++) {
        term *= -x2 / (double)((2 * k - 1) * (2 * k));
        sum += term;
    }
    return sum;
}
struct cd { double re, im; };
// exp(+2*pi*i*num/den), num any integer, den > 0
constexpr cd unit(long long num, long long den) {
    long long a = num % den;
    if (a < 0) a += den;
    // quadrant q = floor(4a/den); remainder angle = 2*pi*(4a - q*den)/(4*den)
    long long q = (4 * a) / den;
    long long rnum = 4 * a - q * den;          // in [0, den)
    double c = 0.0, s = 0.0;
    if (2 * rnum <= den) {                     // angle <= pi/4
        double th = 2.0 * PI * (double)rnum / (4.0 * (double)den);
        c = cos_small(th); s = sin_small(th);
    } else {                                   // use the complement to pi/2
        double th = 2.0 * PI * (double)(den - rnum) / (4.0 * (double)den);
        c = sin_small(th); s = cos_small(th);
    }
    if (rnum == 0) { c = 1.0; s = 0.0; }
    switch (q) {
        case 0: return cd{c, s};
        case 1: return cd{-s, c};
        case 2: return cd{-c, -s};
        default: return cd{s, -c};
    }
}
constexpr int gcd(int a, int b) { return b == 0 ? a : gcd(b, a % b); }
constexpr int first_factor(int r) {
    // split composites so that coprime (prime-factor) splits are preferred
    // and the sub-transforms stay in the hand-written set {2,3,4,5}.
    if (r % 4 == 0 && r != 4) return 4;
    if (r % 2 == 0) return 2;
    if (r % 3 == 0) return 3;
    if (r % 5 == 0) return 5;
    return r;
}
}  // namespace ct

// Multiply v by exp(DIR * 2*pi*i * T / R) with the constant folded; exact
// cases (1, -1, +-i, the eighth roots) use adds only.
template <int T_, int R, int DIR, class C = cplx>
ASC_HD C mul_root(C v) {
    typedef typename scalar_of<C>::type real;
    constexpr int t = ((T_ % R) + R) % R;
    if constexpr (t == 0) {
        return v;
    } else if constexpr (2 * t == R) {
        return cmake(-v.x, -v.y);
    } else if constexpr (4 * t == R) {
        return DIR > 0 ? cmul_pi(v) : cmul_ni(v);
    } else if constexpr (4 * t == 3 * R) {
        return DIR > 0 ? cmul_ni(v) : cmul_pi(v);
    } else {
        constexpr ct::cd w = ct::unit((long long)DIR * t, R);
        constexpr real wr = (real)w.re, wi = (real)w.im;
        if constexpr (8 * t == R || 8 * t == 3 * R || 8 * t == 5 * R || 8 * t == 7 * R) {
            // |wr| == |wi| == sqrt(1/2): (sr + i si) v = sr v + si (i v), then one scale
            constexpr real h = (real)0.70710678118654752440;
            constexpr bool same = (wr > 0) == (wi > 0);
            const C u = same ? cadd_i(v, v) : csub_i(v, v);     // v +- i v
            return cscale(u, wr > 0 ? h : -h);
        } else {
            return cmul_const(v, wr, wi);
        }
    }
}

// ------------------------------------------------------ register butterflies
// dft_reg<R, DIR>(v): v[k] <- sum_n v[n] exp(DIR*2*pi*i*n*k/R), natural order
// in and out, all indices compile-time (v stays in registers).  C = cplx (packed fp32, the
// product) or cplxd (fp64 validation mode).
template <int R, int DIR, class C = cplx>
struct DftReg;

template <int DIR, class C>
struct DftReg<1, DIR, C> {
    static ASC_HD void run(C (&)[1]) {}
};

template <int DIR, class C>
struct DftReg<2, DIR, C> {
    static ASC_HD void run(C (&v)[2]) {
        C a = v[0], b = v[1];
        v[0] = cadd(a, b);
        v[1] = csub(a, b);
    }
};

template <int DIR, class C>
struct DftReg<3, DIR, C> {
    static ASC_HD void run(C (&v)[3]) {
        typedef typename scalar_of<C>::type real;
        constexpr real s60 = (real)((DIR > 0 ? 1.0 : -1.0) * 0.86602540378443864676);
        const C a = v[0], b = v[1], c = v[2];
        const C t1 = cadd(b, c);
        const C t2 = caxpy((real)-0.5, t1, a);
        const C d = csub(b, c);
        v[0] = cadd(a, t1);
        v[1] = caxpy_i(s60, d, t2);      // t2 + i s60 d
        v[2] = caxmy_i(s60, d, t2);      // t2 - i s60 d
    }
};

template <int DIR, class C>
struct DftReg<4, DIR, C> {
    static ASC_HD void run(C (&v)[4]) {
        const C s0 = cadd(v[0], v[2]), s1 = csub(v[0], v[2]);
        const C s2 = cadd(v[1], v[3]), s3 = csub(v[1], v[3]);
        v[0] = cadd(s0, s2);
        v[2] = csub(s0, s2);
        if constexpr (DIR > 0) { v[1] = cadd_i(s1, s3); v[3] = csub_i(s1, s3); }
        else { v[1] = csub_i(s1, s3); v[3] = cadd_i(s1, s3); }
    }
};

template <int DIR, class C>
struct DftReg<5, DIR, C> {
    static ASC_HD void run(C (&v)[5]) {
        typedef typename scalar_of<C>::type real;
        constexpr real c1 = (real)0.30901699437494742410;    // cos(2pi/5)
        constexpr real c2 = (real)-0.80901699437494742410;   // cos(4pi/5)
        constexpr double sg = DIR > 0 ? 1.0 : -1.0;
        constexpr real s1 = (real)(sg * 0.95105651629515357212);  // sin(2pi/5)
        constexpr real s2 = (real)(sg * 0.58778525229247312917);  // sin(4pi/5)
        const C x0 = v[0];
        const C a1 = cadd(v[1], v[4]), b1 = csub(v[1], v[4]);
        const C a2 = cadd(v[2], v[3]), b2 = csub(v[2], v[3]);
        const C p1 = caxpy(c2, a2, caxpy(c1, a1, x0));
        const C p2 = caxpy(c1, a2, caxpy(c2, a1, x0));
        const C u1 = caxpy(s2, b2, cscale(b1, s1));
        const C u2 = caxpy(-s1, b2, cscale(b1, s2));
        v[0] = cadd(cadd(x0, a1), a2);
        v[1] = cadd_i(p1, u1);
        v[4] = csub_i(p1, u1);
        v[2] = cadd_i(p2, u2);
        v[3] = csub_i(p2, u2);
    }
};

// Composite R = A * B.
//  gcd(A,B) == 1: prime-factor (Good-Thomas) map, no twiddles:
//      n = (B*n1 + A*n2) mod R,  k = the unique k with k%A == k1, k%B == k2.
//  otherwise: Cooley-Tukey, n = A*n2 + n1, k = B*k1 + k2, twiddle W_R^(n1*k2).
template <int R, int DIR, class C>
struct DftReg {
    static constexpr int A = ct::first_factor(R);
    static constexpr int B = R / A;
    static_assert(A > 1 && A < R, "unsupported radix (prime > 5)");
    static constexpr bool PFA = ct::gcd(A, B) == 1;

    static constexpr int crt(int k1, int k2) {
        for (int k = 0; k < R; k++)
            if (k % A == k1 && k % B == k2) return k;
        return -1;
    }

    static ASC_HD void run(C (&v)[R]) {
        C t[R];   // t[n1 * B + k2]
        static_for<0, A>([&](auto N1) {
            constexpr int n1 = decltype(N1)::value;
            C u[B];
            static_for<0, B>([&](auto N2) {
                constexpr int n2 = decltype(N2)::value;
                constexpr int src = PFA ? (B * n1 + A * n2) % R : (A * n2 + n1);
                u[n2] = v[src];
            });
            DftReg<B, DIR, C>::run(u);
            static_for<0, B>([&](auto K2) {
                constexpr int k2 = decltype(K2)::value;
                if constexpr (PFA) t[n1 * B + k2] = u[k2];
                else t[n1 * B + k2] = mul_root<n1 * k2, R, DIR, C>(u[k2]);
            });
        });
        static_for<0, B>([&](auto K2) {
            constexpr int k2 = decltype(K2)::value;
            C u[A];
            static_for<0, A>([&](auto N1) {
                constexpr int n1 = decltype(N1)::value;
                u[n1] = t[n1 * B + k2];
            });
            DftReg<A, DIR, C>::run(u);
            static_for<0, A>([&](auto K1) {
                constexpr int k1 = decltype(K1)::value;
                constexpr int dst = PFA ? crt(k1, k2) : (B * k1 + k2);
                v[dst] = u[k1];
            });
        });
    }
};

template <int R, int DIR, class C>
ASC_HD void dft_reg(C (&v)[R]) { DftReg<R, DIR, C>::run(v); }

// w[k] = exp(-2*pi*i*j*k/(S*R)) for k = 1..R-1 from the power-of-two table
// entries of one pass (tw points at the pass's table): k = 2^i is a load,
// any other k is the product w[hb(k)] * w[k - hb(k)] (at most 3 products deep
// for R <= 16, i.e. a few ulp).  Trades LSU wavefronts for FMA-pipe work.
// Fills w[k], k not a power of two, from the power-of-two entries already in w.
template <int R, class C = cplx>
ASC_HD void fill_twiddles(C (&w)[R]) {
    static_for<1, R>([&](auto K) {
        constexpr int k = decltype(K)::value;
        if constexpr ((k & (k - 1)) != 0) {
            constexpr int hb = (k >= 16) ? 16 : (k >= 8) ? 8 : (k >= 4) ? 4 : 2;
            w[k] = cmul(w[hb], w[k - hb]);
        }
    });
}

template <int R>
ASC_HD void pass_twiddles(const cplx* __restrict__ tw, int S, int j, cplx (&w)[R]) {
    static_for<1, R>([&](auto K) {
        constexpr int k = decltype(K)::value;
        if constexpr ((k & (k - 1)) == 0) {
            constexpr int i = (k == 1) ? 0 : (k == 2) ? 1 : (k == 4) ? 2 : (k == 8) ? 3 : (k == 16) ? 4 : 5;
            w[k] = ldg(tw + i * S + j);
        }
    });
    fill_twiddles<R>(w);
}
// ---------------------------------------------------------------- radix list
// In-place decimation-in-frequency order: pass p has radix r(p) and
// sub-stride s(p) = n / (r(0) * ... * r(p)); after all passes position
// i = sum_p d_p * s(p) holds frequency k = sum_p d_p * (r(0)*...*r(p-1)).
template <int... Rs>
struct RadixList {
    static constexpr int count = sizeof...(Rs);
    static constexpr int n = (Rs * ... * 1);
    static constexpr int r(int p) {
        constexpr int a[] = {Rs...};
        return a[p];
    }
    static constexpr int stride(int p) {   // s(p)
        int prod = 1;
        for (int i = 0; i <= p; i++) prod *= r(i);
        return n / prod;
    }
    static constexpr int weight(int p) {   // r(0) * ... * r(p-1)
        int prod = 1;
        for (int i = 0; i < p; i++) prod *= r(i);
        return prod;
    }
    // Pass p's twiddle table holds only the power-of-two multiples
    //   tw[i*s + j] = exp(-2*pi*i * j * 2^i / (s*r)),  2^i < r,  j in [0,s);
    // the other multiples are products of two table values (pass_twiddles).
    static constexpr int npow(int radix) {
        int n = 0;
        for (int k = 1; k < radix; k *= 2) n++;
        return n;
    }
    static constexpr int tw_offset(int p) {
        int off = 0;
        for (int i = 0; i < p; i++) off += npow(r(i)) * stride(i);
        return off;
    }
    static constexpr int tw_total() { return tw_offset(count); }
    static constexpr int max_radix() {
        int m = 0;
        for (int i = 0; i < count; i++) m = r(i) > m ? r(i) : m;
        return m;
    }
    // position of frequency k after the DIF passes
    static ASC_HD int pos_of_freq(int k) {
        int pos = 0;
        static_for<0, count>([&](auto P) {
            constexpr int p = decltype(P)::value;
            constexpr int rp = r(p);
            int d = k % rp;
            k /= rp;
            pos += d * stride(p);
        });
        return pos;
    }
    // frequency held at position i after the DIF passes
    static ASC_HD int freq_of_pos(int i) {
        int k = 0;
        static_for<0, count>([&](auto P) {
            constexpr int p = decltype(P)::value;
            constexpr int sp = stride(p);
            int d = i / sp;
            i -= d * sp;
            k += d * weight(p);
        });
        return k;
    }
};

}  // namespace asc
