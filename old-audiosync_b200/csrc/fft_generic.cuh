// fft_generic.cuh -- four-step transform kernels with RUNTIME radix lists.
//
// The static kernels of fft_kernels.cuh exist for the six lengths of the reference's interval
// schedule.  The reference itself plans FFTW at call time for whatever sample_len arrives
// (src/cross_correlation.c:34, :141-142, :237), so every other length must be O(N log N) too:
// these kernels run the same algorithm (packed real FFT of complex length M = M1 * M2, column
// pass / fused row pass / inverse column pass with the |r| argmax) for any M1, M2 whose factors
// come from {2,3,4,5,6,8,9,10,12,15,16}, with strides, digit maps and twiddles taken from
// tables instead of template arguments.
//
// Lengths that are not 2/3/5-smooth (or have no usable split) are EMBEDDED: the circular
// correlation of period N = 2L that the reference computes equals, for the lags j < 2L it
// looks at, the linear correlation of the periodically extended source
//     r[j] = sum_{n < L} source[(n + j) mod 2L] * sample[n],     n + j < 3L,
// so any transform length N' = 2M >= 3L gives the same r[0 .. 2L) -- the source is read as
// source[i mod 2L] for i < 3L and zero beyond, the argmax looks at indices < 2L only, and the
// peak is rescaled by N / N' (FFTW's c2r is unnormalised: the reference's values carry N).
// No Bluestein pass is needed.
//
// The arithmetic type is a template parameter: float (the product) or double -- the
// fp64-arithmetic validation mode (audiosync_cuda_set_precise), a second oracle for the fp32
// kernels (reference :187-239 computes in double complex throughout).
//
// Same executor convention as fft_kernels.cuh: the bodies also run on the CPU emulator.
#pragma once

#include "fft_kernels.cuh"

namespace asc {

constexpr int GEN_MAX_PASSES = 8;
constexpr int GEN_THREADS = 256;       // CTA size of the large shapes
constexpr int GEN_THREADS_SMALL = 64;  // ... and of shapes whose passes have fewer than ~128 butterflies per CTA
// Resident CTAs per SM a runtime-radix kernel is compiled for.  fp32: GEN_MIN_CTAS CTAs of 256
// threads (85 registers per thread), the occupancy the planner sizes tiles and rows for; fp64: 256 threads.
constexpr int GEN_MIN_CTAS = 3;
constexpr int gen_min_ctas(int nt, bool is_double) { return is_double ? (nt >= 256 ? 1 : 4) : (GEN_MIN_CTAS * 256) / nt; }

// Division of a small unsigned number by a runtime constant without a divide: q = n / d for
// n < 2^31 (Granlund-Montgomery: m = ceil(2^(31 + ceil(log2 d)) / d)); powers of two shift.
struct FastDiv { unsigned m, s; };
inline FastDiv make_fastdiv(unsigned d) {
    FastDiv f{0u, 0u};
    unsigned l = 0;
    while ((1u << l) < d) l++;                   // ceil(log2 d)
    if ((1u << l) == d) { f.m = 0u; f.s = l; return f; }
    const unsigned long long p = 1ull << (31 + l);
    f.m = (unsigned)((p + d - 1) / d);
    f.s = l - 1;
    return f;
}
ASC_HD unsigned fast_div(unsigned n, FastDiv f) {
#if defined(__CUDA_ARCH__)
    return f.m ? (__umulhi(n, f.m) >> f.s) : (n >> f.s);
#else
    return f.m ? ((unsigned)(((unsigned long long)n * f.m) >> 32) >> f.s) : (n >> f.s);
#endif
}

struct GenAxis {
    int n;                         // axis length
    int npass;
    int radix[GEN_MAX_PASSES];
    int stride[GEN_MAX_PASSES];    // s(p) = n / (r(0) * ... * r(p)); in-place DIF order as RadixList
    FastDiv div_stride[GEN_MAX_PASSES];   // / s(p)
    FastDiv div_items[GEN_MAX_PASSES];    // / (n / r(p)): butterflies of one row in pass p
};

// Twiddles W^(j*k), k = 1 .. R-1, of one butterfly from a full table of the axis (`step` = table
// entries per unit of j*k): the power-of-two multiples are read, the others are products of two
// or three of those (as in pass_twiddles) -- four table reads instead of fifteen at radix 16.
template <int R, class C>
ASC_HD void gen_twiddles(const C* __restrict__ tab, int j, int step, C (&w)[R]) {
    static_for<1, R>([&](auto K) {
        constexpr int k = decltype(K)::value;
        if constexpr ((k & (k - 1)) == 0) w[k] = ldg(tab + j * (k * step));
    });
    fill_twiddles<R, C>(w);
}

struct GenShape {
    long long L;        // sample_len
    long long M;        // complex transform length; N' = 2M real points; M == L unless embedded
    long long src_ext;  // real points of the (periodically extended) source: 2L exact, 3L embedded
    int M1, M2;
    int ct;             // columns per tile of the column kernels (fp32: 16 or 8, fp64: 8)
    int nt_col, nt_row; // threads per CTA of the column / row kernels (GEN_THREADS or GEN_THREADS_SMALL)
    int row_pad;        // rows of the row kernel padded by one point per 128 bytes (1) or plain (0)
    int static_rows;    // fp32 plans: M2 has a static row kernel (gen_plan.h: gen_static_rows); the library runs the rows there
    GenAxis col, row;
};

template <typename T> struct GenTraits;
template <> struct GenTraits<float> {
    typedef cplx C;
    static constexpr int CT = 16;      // columns per tile: 128 bytes
    static constexpr int PADSH = 4;    // row padding: one point per 16 (32 banks)
};
template <> struct GenTraits<double> {
    typedef cplxd C;
    static constexpr int CT = 8;
    static constexpr int PADSH = 3;
};

// Packed point n = (real 2n, real 2n + 1) of a signal.  Source: x[i mod 2L] for i < src_ext, zero
// beyond; sample: y[i] for i < L, zero beyond (the zero pad of reference :159-166).  Points below
// `fast_pts` lie wholly inside the array proper and are read as one vector load (`vec`: the pair's
// base is aligned to two elements).
template <class C, typename InT>
ASC_HD C gen_load_point(const InT* __restrict__ x, unsigned n, int sig, long long L, long long src_ext,
                        unsigned fast_pts, bool vec) {
    typedef typename scalar_of<C>::type real;
    if (n < fast_pts) {
        if (vec) {
            if constexpr (sizeof(InT) == 4) {
                const float2 d = ldg(reinterpret_cast<const float2*>(x) + n);
                return cmake((real)d.x, (real)d.y);
            } else {
                const double2 d = ldg(reinterpret_cast<const double2*>(x) + n);
                return cmake((real)d.x, (real)d.y);
            }
        }
        return cmake((real)ldg(x + 2 * (size_t)n), (real)ldg(x + 2 * (size_t)n + 1));
    }
    const long long i0 = 2 * (long long)n, i1 = i0 + 1;
    real a = (real)0, b = (real)0;
    if (sig == 0) {
        if (i0 < src_ext) a = (real)ldg(x + (i0 < 2 * L ? i0 : i0 - 2 * L));
        if (i1 < src_ext) b = (real)ldg(x + (i1 < 2 * L ? i1 : i1 - 2 * L));
    } else {
        if (i0 < L) a = (real)ldg(x + i0);
        if (i1 < L) b = (real)ldg(x + i1);
    }
    return cmake(a, b);
}

// W^k for k = 1 .. R-1 given the power-of-two powers in g[1], g[2], g[4], g[8]: at most three
// products deep (k < 16).
template <int K, class C>
ASC_HD C gen_pow_from_pow2(const C (&g)[9]) {
    if constexpr ((K & (K - 1)) == 0) {
        return g[K];
    } else {
        constexpr int hb = (K >= 8) ? 8 : (K >= 4) ? 4 : 2;
        return cmul(g[hb], gen_pow_from_pow2<K - hb, C>(g));
    }
}

// Runs f(IC<R>) for the runtime radix r (one of the supported set).
template <class F>
ASC_HD void gen_dispatch_radix(int r, F&& f) {
    switch (r) {
        case 2: f(IC<2>{}); break;
        case 3: f(IC<3>{}); break;
        case 4: f(IC<4>{}); break;
        case 5: f(IC<5>{}); break;
        case 6: f(IC<6>{}); break;
        case 8: f(IC<8>{}); break;
        case 9: f(IC<9>{}); break;
        case 10: f(IC<10>{}); break;
        case 12: f(IC<12>{}); break;
        case 15: f(IC<15>{}); break;
        default: f(IC<16>{}); break;
    }
}
constexpr bool gen_radix_supported(int r) {
    return r == 2 || r == 3 || r == 4 || r == 5 || r == 6 || r == 8 || r == 9 || r == 10 || r == 12 || r == 15 || r == 16;
}

// --------------------------------------------------------------------- G_A
// Forward column pass of both signals: grid = (ceil(M2 / CT), 2, pairs).  A thread keeps its
// column (THREADS is a multiple of CT) and walks the butterflies of that column.
template <typename T, typename InT, int CT_ = GenTraits<T>::CT, int NT_ = GEN_THREADS>
struct GenColFwdKernel {
    typedef typename GenTraits<T>::C C;
    static constexpr int CT = CT_;
    static constexpr int THREADS = NT_;
    static constexpr int TR = THREADS / CT;          // butterflies of one column handled per sweep
    static constexpr int MIN_CTAS = gen_min_ctas(NT_, sizeof(T) == 8);
    static_assert(THREADS % CT == 0, "a thread must keep its column");

    struct Params {
        const InT* sources;
        const InT* samples;
        C* planes;               // [pair][2][M]
        PairPeak* peaks;         // cleared here
        const C* wcol;           // exp(-2*pi*i*t/M1), t < M1
        const C* m_lo;           // W_M two-level tables
        const C* m_hi;
        const int* p2f_col;      // frequency held at position i after the DIF passes
        GenShape sh;
        long long src_pitch, smp_pitch;
        int vec_src, vec_smp;    // the arrays may be read two elements at a time
    };
    static size_t smem_bytes(const GenShape& sh) { return (size_t)sh.M1 * CT * sizeof(C) + 16; }

    template <class Ex>
    static ASC_HD void run(Ex& ex, const Params& p, C* __restrict__ buf) {
        const GenShape& sh = p.sh;
        const int M1 = sh.M1, M2 = sh.M2;
        const int c0 = ex.bx() * CT;
        const int sig = ex.by();
        const long long pair = ex.bz();
        const InT* __restrict__ x = sig == 0 ? p.sources + pair * p.src_pitch : p.samples + pair * p.smp_pitch;
        C* __restrict__ out = p.planes + (pair * 2 + sig) * sh.M;
        const bool vec = sig == 0 ? p.vec_src != 0 : p.vec_smp != 0;
        const long long fast_reals = sig == 0 ? (sh.src_ext < 2 * sh.L ? sh.src_ext : 2 * sh.L) : sh.L;
        const unsigned fast_pts = (unsigned)(fast_reals / 2);
        const int P = sh.col.npass;
        for (int ps = 0; ps < P; ps++) {
            const int S = sh.col.stride[ps];
            const bool first = ps == 0, last = ps == P - 1;
            gen_dispatch_radix(sh.col.radix[ps], [&](auto RR) {
                constexpr int R = decltype(RR)::value;
                const int nbf = M1 / R;
                const int tstep = M1 / (S * R);
                const FastDiv dS = sh.col.div_stride[ps];
                ex.phase([&](int tid) {
                    if (first && tid == 0 && ex.bx() == 0 && sig == 0) p.peaks[pair] = cleared_peak();
                    const int c = tid % CT;
                    const unsigned n2 = (unsigned)(c0 + c);
                    if ((int)n2 >= M2) return;
                    auto load = [&](int i0, C (&v)[R]) {
                        if (first) {
                            // packed points n0 + q * dn; when the last one still lies inside the array
                            // proper the whole butterfly is R vector loads at a constant stride
                            typedef typename scalar_of<C>::type real;
                            const unsigned nfirst = (unsigned)i0 * (unsigned)M2 + n2, dn = (unsigned)S * (unsigned)M2;
                            if (vec && nfirst + (unsigned)(R - 1) * dn < fast_pts) {
                                if constexpr (sizeof(InT) == 4) {
                                    const float2* __restrict__ px = reinterpret_cast<const float2*>(x) + nfirst;
                                    static_for<0, R>([&](auto Q) {
                                        const float2 d2 = ldg(px + (size_t)decltype(Q)::value * dn);
                                        v[decltype(Q)::value] = cmake((real)d2.x, (real)d2.y);
                                    });
                                } else {
                                    const double2* __restrict__ px = reinterpret_cast<const double2*>(x) + nfirst;
                                    static_for<0, R>([&](auto Q) {
                                        const double2 d2 = ldg(px + (size_t)decltype(Q)::value * dn);
                                        v[decltype(Q)::value] = cmake((real)d2.x, (real)d2.y);
                                    });
                                }
                            } else {
                                static_for<0, R>([&](auto Q) {
                                    constexpr int q = decltype(Q)::value;
                                    v[q] = gen_load_point<C, InT>(x, nfirst + (unsigned)q * dn, sig, sh.L, sh.src_ext, fast_pts, vec);
                                });
                            }
                        } else {
                            static_for<0, R>([&](auto Q) { v[decltype(Q)::value] = buf[(i0 + decltype(Q)::value * S) * CT + c]; });
                        }
                    };
                    if (!last) {
                        for (int bf = tid / CT; bf < nbf; bf += TR) {
                            const int blk = (int)fast_div((unsigned)bf, dS), j = bf - blk * S;
                            const int i0 = blk * (S * R) + j;
                            C v[R];
                            load(i0, v);
                            dft_reg<R, -1, C>(v);
                            C t[R];
                            gen_twiddles<R, C>(p.wcol, j, tstep, t);
                            buf[i0 * CT + c] = v[0];
                            static_for<1, R>([&](auto K) {
                                constexpr int k = decltype(K)::value;
                                buf[(i0 + k * S) * CT + c] = cmul(v[k], t[k]);
                            });
                        }
                    } else {
                        // S == 1: positions i0 .. i0+R-1 hold bins k1 = f0 + k * Wt (f0 = bin at i0, Wt = M1 / R).
                        // W_M^(n2 * k1) = W_M^(n2 * f0) * (W_M^(n2 * Wt))^k: the second factor from four
                        // per-thread constants (powers 1, 2, 4, 8), the first from the two-level table.
                        const unsigned Wt = (unsigned)(M1 / R);
                        C g[9];
                        static_for<0, 4>([&](auto I) {
                            constexpr int k = 1 << decltype(I)::value;
                            if constexpr (k < R) g[k] = tw2<C>(p.m_lo, p.m_hi, n2 * Wt * (unsigned)k);
                        });
                        for (int bf = tid / CT; bf < nbf; bf += TR) {
                            const int i0 = bf * R;
                            C v[R];
                            load(i0, v);
                            dft_reg<R, -1, C>(v);
                            const unsigned f0 = (unsigned)ldg(p.p2f_col + i0);
                            const C t0 = tw2<C>(p.m_lo, p.m_hi, n2 * f0);
                            C* __restrict__ o = out + (f0 * (unsigned)M2 + n2);
                            o[0] = cmul(v[0], t0);
                            static_for<1, R>([&](auto K) {
                                constexpr int k = decltype(K)::value;
                                o[(size_t)k * Wt * (unsigned)M2] = cmul(v[k], cmul(t0, gen_pow_from_pow2<k, C>(g)));
                            });
                        }
                    }
                });
            });
        }
    }
};

// --------------------------------------------------------------------- G_B
// Forward rows of both planes, split / conj-multiply / merge, inverse rows: grid = (M1/2 + 1, 1, pairs).
// Rows are padded by one point per 128 bytes (phys), which keeps every pass -- also the stride-1
// pass of an even radix, e.g. power-of-two lengths -- free of bank conflicts.
template <typename T, int NT_ = GEN_THREADS>
struct GenRowFusedKernel {
    typedef typename GenTraits<T>::C C;
    static constexpr int PADSH = GenTraits<T>::PADSH;
    static constexpr int THREADS = NT_;
    static constexpr int MIN_CTAS = gen_min_ctas(NT_, sizeof(T) == 8);

    struct Params {
        C* planes;
        const C* wrow;           // exp(-2*pi*i*t/M2), t < M2
        const C* wpos;           // exp(-2*pi*i*freq_of_pos(e)/M2), position order (the split's twiddle)
        const C* m_lo;
        const C* m_hi;
        const int* f2p_row;      // position of frequency
        GenShape sh;
    };
    static ASC_HD int row_pitch(int M2) { return (M2 + (M2 >> PADSH) + 2) & ~1; }     // even: 16-byte rows for bulk copies
    static size_t smem_bytes(const GenShape& sh) { return (size_t)4 * row_pitch(sh.M2) * sizeof(C) + 16; }

    template <class Ex>
    static ASC_HD void run(Ex& ex, const Params& p, C* __restrict__ buf) {
        const GenShape& sh = p.sh;
        const int M1 = sh.M1, M2 = sh.M2;
        const int RP = row_pitch(M2);
        // padded rows (one point per 128 bytes) where the planner found bank conflicts without them:
        // power-of-two-rich row lengths; plain rows otherwise (cheaper addressing)
        const bool padded = sh.row_pad != 0;
        auto phys = [padded](int p) -> int { return padded ? p + (p >> PADSH) : p; };
        const int r = ex.bx();
        const long long pair = ex.bz();
        const bool two = (r != 0) && (2 * r != M1);
        const int nrows = two ? 2 : 1;
        const int k1a = r, k1b = M1 - r;
        C* __restrict__ plane_s = p.planes + pair * 2 * sh.M;
        C* __restrict__ plane_p = plane_s + sh.M;
        const int P = sh.row.npass;

        // stage: slots 0,1 source rows (k1a, k1b); 2,3 sample rows.  Plain rows of whole 16-byte units
        // arrive as bulk copies of the TMA unit (one instruction per row, completion on an mbarrier
        // behind the last row); padded rows as asynchronous copies of one element each (they are
        // element-aligned only), all in flight before the first wait.
        const bool bulk = !padded && ((size_t)M2 * sizeof(C)) % 16 == 0 && (size_t)M2 * sizeof(C) >= 4096;   // short rows: cp.async has the lower latency
        void* mbar = buf + 4 * RP;
        if (bulk) {
            ex.phase([&](int tid) {
                if (tid == 0) mbar_init(mbar, 1);
            });
            ex.phase([&](int tid) {
                if (tid == 0) {
                    const unsigned full = (unsigned)(M2 * sizeof(C));
                    mbar_expect_tx(mbar, (unsigned)(2 * nrows) * full);
                    bulk_load(buf, plane_s + (long long)k1a * M2, full, mbar);
                    bulk_load(buf + 2 * RP, plane_p + (long long)k1a * M2, full, mbar);
                    if (two) {
                        bulk_load(buf + RP, plane_s + (long long)k1b * M2, full, mbar);
                        bulk_load(buf + 3 * RP, plane_p + (long long)k1b * M2, full, mbar);
                    }
                }
                mbar_wait(mbar, 0);
            });
        } else
        ex.phase([&](int tid) {
            for (int slot = 0; slot < 4; slot++) {
                const int rr = slot & 1;
                if (rr == 1 && !two) continue;
                const C* __restrict__ g = (slot >= 2 ? plane_p : plane_s) + (long long)(rr ? k1b : k1a) * M2;
                C* __restrict__ row = buf + slot * RP;
                for (int e = tid; e < M2; e += THREADS) {
                    if constexpr (sizeof(C) == 8) cp_async8(row + phys(e), g + e);
                    else cp_async16(row + phys(e), g + e);
                }
            }
            cp_async_wait_all();
        });
        // (element i0 + q * S of a padded row: when S is a multiple of the padding period the
        // physical stride is the constant S + S / period -- the `regular` passes below)
        // forward DIF on 2 * nrows rows (slots 0,1,2,3 or 0,2)
        for (int ps = 0; ps < P; ps++) {
            const int S = sh.row.stride[ps];
            gen_dispatch_radix(sh.row.radix[ps], [&](auto RR) {
                constexpr int R = decltype(RR)::value;
                const int per_row = M2 / R;
                const int items = per_row * 2 * nrows;
                const int tstep = M2 / (S * R);
                const FastDiv dS = sh.row.div_stride[ps], dI = sh.row.div_items[ps];
                const bool regular = !padded || (S & ((1 << PADSH) - 1)) == 0;
                const int SP = padded ? S + (S >> PADSH) : S;
                ex.phase([&](int tid) {
                    for (int w = tid; w < items; w += THREADS) {
                        const int bw = (int)fast_div((unsigned)w, dI), bf = w - bw * per_row;
                        C* __restrict__ row = buf + (two ? bw : 2 * bw) * RP;
                        const int blk = (int)fast_div((unsigned)bf, dS), j = bf - blk * S;
                        const int i0 = blk * (S * R) + j;
                        C v[R];
                        if (regular) {
                            C* __restrict__ b0 = row + phys(i0);
                            static_for<0, R>([&](auto Q) { v[decltype(Q)::value] = b0[decltype(Q)::value * SP]; });
                            dft_reg<R, -1, C>(v);
                            C t[R];
                            gen_twiddles<R, C>(p.wrow, j, tstep, t);
                            b0[0] = v[0];
                            static_for<1, R>([&](auto K) { b0[decltype(K)::value * SP] = cmul(v[decltype(K)::value], t[decltype(K)::value]); });
                        } else {
                            static_for<0, R>([&](auto Q) { v[decltype(Q)::value] = row[phys(i0 + decltype(Q)::value * S)]; });
                            dft_reg<R, -1, C>(v);
                            row[phys(i0)] = v[0];
                            if (S > 1) {
                                C t[R];
                                gen_twiddles<R, C>(p.wrow, j, tstep, t);
                                static_for<1, R>([&](auto K) { row[phys(i0 + decltype(K)::value * S)] = cmul(v[decltype(K)::value], t[decltype(K)::value]); });
                            } else {
                                static_for<1, R>([&](auto K) { row[phys(i0 + decltype(K)::value)] = v[decltype(K)::value]; });
                            }
                        }
                    }
                });
            });
        }
        // split + conj-multiply (reference :232-233) + merge, into the source rows
        ex.phase([&](int tid) {
            const C wk1 = tw2<C>(p.m_lo, p.m_hi, (unsigned)k1a);
            if (two) {
                C* __restrict__ zs_a = buf;
                C* __restrict__ zs_b = buf + RP;
                C* __restrict__ zp_a = buf + 2 * RP;
                C* __restrict__ zp_b = buf + 3 * RP;
                for (int e = tid; e < M2; e += THREADS) {
                    const int pa = phys(e), pb = phys(M2 - 1 - e);
                    const C w2 = cmul(ldg(p.wpos + e), wk1);
                    C qk, qmk;
                    split_mul_merge_w2<C>(zs_a[pa], zs_b[pb], zp_a[pa], zp_b[pb], w2, qk, qmk);
                    zs_a[pa] = qk;
                    zs_b[pb] = qmk;
                }
            } else {
                C* __restrict__ zs = buf;
                C* __restrict__ zp = buf + 2 * RP;
                const int items = r == 0 ? M2 / 2 + 1 : (M2 + 1) / 2;
                for (int e = tid; e < items; e += THREADS) {
                    int ea, eb;      // positions
                    if (r == 0) {
                        ea = ldg(p.f2p_row + e);
                        eb = ldg(p.f2p_row + (e == 0 ? 0 : M2 - e));
                    } else {
                        ea = e;
                        eb = M2 - 1 - e;
                    }
                    const C w2 = cmul(ldg(p.wpos + ea), wk1);
                    const int pa = phys(ea), pb = phys(eb);
                    C qk, qmk;
                    split_mul_merge_w2<C>(zs[pa], zs[pb], zp[pa], zp[pb], w2, qk, qmk);
                    zs[pa] = qk;
                    if (pa != pb) zs[pb] = qmk;
                }
            }
        });
        // inverse DIT on nrows rows (slots 0,1), passes P-1 .. 1 in place
        for (int ps = P - 1; ps >= 1; ps--) {
            const int S = sh.row.stride[ps];
            gen_dispatch_radix(sh.row.radix[ps], [&](auto RR) {
                constexpr int R = decltype(RR)::value;
                const int per_row = M2 / R;
                const int items = per_row * nrows;
                const int tstep = M2 / (S * R);
                const FastDiv dS = sh.row.div_stride[ps], dI = sh.row.div_items[ps];
                const bool regular = !padded || (S & ((1 << PADSH) - 1)) == 0;
                const int SP = padded ? S + (S >> PADSH) : S;
                ex.phase([&](int tid) {
                    for (int w = tid; w < items; w += THREADS) {
                        const int rw = (int)fast_div((unsigned)w, dI), bf = w - rw * per_row;
                        C* __restrict__ row = buf + rw * RP;
                        const int blk = (int)fast_div((unsigned)bf, dS), j = bf - blk * S;
                        const int i0 = blk * (S * R) + j;
                        C v[R];
                        if (regular) {
                            C* __restrict__ b0 = row + phys(i0);
                            C t[R];
                            gen_twiddles<R, C>(p.wrow, j, tstep, t);
                            v[0] = b0[0];
                            static_for<1, R>([&](auto Q) { v[decltype(Q)::value] = cmulc(b0[decltype(Q)::value * SP], t[decltype(Q)::value]); });
                            dft_reg<R, +1, C>(v);
                            static_for<0, R>([&](auto K) { b0[decltype(K)::value * SP] = v[decltype(K)::value]; });
                        } else {
                            v[0] = row[phys(i0)];
                            if (S > 1) {
                                C t[R];
                                gen_twiddles<R, C>(p.wrow, j, tstep, t);
                                static_for<1, R>([&](auto Q) { v[decltype(Q)::value] = cmulc(row[phys(i0 + decltype(Q)::value * S)], t[decltype(Q)::value]); });
                            } else {
                                static_for<1, R>([&](auto Q) { v[decltype(Q)::value] = row[phys(i0 + decltype(Q)::value)]; });
                            }
                            dft_reg<R, +1, C>(v);
                            static_for<0, R>([&](auto K) { row[phys(i0 + decltype(K)::value * S)] = v[decltype(K)::value]; });
                        }
                    }
                });
            });
        }
        // last inverse pass (pass 0: one block per row, butterfly j yields the natural-order points
        // n2 = j + k * S): times conj W_M^(n2 * k1) = conj(W_M^(j * k1) * (W_M^(S * k1))^k), straight
        // to row k1 of plane 0 -- consecutive threads, consecutive points
        {
            const int S = sh.row.stride[0];
            gen_dispatch_radix(sh.row.radix[0], [&](auto RR) {
                constexpr int R = decltype(RR)::value;
                const int tstep = M2 / (S * R);           // == 1
                const bool regular = !padded || (S & ((1 << PADSH) - 1)) == 0;
                const int SP = padded ? S + (S >> PADSH) : S;
                ex.phase([&](int tid) {
                    for (int w = tid; w < nrows * S; w += THREADS) {
                        const int rw = w >= S ? 1 : 0, j = w - rw * S;
                        const unsigned k1 = (unsigned)(rw ? k1b : k1a);
                        C* __restrict__ row = buf + rw * RP;
                        C* __restrict__ o = plane_s + (size_t)k1 * (unsigned)M2;
                        {
                            C v[R];
                            {
                                // twiddles from their four power-of-two entries as they are used (a full
                                // t[R] beside v[R] would not fit the 85-register budget in this pass)
                                C t[9];
                                static_for<0, 4>([&](auto I) {
                                    constexpr int k = 1 << decltype(I)::value;
                                    if constexpr (k < R) t[k] = ldg(p.wrow + j * (k * tstep));
                                });
                                if (regular) {
                                    C* __restrict__ b0 = row + phys(j);
                                    v[0] = b0[0];
                                    static_for<1, R>([&](auto Q) { v[decltype(Q)::value] = cmulc(b0[decltype(Q)::value * SP], gen_pow_from_pow2<decltype(Q)::value, C>(t)); });
                                } else {
                                    v[0] = row[phys(j)];
                                    static_for<1, R>([&](auto Q) { v[decltype(Q)::value] = cmulc(row[phys(j + decltype(Q)::value * S)], gen_pow_from_pow2<decltype(Q)::value, C>(t)); });
                                }
                            }
                            dft_reg<R, +1, C>(v);
                            // the row's constants are formed here, after the butterfly (a thread runs this
                            // loop once or twice: keeping them live across it only costs registers)
                            C g[9];
                            static_for<0, 4>([&](auto I) {
                                constexpr int k = 1 << decltype(I)::value;
                                if constexpr (k < R) g[k] = tw2<C>(p.m_lo, p.m_hi, (unsigned)(S * k) * k1);
                            });
                            const C t0 = tw2<C>(p.m_lo, p.m_hi, (unsigned)j * k1);
                            o[j] = cmulc(v[0], t0);
                            static_for<1, R>([&](auto K) {
                                constexpr int k = decltype(K)::value;
                                o[j + k * S] = cmulc(v[k], cmul(t0, gen_pow_from_pow2<k, C>(g)));
                            });
                        }
                    }
                });
            });
        }
    }
};

// --------------------------------------------------------------------- G_C
// Inverse column pass.  fp32: |r| argmax epilogue over the indices < limit (= 2L), the correlation
// is never written.  fp64: r[0 .. limit) is written to `r_out` (the dead sample plane) and resolved
// by argmax_f64_kernel, which keeps full double keys.  grid = (pairs, ceil(M2 / CT)).
template <typename T, int CT_ = GenTraits<T>::CT, int NT_ = GEN_THREADS>
struct GenColInvKernel {
    typedef typename GenTraits<T>::C C;
    static constexpr int CT = CT_;
    static constexpr int THREADS = NT_;
    static constexpr int TR = THREADS / CT;
    static constexpr int MIN_CTAS = gen_min_ctas(NT_, sizeof(T) == 8);

    struct Params {
        const C* planes;
        PairPeak* peaks;
        const C* wcol;
        const int* p2f_col;
        GenShape sh;
        T* r_out;                // fp64 only: [pair][2M] reals (aliases plane 1 of the pair)
    };
    static size_t smem_bytes(const GenShape& sh) {
        const size_t tile = (size_t)sh.M1 * CT * sizeof(C);
        return (tile > 512 ? tile : 512) + 16;
    }

    template <class Ex>
    static ASC_HD void run(Ex& ex, const Params& p, C* __restrict__ buf) {
        const GenShape& sh = p.sh;
        const int M1 = sh.M1, M2 = sh.M2;
        const int c0 = ex.by() * CT;
        const long long pair = ex.bx();
        const C* __restrict__ in = p.planes + pair * 2 * sh.M;
        const unsigned limit = (unsigned)(2 * sh.L);          // < 2^31: M < 2^30
        const int P = sh.col.npass;
        for (int ps = 0; ps < P - 1; ps++) {
            const int S = sh.col.stride[ps];
            const bool first = ps == 0;
            gen_dispatch_radix(sh.col.radix[ps], [&](auto RR) {
                constexpr int R = decltype(RR)::value;
                const int nbf = M1 / R;
                const int tstep = M1 / (S * R);
                const FastDiv dS = sh.col.div_stride[ps];
                ex.phase([&](int tid) {
                    const int c = tid % CT;
                    const int n2 = c0 + c;
                    if (n2 >= M2) return;
                    for (int bf = tid / CT; bf < nbf; bf += TR) {
                        const int blk = (int)fast_div((unsigned)bf, dS), j = bf - blk * S;
                        const int i0 = blk * (S * R) + j;
                        C v[R];
                        if (first) {
                            const C* __restrict__ g0 = in + ((unsigned)i0 * (unsigned)M2 + (unsigned)n2);
                            static_for<0, R>([&](auto Q) { v[decltype(Q)::value] = ldg(g0 + (size_t)decltype(Q)::value * S * (unsigned)M2); });
                        } else {
                            static_for<0, R>([&](auto Q) { v[decltype(Q)::value] = buf[(i0 + decltype(Q)::value * S) * CT + c]; });
                        }
                        dft_reg<R, +1, C>(v);
                        C t[R];
                        gen_twiddles<R, C>(p.wcol, j, tstep, t);
                        buf[i0 * CT + c] = v[0];
                        static_for<1, R>([&](auto K) {
                            constexpr int k = decltype(K)::value;
                            buf[(i0 + k * S) * CT + c] = cmulc(v[k], t[k]);
                        });
                    }
                });
            });
        }
        // last pass (S == 1): positions i0 .. i0+R-1 hold n1 = f0 + k * Wt; packed point
        // n = n1 * M2 + n2 carries r[2n] (real part) and r[2n + 1] (imaginary part)
        const bool only = P == 1;
        gen_dispatch_radix(sh.col.radix[P - 1], [&](auto RR) {
            constexpr int R = decltype(RR)::value;
            const int nbf = M1 / R;
            const unsigned Wt = (unsigned)(M1 / R);
            // butterfly bf of column n2 -> v[0 .. R), index of v[0].x
            auto butterfly = [&](int bf, int c, int n2, C (&v)[R]) -> unsigned {
                const int i0 = bf * R;
                if (only) {
                    const C* __restrict__ g0 = in + ((unsigned)i0 * (unsigned)M2 + (unsigned)n2);
                    static_for<0, R>([&](auto Q) { v[decltype(Q)::value] = ldg(g0 + (size_t)decltype(Q)::value * (unsigned)M2); });
                } else {
                    static_for<0, R>([&](auto Q) { v[decltype(Q)::value] = buf[(i0 + decltype(Q)::value) * CT + c]; });
                }
                dft_reg<R, +1, C>(v);
                return 2u * ((unsigned)ldg(p.p2f_col + i0) * (unsigned)M2 + (unsigned)n2);
            };
            if constexpr (sizeof(T) == 4) {
                ex.phase_argmax(
                    [&](int tid) -> ArgmaxPair {
                        ArgmaxAcc acc;
                        const unsigned int seen = ex.peek_bits(&p.peaks[pair].second_bits);
                        if (seen != 0u) acc.thr = float_from_order_bits(seen);
                        const int c = tid % CT;
                        const int n2 = c0 + c;
                        if (n2 < M2)
                        for (int bf = tid / CT; bf < nbf; bf += TR) {
                            C v[R];
                            const unsigned i_first = butterfly(bf, c, n2, v);
                            // only values that reach the running second peak can matter
                            float gm = fmaxf(fabsf(v[0].x), fabsf(v[0].y));
                            static_for<1, R>([&](auto K) { gm = fmaxf(gm, fmaxf(fabsf(v[decltype(K)::value].x), fabsf(v[decltype(K)::value].y))); });
                            if (!(gm >= acc.thr) && i_first != 0u && gm == gm) continue;
                            static_for<0, R>([&](auto K) {
                                constexpr int k = decltype(K)::value;
                                const unsigned i_re = i_first + 2u * (unsigned)k * Wt * (unsigned)M2;
                                if (i_re < limit) {
                                    if (i_re == 0u) acc.consider_seed(v[k].x, &p.peaks[pair]);
                                    else acc.consider(v[k].x, i_re);
                                }
                                if (i_re + 1u < limit) acc.consider(v[k].y, i_re + 1u);
                            });
                        }
                        return acc.result();
                    },
                    &p.peaks[pair].key, &p.peaks[pair].second_bits, buf);
            } else {
                T* __restrict__ r = p.r_out + (pair * 4 + 2) * sh.M;     // plane 1 of the pair, as reals
                ex.phase([&](int tid) {
                    const int c = tid % CT;
                    const int n2 = c0 + c;
                    if (n2 >= M2) return;
                    for (int bf = tid / CT; bf < nbf; bf += TR) {
                        C v[R];
                        const unsigned i_first = butterfly(bf, c, n2, v);
                        static_for<0, R>([&](auto K) {
                            constexpr int k = decltype(K)::value;
                            const unsigned i_re = i_first + 2u * (unsigned)k * Wt * (unsigned)M2;
                            if (i_re < limit) r[i_re] = v[k].x;
                            if (i_re + 1u < limit) r[i_re + 1u] = v[k].y;
                        });
                    }
                });
            }
        });
    }
};

// Entry for kernels whose shared-memory buffer is not cplx-typed.
#if defined(__CUDACC__)
template <class K>
__global__ void __launch_bounds__(K::THREADS, K::MIN_CTAS)
gen_kernel_entry(const typename K::Params p) {
    extern __shared__ __align__(128) unsigned char asc_smem_gen[];
    pdl_prologue();
    DeviceExec ex;
    ex.x_ = (int)blockIdx.x; ex.y_ = (int)blockIdx.y; ex.z_ = (int)blockIdx.z;
    K::run(ex, p, reinterpret_cast<typename K::C*>(asc_smem_gen));
}
#endif

}  // namespace asc
