// fft_kernels.cuh -- the three transform kernels of the four-step plan.
//
// Complex length M = L (two reals packed per complex point), split M = M1 * M2,
// point n = n1*M2 + n2, bin k = k1 + M1*k2.  Per pair, per wave:
//
//   K_A  ColFwdKernel   one CTA per (16-column tile, signal): M1-point forward
//        FFT down the columns n2 of the packed input (read straight from the
//        caller's real array; the zero half of the padded sample is never read),
//        times W_M^(n2*k1), written as plane[k1][n2].
//   K_B  RowFusedKernel one CTA per row pair (k1, M1-k1): M2-point forward FFT
//        of those rows of both planes, the real-FFT split, the conj-multiply,
//        the merge for the inverse real FFT, and the M2-point inverse FFT of
//        the two product rows, times conj W_M^(n2*k1), written back in place.
//        (reference src/cross_correlation.c:232-233 lives inside this kernel.)
//   K_C  ColInvKernel   one CTA per 16-column tile: M1-point inverse FFT down
//        the columns and the |r| argmax epilogue (reference :52-67, :242) --
//        the correlation itself is never written to memory.
//
// All passes are in-place radix passes in shared memory (decimation in
// frequency forward, decimation in time for the inverse rows).  Tiles and rows
// are staged global -> shared by the TMA unit -- boxes of a 3-D tensor map for the
// column tiles (cp.async.bulk.tensor), plain bulk copies for the contiguous rows,
// completion on an mbarrier -- so that no thread spends instructions on the load
// and the load of one CTA overlaps the butterflies of the other CTAs on the SM;
// K_B's product rows leave the same way (cp.async.bulk shared -> global).  Only
// K_A has a second path: its first pass loads through registers where the input
// cannot be staged (fp64, int16, or fp32 not 16-byte aligned).  The last pass is fused
// with the global store / epilogue.
//
// Kernel bodies are written against an executor (DeviceExec on the GPU,
// tests/emu's HostExec on the CPU) that runs one "phase" for every thread and
// then synchronises, so the same source is what the emulator checks.
#pragma once

#include "common.cuh"
#include "fft_device.cuh"

namespace asc {

constexpr int COL_T = 16;          // columns per tile: 16 * 8 B = one 128-byte line

// Resident CTAs per SM a transform kernel is built for (its register budget follows from it):
// as many as its tile allows in the SM's 228 KB of shared memory (1 KB per CTA is reserved),
// and as 1024 threads allow, at most 3 -- 960 threads of 64 registers.
constexpr int ctas_per_sm(size_t smem, int threads) {
    const int by_smem = (int)((228u * 1024u) / (smem + 1024u));
    const int by_threads = 1024 / threads;
    const int n = by_smem < by_threads ? by_smem : by_threads;
    return n >= 3 ? 3 : (n >= 1 ? n : 1);
}
constexpr unsigned TW2_BITS = 10;  // two-level twiddle tables: a = hi * 1024 + lo
constexpr unsigned TW2_MASK = (1u << TW2_BITS) - 1u;

// exp(-2*pi*i*a/base) from the two-level tables (both halves correctly rounded
// from fp64 on the host; one complex product here).
template <class C>
ASC_HD C tw2(const C* __restrict__ lo, const C* __restrict__ hi, unsigned a) {
    return cmul(ldg(lo + (a & TW2_MASK)), ldg(hi + (a >> TW2_BITS)));
}

// Column tiles staged by the TMA unit: `rows` tile rows are covered by tile_boxes(rows) boxes
// of tile_box_rows(rows) rows (a tensor-map box holds at most 256), the last one shifted up so
// that it ends on the last row (overlapping rows are simply loaded twice).
constexpr int tile_boxes(int rows) { return (rows + 255) / 256; }
constexpr int tile_box_rows(int rows) { return (rows + tile_boxes(rows) - 1) / tile_boxes(rows); }
constexpr int tile_box_start(int rows, int i) {
    return i * tile_box_rows(rows) + tile_box_rows(rows) <= rows ? i * tile_box_rows(rows) : rows - tile_box_rows(rows);
}

// Packed point n = (x[2n], x[2n + 1]).  vec: one load of both elements (float2, double2, short2;
// the base is aligned to two elements); otherwise two element loads.  A base is only guaranteed
// element alignment: a view at an odd element offset, such as x[1:], has no more.
template <typename InT>
ASC_HD cplx load_packed(const InT* __restrict__ x, long long n, bool vec = true);

template <>
ASC_HD cplx load_packed<float>(const float* __restrict__ x, long long n, bool vec) {
    if (vec) return ldg(reinterpret_cast<const float2*>(x) + n);
    return cmake(ldg(x + 2 * n), ldg(x + 2 * n + 1));
}
template <>
ASC_HD cplx load_packed<double>(const double* __restrict__ x, long long n, bool vec) {
    if (vec) {
        const double2 d = ldg(reinterpret_cast<const double2*>(x) + n);
        return cmake(in_real<float>(d.x), in_real<float>(d.y));
    }
    return cmake(in_real<float>(ldg(x + 2 * n)), in_real<float>(ldg(x + 2 * n + 1)));
}
template <>
ASC_HD cplx load_packed<int16_t>(const int16_t* __restrict__ x, long long n, bool vec) {
    if (vec) {
        const short2 s = ldg(reinterpret_cast<const short2*>(x) + n);
        return cmake(in_real<float>(s.x), in_real<float>(s.y));
    }
    return cmake(in_real<float>(ldg(x + 2 * n)), in_real<float>(ldg(x + 2 * n + 1)));
}

// Running |r| argmax of one thread (reference src/cross_correlation.c:52-67 as
// a max over packed keys, see common.cuh) plus the SECOND peak: the largest
// |r[i]| over every entry i >= 1 other than the winner (SURVEY 8f rank 4; the
// oracle's `second`, which makes "the peak is unique" observable).  The packed key
// is only built for candidates that can still change either; a NaN never passes
// `a >= thr`.
//
// The threshold argument -- a value below the running second peak can be neither the
// peak nor the second -- holds for every entry i >= 1 but not for the signed seed
// r[0]: a negative r[0] loses to any |r[i]| while possibly being the largest magnitude,
// so its |r[0]| must not raise `thr`, the warp's bound or the pair's published
// second_bits.  It never enters `second`; the seed's thread stores it in
// PairPeak::seed_bits, and pair_second() joins it to the second peak at the end.
struct ArgmaxPair {
    unsigned long long best;
    float second;
};

struct ArgmaxAcc {
    unsigned long long best = 0ull;
    float second = 0.0f;             // largest |v| seen by this thread except `best`
    float thr = 0.0f;                // lower bound of the pair's final second peak: smaller magnitudes are skipped
    ASC_HD void update(unsigned long long key, float a) {
        if (key > best) {
            if (best != 0ull && !argmax_key_is_seed(best)) second = fmaxf(second, argmax_key_mag(best));
            best = key;
        } else {
            second = fmaxf(second, a);
        }
        thr = fmaxf(thr, second);    // this thread's own second peak bounds the pair's from below
    }
    ASC_HD void consider(float v, uint32_t index) {   // index >= 1
        const float a = fabsf(v);
        if (a >= thr) update(argmax_key_abs(v, index), a);
    }
    ASC_HD void consider_seed(float v, PairPeak* pk) {   // index 0, signed
        update(argmax_key_seed(v), 0.0f);
        pk->seed_bits = float_order_bits(fabsf(v));
    }
    // bound for the warp's threshold: the seed's magnitude is none (see above)
    ASC_HD float best_mag() const { return best != 0ull && !argmax_key_is_seed(best) ? argmax_key_mag(best) : 0.0f; }
    ASC_HD ArgmaxPair result() const { ArgmaxPair r; r.best = best; r.second = second; return r; }
};

// Merges the (peak key, second peak) pair (ob, os) into (best, second).  Pairs merge
// associatively: the larger key leads, the smaller key's magnitude joins the two seconds
// (unless it is the seed's, see ArgmaxAcc).  At grid level the key an atomicMax displaces (or
// fails to displace) is merged with os = 0: over all CTAs max(min(old, mine)) is exactly the
// second largest CTA peak.
ASC_HD void argmax_merge(unsigned long long& best, float& second, unsigned long long ob, float os) {
    const unsigned long long lose = ob > best ? best : ob;
    best = ob > best ? ob : best;
    second = fmaxf(second, os);
    if (lose != 0ull && !argmax_key_is_seed(lose)) second = fmaxf(second, argmax_key_mag(lose));
}

// --------------------------------------------------------------------- K_A
// TMA (fp32 input, 16-byte aligned): the tile is staged in shared memory before pass 0 as boxes
// of a tensor map through the TMA unit, completion on an mbarrier, and the zero half of the
// padded sample is never touched; otherwise (fp64 or int16 input, or unaligned fp32 pointers) the
// first pass loads, converts and packs through registers.
//
// TMA staging of the SOURCE tile: the CTA's shared memory is exactly the tile, so the 8-byte
// mbarrier sits at its very end and the last tile row (128 bytes) is not staged; pass 0 reads
// that row from global memory, and the thread whose butterfly writes the barrier's bytes
// invalidates it first.  (The sample tile has its unstaged upper half to spare.)
template <class RL, int M2_, int NT, typename InT, bool TMA>
struct ColFwdKernel {
    static constexpr int M1 = RL::n;
    static constexpr int M2 = M2_;                  // row length (compile time: index products fold)
    static constexpr int P = RL::count;
    static constexpr int THREADS = NT;
    static constexpr size_t SMEM = (size_t)M1 * COL_T * sizeof(cplx);
    static constexpr int MIN_CTAS = ctas_per_sm(SMEM, NT);
    static_assert(NT % COL_T == 0, "a thread must keep its column across items");
    static_assert(P >= 2, "column plans need at least two passes");
    static_assert(!TMA || std::is_same<InT, float>::value, "TMA staging copies packed fp32 pairs verbatim");
    static_assert(!TMA || M1 >= 4, "tile too small for a box");
    static_assert(M1 % 2 == 0, "the zero half of the sample must be whole tile rows");

    struct Params {
        const InT* sources;      // [pair][2L] reals
        const InT* samples;      // [pair][L] reals
        cplx* planes;            // [pair][2][M1*M2]: plane 0 source, plane 1 sample
        PairPeak* peaks;         // [pair]: argmax slot, cleared here for K_C
        const cplx* tw;          // RL pass tables (forward sign, power-of-two multiples)
        const cplx* tc;          // [M1/R_last][16]: W_M^(c*f0)
        const cplx* m_lo;        // W_M two-level tables
        const cplx* m_hi;
        long long L;             // sample_len == M = M1 * M2
        long long src_pitch;     // elements between consecutive pairs' sources / samples;
        long long smp_pitch;     // 0 = packed ([pair][2L] and [pair][L])
        // register path: every pair's sources / samples start aligned to two elements (one load
        // per packed point); CTA-uniform.  These sit in the padding before the tensor maps.
        int vec_src, vec_smp;
        // TMA: [pair][M1 or M1/2 rows][2*M2 floats] views of sources / samples, boxes of
        // 32 floats x tile_box_rows(M1 - 1) resp. tile_box_rows(M1 / 2) rows
        CUtensorMap tm_src, tm_smp;
    };
    static constexpr int SRC_ROWS = M1 - 1, SMP_ROWS = M1 / 2;   // rows the TMA unit stages

    // grid = (M2 / 16, 2, pairs)
    template <class Ex>
    static ASC_HD void run(Ex& ex, const Params& p, cplx* __restrict__ buf) {
        const int c0 = ex.bx() * COL_T;
        const int sig = ex.by();
        const long long pair = ex.bz();
        const long long M = p.L;
        const InT* __restrict__ x = sig == 0 ? p.sources + pair * (p.src_pitch ? p.src_pitch : 2 * M)
                                             : p.samples + pair * (p.smp_pitch ? p.smp_pitch : M);
        // number of valid packed points: source M, sample M/2 (upper half is the zero pad)
        const long long nvalid = sig == 0 ? M : M / 2;
        [[maybe_unused]] const bool vec = sig == 0 ? p.vec_src != 0 : p.vec_smp != 0;
        cplx* __restrict__ out = p.planes + (pair * 2 + sig) * M;
        const bool clears_peak = ex.bx() == 0 && sig == 0;

        [[maybe_unused]] void* mbar = reinterpret_cast<char*>(buf) + SMEM - 8;
        if constexpr (TMA) {
            ex.phase([&](int tid) {
                if (tid == 0) {
                    if (clears_peak) p.peaks[pair] = cleared_peak();
                    mbar_init(mbar, 1);
                }
            });
            ex.phase([&](int tid) {
                if (tid == 0) {
                    const char* __restrict__ raw = reinterpret_cast<const char*>(x) + (size_t)c0 * sizeof(cplx);
                    constexpr size_t pitch = (size_t)M2 * sizeof(cplx);
                    if (sig == 0) {
                        constexpr int NB = tile_boxes(SRC_ROWS), BR = tile_box_rows(SRC_ROWS);
                        mbar_expect_tx(mbar, (unsigned)(NB * BR * 128));
                        static_for<0, NB>([&](auto I) {
                            constexpr int r0 = tile_box_start(SRC_ROWS, decltype(I)::value);
                            tma_load_rows(buf + r0 * COL_T, &p.tm_src, 2 * c0, r0, (int)pair, mbar, raw + r0 * pitch, pitch, BR);
                        });
                    } else {
                        constexpr int NB = tile_boxes(SMP_ROWS), BR = tile_box_rows(SMP_ROWS);
                        mbar_expect_tx(mbar, (unsigned)(NB * BR * 128));
                        static_for<0, NB>([&](auto I) {
                            constexpr int r0 = tile_box_start(SMP_ROWS, decltype(I)::value);
                            tma_load_rows(buf + r0 * COL_T, &p.tm_smp, 2 * c0, r0, (int)pair, mbar, raw + r0 * pitch, pitch, BR);
                        });
                    }
                }
                mbar_wait(mbar, 0);
            });
        }

        static_for<0, P>([&](auto PP) {
            constexpr int ps = decltype(PP)::value;
            constexpr int R = RL::r(ps);
            constexpr int S = RL::stride(ps);
            constexpr bool first = ps == 0, last = ps == P - 1;
            constexpr bool from_global = first && !TMA;
            constexpr int items = (M1 / R) * COL_T;
            ex.phase([&](int tid) {
                if (from_global && clears_peak && tid == 0) p.peaks[pair] = cleared_peak();
                const int c = tid & (COL_T - 1);          // fixed column of this thread
                if constexpr (!last) {
                    // HZ: first pass of a staged SAMPLE tile.  Inputs q >= R/2 are rows of the
                    // zero pad (i0 + q*S >= M1/2): zeros in registers, no shared-memory reads.
                    auto items_loop = [&](auto HZ) {
                        [[maybe_unused]] constexpr bool hz = decltype(HZ)::value;
                        cplx t[R];
                        for (int w = tid; w < items; w += NT) {
                            const int bf = w >> 4;
                            const int blk = (S * R == M1) ? 0 : bf / S;    // pass 0: one block
                            const int j = bf - blk * S;
                            const int i0 = blk * (S * R) + j;
                            cplx v[R];
                            if constexpr (from_global) {
                                static_for<0, R>([&](auto Q) {
                                    constexpr int q = decltype(Q)::value;
                                    const long long n = (long long)(i0 + q * S) * M2 + c0 + c;
                                    v[q] = n < nvalid ? load_packed<InT>(x, n, vec) : cmake(0.f, 0.f);
                                });
                            } else {
                                static_for<0, R>([&](auto Q) {
                                    constexpr int q = decltype(Q)::value;
                                    if constexpr (hz && 2 * q >= R) {
                                        v[q] = cmake(0.f, 0.f);
                                    } else if constexpr (TMA && first && !hz && q == R - 1) {
                                        // tile row M1 - 1 is not staged (the mbarrier sits there)
                                        if (i0 == S - 1) v[q] = load_packed<InT>(x, (long long)(M1 - 1) * M2 + c0 + c);
                                        else v[q] = buf[(i0 + q * S) * COL_T + c];
                                    } else {
                                        v[q] = buf[(i0 + q * S) * COL_T + c];
                                    }
                                });
                                if constexpr (TMA && first) {
                                    if (i0 == S - 1 && c == COL_T - 1) mbar_inval(mbar);   // overwritten below
                                }
                            }
                            dft_reg<R, -1>(v);
                            pass_twiddles<R>(p.tw + RL::tw_offset(ps), S, j, t);
                            buf[i0 * COL_T + c] = v[0];
                            static_for<1, R>([&](auto K) {
                                constexpr int k = decltype(K)::value;
                                buf[(i0 + k * S) * COL_T + c] = cmul(v[k], t[k]);
                            });
                        }
                    };
                    if constexpr (first && TMA) {
                        static_assert(R % 2 == 0 && S * R == M1, "zero-pad rows must be the inputs q >= R/2 of pass 0");
                        if (sig == 1) items_loop(std::true_type{});
                        else items_loop(std::false_type{});
                    } else {
                        items_loop(std::false_type{});
                    }
                } else {
                    // S == 1: positions i0 .. i0+R-1 hold bins k1 = f0 + k*Wt, f0 < Wt.
                    // W_M^(n2*k1) = W_M^(n2*f0) * (W_M^(n2*Wt))^k; the second factor is a
                    // per-thread constant, the first is tc[f0][c] * W_M^(c0*f0).
                    constexpr int Wt = RL::weight(ps);
                    const unsigned n2 = (unsigned)(c0 + c);
                    // Wide last radix (R > 8): only the power-of-two multiples are held; the
                    // others are formed as products where they are used (as in pass_twiddles),
                    // so the per-thread constants do not crowd out the butterfly's registers.
                    constexpr bool lean_g = R > 8;
                    cplx g[R];
                    if constexpr (!lean_g) {
                        // g[k] = g[1]^k by products (k = 2: g1*g1, 3: g2*g1, 4: g2*g2, 5: g4*g1, ...:
                        // at most three roundings) instead of two scattered table reads per k, which
                        // miss the small L1 left beside the tiles (K_A 7.32 -> 6.81 us/pair)
                        static_assert(R <= 8, "power chain written for k < 8");
                        g[1] = tw2(p.m_lo, p.m_hi, n2 * (unsigned)Wt);
                        static_for<2, R>([&](auto K) {
                            constexpr int k = decltype(K)::value;
                            g[k] = (k % 2 == 0) ? cmul(g[k / 2], g[k / 2]) : cmul(g[k - 1], g[1]);
                        });
                    } else {
                        static_for<1, R>([&](auto K) {
                            constexpr int k = decltype(K)::value;
                            if constexpr (!lean_g || (k & (k - 1)) == 0)
                                g[k] = tw2(p.m_lo, p.m_hi, n2 * (unsigned)(Wt * k));
                        });
                    }
                    // The twiddle loads of a chunk of items are issued together ahead of the
                    // butterflies (three dependent table reads per item would otherwise be exposed
                    // once per item: the tables do not stay in the small L1 left beside the tiles).
                    constexpr int ITER = (items + NT - 1) / NT;
                    constexpr int CH = ITER <= 6 ? ITER : 4;
                    // STEP: consecutive items of a thread are NT/16 blocks apart; when that is a
                    // whole number MSTEP of units of the leading digit (M1/r0 positions), the bin
                    // f0 advances by MSTEP per item and W_M^(n2*f0) by the per-thread constant
                    // W_M^(n2*MSTEP): one product per item instead of the digit reversal, three
                    // table reads (L2 latency) and two products (K_A 7.87 -> 7.31 us/pair).
                    constexpr int DB = NT / COL_T, UNIT = RL::stride(0) / R;
                    constexpr bool STEP = ITER > 1 && DB % UNIT == 0;
                    constexpr int MSTEP = STEP ? DB / UNIT : 0;
                    [[maybe_unused]] int f0_run = 0;
                    [[maybe_unused]] cplx t0_run = cmake(1.f, 0.f), gstep = cmake(1.f, 0.f);
                    if constexpr (STEP) {
                        f0_run = RL::freq_of_pos(((tid < items ? tid : 0) >> 4) * R);
                        t0_run = cmul(ldg(p.tc + f0_run * COL_T + c), tw2(p.m_lo, p.m_hi, (unsigned)c0 * (unsigned)f0_run));
                        gstep = tw2(p.m_lo, p.m_hi, n2 * (unsigned)MSTEP);
                    }
                    for (int it0 = 0; it0 < ITER; it0 += CH) {
                        int f0s[CH];
                        cplx t0s[CH];
                        static_for<0, CH>([&](auto I) {
                            constexpr int i = decltype(I)::value;
                            if constexpr (STEP) {
                                f0s[i] = f0_run;
                                t0s[i] = t0_run;
                                f0_run += MSTEP;
                                t0_run = cmul(t0_run, gstep);
                            } else {
                                const int w = tid + (it0 + i) * NT;
                                f0s[i] = RL::freq_of_pos(((w < items ? w : 0) >> 4) * R);
                                t0s[i] = cmul(ldg(p.tc + f0s[i] * COL_T + c),
                                              tw2(p.m_lo, p.m_hi, (unsigned)c0 * (unsigned)f0s[i]));
                            }
                        });
                        static_for<0, CH>([&](auto I) {
                            constexpr int i = decltype(I)::value;
                            const int w = tid + (it0 + i) * NT;
                            if (w < items) {
                                const int i0 = (w >> 4) * R;
                                cplx v[R];
                                static_for<0, R>([&](auto Q) {
                                    constexpr int q = decltype(Q)::value;
                                    v[q] = buf[(i0 + q) * COL_T + c];
                                });
                                dft_reg<R, -1>(v);
                                const cplx t0 = t0s[i];
                                cplx* __restrict__ o = out + ((unsigned)f0s[i] * (unsigned)M2 + n2);   // < M < 2^31
                                o[0] = cmul(v[0], t0);
                                static_for<1, R>([&](auto K) {
                                    constexpr int k = decltype(K)::value;
                                    cplx gk;
                                    if constexpr (!lean_g || (k & (k - 1)) == 0) {
                                        gk = g[k];
                                    } else {
                                        constexpr int hb = (k >= 16) ? 16 : (k >= 8) ? 8 : (k >= 4) ? 4 : 2;
                                        constexpr int rest = k - hb;
                                        if constexpr ((rest & (rest - 1)) == 0) {
                                            gk = cmul(g[hb], g[rest]);
                                        } else {
                                            constexpr int hb2 = (rest >= 8) ? 8 : (rest >= 4) ? 4 : 2;
                                            constexpr int rest2 = rest - hb2;
                                            static_assert(R <= 24, "k < 24: at most four one-bits, and then the last two are 2 + 1");
                                            if constexpr ((rest2 & (rest2 - 1)) == 0) gk = cmul(g[hb], cmul(g[hb2], g[rest2]));
                                            else gk = cmul(cmul(g[hb], g[hb2]), cmul(g[rest2 & ~1], g[1]));
                                        }
                                    }
                                    o[(size_t)k * Wt * M2] = cmul(v[k], cmul(t0, gk));
                                });
                            }
                        });
                    }
                }
            });
        });
    }
};

// --------------------------------------------------------------------- K_C
// The tile is staged with boxes of a tensor map over plane 0 (rows 0 .. M1-2; the last row and
// the mbarrier as in ColFwdKernel).  TMA staging is the only path; the TMA parameter is kept,
// fixed to true, so that callers which name ColInvKernel<..., true> (tests/emu) keep building.
template <class RL, int M2_, int NT, bool TMA = true>
struct ColInvKernel {
    static_assert(TMA, "K_C's tiles are always staged by the TMA unit");
    static constexpr int M1 = RL::n;
    static constexpr int M2 = M2_;
    static constexpr int P = RL::count;
    static constexpr int THREADS = NT;
    static constexpr size_t SMEM = (size_t)M1 * COL_T * sizeof(cplx);
    static constexpr int MIN_CTAS = ctas_per_sm(SMEM, NT);
    static_assert(NT % COL_T == 0, "a thread must keep its column across items");
    static_assert(NT % 32 == 0, "the argmax epilogue votes per warp");
    static_assert(P >= 2, "column plans need at least two passes");

    struct Params {
        const cplx* planes;      // [pair][2][M1*M2]; plane 0 holds the K_B output
        PairPeak* peaks;         // [pair]
        const cplx* tw;          // RL pass tables (forward sign; conjugated here)
        long long L;
        CUtensorMap tm;          // [2 * pair][M1 rows][2*M2 floats] view of the planes
    };
    static constexpr int TMA_ROWS = M1 - 1;

    // grid = (pairs, M2 / 16): the pair index runs fastest, so the tiles of one pair are
    // spread over the launch and later tiles see the running maximum of earlier ones.
    template <class Ex>
    static ASC_HD void run(Ex& ex, const Params& p, cplx* __restrict__ buf) {
        const int c0 = ex.by() * COL_T;
        const long long pair = ex.bx();
        const long long M = p.L;
        const cplx* __restrict__ in = p.planes + pair * 2 * M;

        // stage the tile
        void* mbar = reinterpret_cast<char*>(buf) + SMEM - 8;
        ex.phase([&](int tid) {
            if (tid == 0) mbar_init(mbar, 1);
        });
        ex.phase([&](int tid) {
            if (tid == 0) {
                constexpr int NB = tile_boxes(TMA_ROWS), BR = tile_box_rows(TMA_ROWS);
                constexpr size_t pitch = (size_t)M2 * sizeof(cplx);
                const char* __restrict__ raw = reinterpret_cast<const char*>(in + c0);
                mbar_expect_tx(mbar, (unsigned)(NB * BR * 128));
                static_for<0, NB>([&](auto I) {
                    constexpr int r0 = tile_box_start(TMA_ROWS, decltype(I)::value);
                    tma_load_rows(buf + r0 * COL_T, &p.tm, 2 * c0, r0, (int)(2 * pair), mbar, raw + r0 * pitch, pitch, BR);
                });
            }
            mbar_wait(mbar, 0);
        });

        static_for<0, P - 1>([&](auto PP) {
            constexpr int ps = decltype(PP)::value;
            constexpr int R = RL::r(ps);
            constexpr int S = RL::stride(ps);
            constexpr int items = (M1 / R) * COL_T;
            ex.phase([&](int tid) {
                const int c = tid & (COL_T - 1);
                cplx t[R];
                for (int w = tid; w < items; w += NT) {
                    const int bf = w >> 4;
                    const int blk = (S * R == M1) ? 0 : bf / S;    // pass 0: one block
                    const int j = bf - blk * S;
                    const int i0 = blk * (S * R) + j;
                    cplx v[R];
                    static_for<0, R>([&](auto Q) {
                        constexpr int q = decltype(Q)::value;
                        if constexpr (ps == 0 && q == R - 1) {
                            // tile row M1 - 1 is not staged (the mbarrier sits there)
                            if (i0 == S - 1) v[q] = ldg(in + ((long long)(M1 - 1) * M2 + c0 + c));
                            else v[q] = buf[(i0 + q * S) * COL_T + c];
                        } else {
                            v[q] = buf[(i0 + q * S) * COL_T + c];
                        }
                    });
                    if constexpr (ps == 0) {
                        if (i0 == S - 1 && c == COL_T - 1) mbar_inval(mbar);   // overwritten below
                    }
                    dft_reg<R, +1>(v);
                    pass_twiddles<R>(p.tw + RL::tw_offset(ps), S, j, t);
                    buf[i0 * COL_T + c] = v[0];
                    static_for<1, R>([&](auto K) {
                        constexpr int k = decltype(K)::value;
                        buf[(i0 + k * S) * COL_T + c] = cmulc(v[k], t[k]);
                    });
                }
            });
        });

        // last pass + argmax epilogue: packed point n = n1*M2 + n2 carries
        // r[2n] (real part) and r[2n+1] (imaginary part).
        //
        // Only values that reach the running SECOND peak can matter (they may become the
        // peak or the second peak), so a butterfly's 2R outputs are first reduced with fmax
        // and compared with a threshold; the exact key logic runs only when the test passes.
        // The threshold starts from the pair's running second peak in global memory (earlier
        // CTAs of this launch) and is raised to the warp's own bound after every hit, so the
        // slow path is taken O(log) times per warp.
        {
            constexpr int ps = P - 1;
            constexpr int R = RL::r(ps);
            constexpr int Wt = RL::weight(ps);
            constexpr int items = (M1 / R) * COL_T;
            ex.phase_argmax(
                [&](int tid) -> ArgmaxPair {
                    ArgmaxAcc acc;
                    const unsigned int seen = ex.peek_bits(&p.peaks[pair].second_bits);
                    if (seen != 0u) acc.thr = float_from_order_bits(seen);
                    const int c = tid & (COL_T - 1);
                    const bool col0 = (c0 + c) == 0;
                    for (int w0 = 0; w0 < items; w0 += NT) {      // warp-uniform trip count
                        const int w = w0 + tid;
                        const bool act = w < items;
                        const int blk = (act ? w : 0) >> 4;
                        const int i0 = blk * R;
                        cplx v[R];
                        static_for<0, R>([&](auto Q) {
                            constexpr int q = decltype(Q)::value;
                            v[q] = buf[(i0 + q) * COL_T + c];
                        });
                        dft_reg<R, +1>(v);
                        float gm = fmaxf(fabsf(v[0].x), fabsf(v[0].y));
                        static_for<1, R>([&](auto K) {
                            constexpr int k = decltype(K)::value;
                            gm = fmaxf(gm, fmaxf(fabsf(v[k].x), fabsf(v[k].y)));
                        });
                        const bool has_seed = col0 && i0 == 0;      // r[0]: signed seed, exact path always
                        const bool need = act && (gm >= acc.thr || has_seed);
                        if (ex.any(need)) {
                            if (need) {
                                const int f0 = RL::freq_of_pos(i0);
                                static_for<0, R>([&](auto K) {
                                    constexpr int k = decltype(K)::value;
                                    const int n1 = f0 + k * Wt;
                                    const uint32_t i_re = 2u * ((uint32_t)n1 * (uint32_t)M2 + (uint32_t)(c0 + c));
                                    if (has_seed && n1 == 0) acc.consider_seed(v[k].x, &p.peaks[pair]);
                                    else acc.consider(v[k].x, i_re);
                                    acc.consider(v[k].y, i_re + 1u);
                                });
                            }
                            acc.thr = fmaxf(acc.thr, ex.warp_second(acc.best_mag(), acc.second));
                        }
                    }
                    return acc.result();
                },
                &p.peaks[pair].key, &p.peaks[pair].second_bits, buf);
        }
    }
};

// --------------------------------------------------------------------- K_B
// The pair (k, M-k) computation shared by the fused row kernel and the
// single-CTA short-length kernel.
//   a = Zs[k], b = Zs[M-k], c = Zp[k], d = Zp[M-k], w = exp(-2*pi*i*k/N).
//   2X[k] = s + u,  2X[M-k] = conj(s - u)  with s = a + conj b, u = w*(-i)(a - conj b)
//   p1 = 4 P[k] = 2X[k] conj(2Y[k]);  p2 = conj(4 P[M-k]) = (s-u) conj(s'-u')
//   Q[k] = ((p1+p2) + i conj(w)(p1-p2)) / 4;  Q[M-k] = conj((p1+p2) - i conj(w)(p1-p2)) / 4
ASC_HD void split_mul_merge(cplx a, cplx b, cplx c, cplx d, cplx w, cplx& qk, cplx& qmk) {
    const cplx s = cmake(a.x + b.x, a.y - b.y);
    const cplx t = cmake(a.x - b.x, a.y + b.y);
    const cplx u = cmul(w, cmake(t.y, -t.x));
    const cplx s2 = cmake(c.x + d.x, c.y - d.y);
    const cplx t2 = cmake(c.x - d.x, c.y + d.y);
    const cplx u2 = cmul(w, cmake(t2.y, -t2.x));
    const cplx p1 = cmulc(cadd(s, u), cadd(s2, u2));
    const cplx p2 = cmulc(csub(s, u), csub(s2, u2));
    const cplx g = cadd(p1, p2);
    const cplx e = csub(p1, p2);
    // h = i * conj(w) * e
    const cplx ce = cmulc(e, w);
    const cplx h = cmake(-ce.y, ce.x);
    qk = cmake(0.25f * (g.x + h.x), 0.25f * (g.y + h.y));
    qmk = cmake(0.25f * (g.x - h.x), -0.25f * (g.y - h.y));
}

// The same step with the twiddle folded: with s = a + conj b, t = a - conj b (and s', t' from
// c, d), u = -i w t gives u conj(u') = t conj(t') and
//   (p1 + p2) / 2 = G = s conj(s') + t conj(t')
//   i conj(w) (p1 - p2) / 2 = H = t conj(s') - conj(w^2) s conj(t')
// so only w^2 = exp(-2*pi*i*k/M) is needed.  Returns 2 Q[k] = G + H and 2 Q[M-k] = conj(G - H):
// the caller folds the factor 1/2 into a later twiddle.  18 packed instructions instead of 34.
// C: cplx (the product) or cplxd (the runtime-radix kernels' fp64 mode).
template <class C>
ASC_HD void split_mul_merge_w2(C a, C b, C c, C d, C w2, C& qk2, C& qmk2) {
    const C s = cconj_add(a, b), t = cconj_sub(a, b);
    const C s2 = cconj_add(c, d), t2 = cconj_sub(c, d);
    const C g = cmulc_acc(t, t2, cmulc(s, s2));
    const C x = cmulc(s, t2);
    const C h = cmulc_nacc(x, w2, cmulc(t, s2));
    qk2 = cadd(g, h);
    const C e = csub(g, h);
    qmk2 = cmake(e.x, -e.y);
}

// GCC-PHAT weighting: one spectrum value as a unit phasor, 0 where its squared magnitude is 0.
// The value is first scaled by the power of two that brings its larger component into [1, 2):
// exact, it keeps the squares in range at any input level, and it makes the phasor a function of
// the value's direction alone, so that scaling either input by a power of two leaves the weighted
// correlation unchanged bit for bit.
ASC_HD float phat_rsqrt(float q) {
#if defined(__CUDA_ARCH__)
    return rsqrtf(q);
#else
    return 1.0f / sqrtf(q);
#endif
}
ASC_HD double phat_rsqrt(double q) {
#if defined(__CUDA_ARCH__)
    return rsqrt(q);
#else
    return 1.0 / sqrt(q);
#endif
}
ASC_HD cplx unit_phasor(cplx z) {
    const float m = fmaxf(fabsf(z.x), fabsf(z.y));
    uint32_t b;
    memcpy(&b, &m, 4);
    int e = (int)(b >> 23);                                   // m in [2^(e-127), 2^(e-126))
    e = e < 1 ? 1 : (e > 253 ? 253 : e);
    const uint32_t sb = (uint32_t)(254 - e) << 23;            // 2^(127 - e)
    float s;
    memcpy(&s, &sb, 4);
    const float x = z.x * s, y = z.y * s;
    const float q = fmaf(x, x, y * y);
    const float r = q > 0.0f ? phat_rsqrt(q) : 0.0f;
    return cmake(x * r, y * r);
}
ASC_HD cplxd unit_phasor(cplxd z) {
    const double m = fmax(fabs(z.x), fabs(z.y));
    uint64_t b;
    memcpy(&b, &m, 8);
    int e = (int)(b >> 52);                                   // m in [2^(e-1023), 2^(e-1022))
    e = e < 1 ? 1 : (e > 2045 ? 2045 : e);
    const uint64_t sb = (uint64_t)(2046 - e) << 52;           // 2^(1023 - e)
    double s;
    memcpy(&s, &sb, 8);
    const double x = z.x * s, y = z.y * s;
    const double q = fma(x, x, y * y);
    const double r = q > 0.0 ? phat_rsqrt(q) : 0.0;
    return cmake(x * r, y * r);
}

// The PHAT form of the split / multiply / merge step: W[k] = X[k] conj(Y[k]) / (|X[k]| |Y[k]|) takes
// the place of the product.  Whitening needs X and Y themselves, hence w = exp(-2*pi*i*k/N) rather
// than w^2: 2X[k] = s + u and conj(2X[M-k]) = s - u with u = -i w t (s, t from a, b as in
// split_mul_merge_w2; Y from c, d alike).  X and Y are normalised separately (unit_phasor), then
// p1 = W[k], p2 = conj(W[M-k]) are merged as in split_mul_merge.  SCALE is the output convention of
// the step this replaces: 1 gives Q[k] (split_mul_merge), 2 gives 2 Q[k] (split_mul_merge_w2), so
// that the inverse passes, the argmax and peak_scale are those of the unweighted path.
template <int SCALE, class C>
ASC_HD void split_phat_merge(C a, C b, C c, C d, C w, C& qk, C& qmk) {
    static_assert(SCALE == 1 || SCALE == 2, "output convention of split_mul_merge or split_mul_merge_w2");
    const C s = cconj_add(a, b), t = cconj_sub(a, b);
    const C s2 = cconj_add(c, d), t2 = cconj_sub(c, d);
    const C u = cmul_ni(cmul(w, t)), u2 = cmul_ni(cmul(w, t2));
    const C p1 = cmulc(unit_phasor(cadd(s, u)), unit_phasor(cadd(s2, u2)));
    const C p2 = cmulc(unit_phasor(csub(s, u)), unit_phasor(csub(s2, u2)));
    C g = cadd(p1, p2);
    C h = cmul_pi(cmulc(csub(p1, p2), w));                    // i conj(w) (p1 - p2)
    if constexpr (SCALE == 2) {
        g = cadd(g, g);
        h = cadd(h, h);
    }
    qk = cadd(g, h);
    const C e = csub(g, h);
    qmk = cmake(e.x, -e.y);
}

// PHAT: the forward spectra are whitened in the split step (split_phat_merge) and the rest of the
// kernel is unchanged.  Params::rev, m_lo and m_hi then hold the split's half-angle tables,
// exp(-2*pi*i*freq_of_pos(e)/(2*M2)) and W_N (N = 2M), so that w = W_N^k1 * rev[e] factors like w^2.
template <class RL, int M1_, int NT, bool PHAT = false>
struct RowFusedKernel {
    static constexpr int M2 = RL::n;
    static constexpr int M1 = M1_;  // 0: the number of rows is a launch parameter (Params::m1) -- the rows of a
                                    // runtime-radix plan whose row length has a static kernel (gen_plan.h)
    static constexpr int P = RL::count;
    static constexpr int THREADS = NT;
    static constexpr int RP = M2;   // row pitch in shared memory
    static constexpr size_t SMEM = (size_t)4 * RP * sizeof(cplx);
    static constexpr int MIN_CTAS = ctas_per_sm(SMEM, NT);
    static constexpr int R0 = RL::r(0);
    static constexpr int S0 = RL::stride(0);
    static_assert(M2 % 2 == 0, "row length must be even (16-byte chunks, bulk store size)");
    static_assert(P >= 2, "row plans need at least two passes");
    static_assert(S0 * R0 == M2 && S0 >= 16, "pass 0 must own the last two points of a row as its last two items");

    // A pass whose sub-stride S is below 16 (but not 1) would have half-warps
    // straddle blocks and collide in the banks; give each block 16 thread slots
    // (S active) instead.  S == 1 passes must use an odd radix (conflict-free).
    static constexpr int slots(int S) { return (S > 1 && S < 16) ? 16 : S; }

    struct Params {
        cplx* planes;            // [pair][2][M1*M2]
        const cplx* tw;          // RL pass tables (forward sign, power-of-two multiples)
        const cplx* rev;         // [M2]: exp(-2*pi*i*freq_of_pos(e)/M2), position order
        const cplx* m_lo;        // W_M tables
        const cplx* m_hi;
        long long L;
        const cplx* rtab;        // [M1][TABP]: per row k1 the final-pass tables (fft_plan.h: build_row_tab)
        int m1 = 0;              // rows per plane when M1_ == 0
    };
    // Final-pass twiddle tables of one row k1: S0 entries 0.5 * W_M^(j*k1) (the factor 1/2 of the
    // merge step rides here, exactly), then R0 entries W_M^(k*S0*k1); padded to an even count so
    // that a row is a whole number of 16-byte units for the bulk copy.
    static constexpr int TABP = (S0 + R0 + 1) & ~1;
    // split phase: thread (a, b) = (tid / 64, tid % 64) of an A x 64 grid over (d0, e1)
    static_assert(NT % 64 == 0, "the split phase maps threads to an (NT/64) x 64 grid");
    static constexpr int SPLIT_A = NT / 64;
    static constexpr int SPLIT_XN = (R0 + SPLIT_A - 1) / SPLIT_A;
    static constexpr int SPLIT_MN = (S0 + 63) / 64;
    static_assert(2 * TABP + 1 <= 2 * RP, "final-pass twiddle tables and their mbarrier must fit the dead sample rows");

    // grid = (M1/2 + 1, 1, pairs); CTA r owns rows r and M1 - r.
    template <class Ex>
    static ASC_HD void run(Ex& ex, const Params& p, cplx* __restrict__ buf) {
        const int r = ex.bx();
        const long long pair = ex.bz();
        const long long M = p.L;
        const int m1 = M1 > 0 ? M1 : p.m1;
        const bool two = (r != 0) && (2 * r != m1);
        const int nrows = two ? 2 : 1;
        const int k1a = r, k1b = m1 - r;   // k1b unused when !two
        cplx* __restrict__ plane_s = p.planes + pair * 2 * M;
        cplx* __restrict__ plane_p = plane_s + M;
        // final-pass twiddle tables of the two rows, copied into the (then dead) sample rows
        cplx* __restrict__ tab = buf + 2 * RP;                // [2][TABP]
        void* tabbar = buf + 2 * RP + 2 * TABP;               // mbarrier of that copy

        // ---- stage the 2*nrows rows.  smem slots: 0,1 source rows; 2,3 sample rows.
        // Four bulk copies of the TMA unit, issued by one thread, awaited by all.
        // The CTA's shared memory is exactly the four rows, so the 8-byte mbarrier sits on the
        // last point of slot 3; the last two points of that row are not staged -- forward pass 0
        // reads them from global memory instead -- and the thread whose butterfly writes them
        // first invalidates the barrier.
        {
            void* mbar = buf + 4 * RP - 1;
            ex.phase([&](int tid) {
                if (tid == 0) mbar_init(mbar, 1);
            });
            ex.phase([&](int tid) {
                if (tid == 0) {
                    constexpr unsigned full = (unsigned)(M2 * sizeof(cplx));
                    mbar_expect_tx(mbar, two ? 4u * full - 16u : 2u * full);
                    bulk_load(buf, plane_s + (long long)k1a * M2, full, mbar);
                    bulk_load(buf + 2 * RP, plane_p + (long long)k1a * M2, full, mbar);
                    if (two) {
                        bulk_load(buf + RP, plane_s + (long long)k1b * M2, full, mbar);
                        bulk_load(buf + 3 * RP, plane_p + (long long)k1b * M2, full - 16u, mbar);
                    }
                }
                mbar_wait(mbar, 0);
            });
        }

        // ---- forward DIF on 2*nrows rows.  One pass over the nb rows in shared-memory slots
        // slot0, slot0 + sstep, ... by threads t = 0 .. nt-1.
        auto fwd_pass = [&](auto PP, int t, int nt, int slot0, int sstep, int nb) {
            constexpr int ps = decltype(PP)::value;
            constexpr int R = RL::r(ps);
            constexpr int S = RL::stride(ps);
            constexpr int SL = slots(S);
            constexpr int per_row = (M2 / (S * R)) * SL;
            const int items = per_row * nb;
            // pass 0: items (slot 3, i0 = S-2) and (slot 3, i0 = S-1) are the last two of a call
            // whose last row is slot 3
            [[maybe_unused]] const int tail_w = (slot0 + (nb - 1) * sstep == 3) ? items - 2 : 0x7fffffff;
            {
                for (int w = t; w < items; w += nt) {
                    const int bw = w / per_row;
                    const int bf = w - bw * per_row;
                    const int blk = (per_row == SL) ? 0 : bf / SL;   // pass 0: one block per row
                    const int j = bf - blk * SL;
                    if (SL != S && j >= S) continue;
                    cplx* __restrict__ row = buf + (slot0 + bw * sstep) * RP;
                    const int i0 = blk * (S * R) + j;
                    cplx v[R];
                    static_for<0, R>([&](auto Q) {
                        constexpr int q = decltype(Q)::value;
                        v[q] = row[i0 + q * S];
                    });
                    if constexpr (ps == 0) {
                        // the two points of slot 3 the staging left out (see above): the last two
                        // items of the pass; what the shared-memory read returned for them was the
                        // barrier's bytes
                        if (w >= tail_w) {
                            v[R - 1] = ldg(plane_p + (long long)k1b * M2 + (i0 + (R - 1) * S));
                            if (w == tail_w + 1) mbar_inval(buf + 4 * RP - 1);   // this thread overwrites it below
                        }
                    }
                    dft_reg<R, -1>(v);
                    row[i0] = v[0];
                    if constexpr (S > 1) {
                        cplx t[R];
                        pass_twiddles<R>(p.tw + RL::tw_offset(ps), S, j, t);
                        static_for<1, R>([&](auto K) {
                            constexpr int k = decltype(K)::value;
                            row[i0 + k * S] = cmul(v[k], t[k]);
                        });
                    } else {
                        static_for<1, R>([&](auto K) {
                            constexpr int k = decltype(K)::value;
                            row[i0 + k] = v[k];
                        });
                    }
                }
            }
        };
        static_for<0, P>([&](auto PP) {
            ex.phase([&](int tid) { fwd_pass(PP, tid, NT, 0, two ? 1 : 2, 2 * nrows); });   // slots 0,1,2,3 or 0,2
        });

        // ---- split + conj-multiply + merge, in place into the source rows.
        {
            // two rows -> every position e of row a pairs with position M2-1-e of row b
            // (bin M2-1-k2); row M1/2 alone -> same map inside one row, e < M2/2; row 0
            // alone -> bins (k2, M2-k2), e <= M2/2.
            // w^2 = exp(-2*pi*i*(k1a + M1*k2)/M) = W_M^k1a * rev[position of k2].
            ex.phase([&](int tid) {
                const cplx wk1 = tw2(p.m_lo, p.m_hi, (unsigned)k1a);
                if (two) {
                    cplx* __restrict__ zs_a = buf;
                    cplx* __restrict__ zs_b = buf + RP;
                    cplx* __restrict__ zp_a = buf + 2 * RP;
                    cplx* __restrict__ zp_b = buf + 3 * RP;
                    // Position e = d0*S0 + e1 (d0 < R0, e1 < S0) holds bin d0 + freq_of_pos(e1), so
                    // rev[e] = rev[d0*S0] * rev[e1].  Thread (a, b) = (tid / 64, tid % 64) takes
                    // d0 = a, a + A, ... and e1 = b, b + 64, ...: its w^2 values are products of
                    // SPLIT_XN + SPLIT_MN per-thread constants read once from the first S0 (+ R0
                    // strided) entries of rev -- 2 KB that stay in L1 -- instead of one read of the
                    // whole 19 KB table from L2 per item.  Lanes still walk contiguous positions.
                    cplx ax[SPLIT_XN], cm[SPLIT_MN];
                    const int sa = tid >> 6, sb = tid & 63;
                    static_for<0, SPLIT_XN>([&](auto X) {
                        const int d0 = sa + decltype(X)::value * SPLIT_A;
                        ax[decltype(X)::value] = cmul(ldg(p.rev + (d0 < R0 ? d0 : 0) * S0), wk1);
                    });
                    static_for<0, SPLIT_MN>([&](auto Mm) {
                        const int e1 = sb + decltype(Mm)::value * 64;
                        cm[decltype(Mm)::value] = ldg(p.rev + (e1 < S0 ? e1 : 0));
                    });
                    static_for<0, SPLIT_MN>([&](auto Mm) {
#if defined(__CUDA_ARCH__)
                        // compiler fence after every second e1 step: four items in flight per
                        // thread (no fence: +0.14 us/pair, a fence after every step: +0.1)
                        if constexpr (decltype(Mm)::value > 0 && decltype(Mm)::value % 2 == 0)
                            asm volatile("" ::: "memory");
#endif
                        static_for<0, SPLIT_XN>([&](auto X) {
                            const int d0 = sa + decltype(X)::value * SPLIT_A;
                            const int e1 = sb + decltype(Mm)::value * 64;
                            if (d0 < R0 && e1 < S0) {
                                const int e = d0 * S0 + e1;
                                const int pb = M2 - 1 - e;
                                const cplx w2 = cmul(ax[decltype(X)::value], cm[decltype(Mm)::value]);
                                cplx qk, qmk;
                                if constexpr (PHAT) split_phat_merge<2>(zs_a[e], zs_b[pb], zp_a[e], zp_b[pb], w2, qk, qmk);
                                else split_mul_merge_w2(zs_a[e], zs_b[pb], zp_a[e], zp_b[pb], w2, qk, qmk);
                                zs_a[e] = qk;
                                zs_b[pb] = qmk;
                            }
                        });
                    });
                } else {
                    cplx* __restrict__ zs = buf;
                    cplx* __restrict__ zp = buf + 2 * RP;
                    const int items = r == 0 ? M2 / 2 + 1 : M2 / 2;
                    for (int e = tid; e < items; e += NT) {
                        int pa, pb;
                        if (r == 0) {
                            pa = RL::pos_of_freq(e);
                            pb = RL::pos_of_freq(e == 0 ? 0 : M2 - e);
                        } else {
                            pa = e;
                            pb = M2 - 1 - e;
                        }
                        const cplx w2 = cmul(ldg(p.rev + pa), wk1);
                        cplx qk, qmk;
                        if constexpr (PHAT) split_phat_merge<2>(zs[pa], zs[pb], zp[pa], zp[pb], w2, qk, qmk);
                        else split_mul_merge_w2(zs[pa], zs[pb], zp[pa], zp[pb], w2, qk, qmk);
                        zs[pa] = qk;
                        if (pa != pb) zs[pb] = qmk;
                    }
                }
            });
        }

        // ---- the sample rows are dead now: the TMA unit fetches the final-pass twiddle tables of
        // the two rows into them while the first inverse passes run (waited for in the last one).
        ex.single([&]() {
            constexpr unsigned bytes = (unsigned)(TABP * sizeof(cplx));
            mbar_init(tabbar, 1);
            mbar_expect_tx(tabbar, (unsigned)nrows * bytes);
            bulk_load(tab, p.rtab + (long long)k1a * TABP, bytes, tabbar);
            if (two) bulk_load(tab + TABP, p.rtab + (long long)k1b * TABP, bytes, tabbar);
        });

        // ---- inverse DIT on nrows rows (slots 0,1), passes P-1 .. 0.  One pass over rows
        // r0 .. r0+nr-1 by threads t = 0 .. nt-1.
        auto inv_pass = [&](auto PP, int t, int nt, int r0, int nr) {
            constexpr int ps = P - 1 - decltype(PP)::value;
            constexpr int R = RL::r(ps);
            constexpr int S = RL::stride(ps);
            constexpr int SL = slots(S);
            constexpr bool last = ps == 0;
            constexpr int per_row = (M2 / (S * R)) * SL;
            const int items = per_row * nr;
            {
                if constexpr (last) mbar_wait(tabbar, 0);      // the tables requested after the split have landed
                for (int w = t; w < items; w += nt) {
                    const int rw = w / per_row;
                    const int rr = r0 + rw;
                    const int bf = w - rw * per_row;
                    const int blk = (per_row == SL) ? 0 : bf / SL;   // pass 0: one block per row
                    const int j = bf - blk * SL;
                    if (SL != S && j >= S) continue;
                    cplx* __restrict__ row = buf + rr * RP;
                    const int i0 = blk * (S * R) + j;
                    cplx v[R];
                    v[0] = row[i0];
                    if constexpr (S > 1) {
                        cplx t[R];
                        pass_twiddles<R>(p.tw + RL::tw_offset(ps), S, j, t);
                        static_for<1, R>([&](auto Q) {
                            constexpr int q = decltype(Q)::value;
                            v[q] = cmulc(row[i0 + q * S], t[q]);
                        });
                    } else {
                        static_for<1, R>([&](auto Q) {
                            constexpr int q = decltype(Q)::value;
                            v[q] = row[i0 + q];
                        });
                    }
                    dft_reg<R, +1>(v);
                    if constexpr (!last) {
                        static_for<0, R>([&](auto K) {
                            constexpr int k = decltype(K)::value;
                            row[i0 + k * S] = v[k];
                        });
                    } else {
                        // natural order n2 = j + k*S0; conj W_M^(n2*k1) = conj(ab[j] * g[k]); in place
                        const cplx t0 = tab[rr * TABP + j];
                        row[j] = cmulc(v[0], t0);
                        static_for<1, R>([&](auto K) {
                            constexpr int k = decltype(K)::value;
                            row[j + k * S] = cmulc(v[k], cmul(t0, tab[rr * TABP + S0 + k]));
                        });
                    }
                }
                if constexpr (last) fence_async_proxy();   // rows are read by the bulk store below
            }
        };
        static_for<0, P>([&](auto PP) {
            ex.phase([&](int tid) { inv_pass(PP, tid, NT, 0, nrows); });
        });

        // ---- the product rows leave through the TMA unit, back in place (row k1 of plane 0).
        ex.single([&]() {
            bulk_store(plane_s + (long long)k1a * M2, buf, (unsigned)(M2 * sizeof(cplx)));
            if (two) bulk_store(plane_s + (long long)k1b * M2, buf + RP, (unsigned)(M2 * sizeof(cplx)));
            bulk_store_commit_and_drain();
        });
    }
};

// ------------------------------------------------------------- device entry
// Executor used on the GPU.  Methods are __host__ __device__ only so that the
// kernel bodies (shared with the CPU emulator) instantiate cleanly; the host
// side of them is never called.
struct DeviceExec {
    // Block coordinates the kernel body sees (the entry copies blockIdx).
    int x_ = 0, y_ = 0, z_ = 0;
    ASC_HD int bx() const { return x_; }
    ASC_HD int by() const { return y_; }
    ASC_HD int bz() const { return z_; }
    template <class F>
    ASC_HD void phase(F&& f) {
#if defined(__CUDA_ARCH__)
        f((int)threadIdx.x);
        __syncthreads();
#endif
    }
    // f() on one thread of the CTA, after the barrier of the preceding phase.
    template <class F>
    ASC_HD void single(F&& f) {
#if defined(__CUDA_ARCH__)
        if (threadIdx.x == 0) f();
#endif
    }
    // warp vote / warp maximum of a non-negative threshold (negative or NaN counts as 0);
    // every lane of the warp must call them.
    ASC_HD bool any(bool b) const {
#if defined(__CUDA_ARCH__)
        return __any_sync(0xffffffffu, b);
#else
        return b;
#endif
    }
    // Second largest of the warp's (best magnitude, second) pairs: the largest value among
    // every lane's `second` and every lane's best magnitude except ONE lane holding the
    // warp maximum -- a lower bound of the pair's final second peak.  Inputs are >= 0.
    ASC_HD float warp_second(float best_mag, float second) const {
#if defined(__CUDA_ARCH__)
        const unsigned bm = __float_as_uint(fmaxf(best_mag, 0.0f));
        const unsigned top = __reduce_max_sync(0xffffffffu, bm);
        const unsigned holders = __ballot_sync(0xffffffffu, bm == top);
        const bool winner = (threadIdx.x & 31u) == (unsigned)(__ffs(holders) - 1);
        const float cand = winner ? second : fmaxf(second, best_mag);
        return __uint_as_float(__reduce_max_sync(0xffffffffu, __float_as_uint(fmaxf(cand, 0.0f))));
#else
        (void)best_mag;
        return second;
#endif
    }
    // current value of a key / bit pattern other CTAs of this launch update with atomicMax
    ASC_HD unsigned long long peek_key(const unsigned long long* k) const {
#if defined(__CUDA_ARCH__)
        return __ldcg(k);
#else
        return *k;
#endif
    }
    ASC_HD unsigned int peek_bits(const unsigned int* k) const {
#if defined(__CUDA_ARCH__)
        return __ldcg(k);
#else
        return *k;
#endif
    }
    // CTA-wide (peak key, second peak) of the per-thread pairs (argmax_merge), then one
    // atomicMax on *dst and one on *dst_second.  `scratch`: at least 32 * 12 bytes of the CTA's
    // dynamic shared memory; it may alias data f() reads (a barrier separates the two uses).
    // No static shared memory, so the column kernels keep 3 CTAs per SM.
    template <class F>
    ASC_HD void phase_argmax(F&& f, unsigned long long* dst, unsigned int* dst_second, void* scratch) {
#if defined(__CUDA_ARCH__)
        unsigned long long* s_best = reinterpret_cast<unsigned long long*>(scratch);   // [32]
        float* s_sec = reinterpret_cast<float*>(s_best + 32);                          // [32]
        const ArgmaxPair mine = f((int)threadIdx.x);
        unsigned long long best = mine.best;
        float second = mine.second;
        for (int o = 16; o > 0; o >>= 1)
            argmax_merge(best, second, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, second, o));
        const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
        const int nw = (blockDim.x + 31) >> 5;
        __syncthreads();                      // every warp is done reading what `scratch` aliases
        if (lane == 0) { s_best[wid] = best; s_sec[wid] = second; }
        __syncthreads();
        if (wid == 0) {
            best = lane < nw ? s_best[lane] : 0ull;
            second = lane < nw ? s_sec[lane] : 0.0f;
            for (int o = 16; o > 0; o >>= 1)
                argmax_merge(best, second, __shfl_xor_sync(0xffffffffu, best, o), __shfl_xor_sync(0xffffffffu, second, o));
            if (lane == 0) {
                const unsigned long long old = atomicMax(dst, best);
                if (old != best) argmax_merge(best, second, old, 0.0f);
                atomicMax(dst_second, float_order_bits(second));
            }
        }
#endif
    }
};

#if defined(__CUDACC__)
// Resident CTAs per SM the register allocation must allow: the static four-step kernels are
// sized (shared memory) for 3 CTAs per SM; kernels without a MIN_CTAS member ask for 1.
template <class K, class = void>
struct min_ctas_of { static constexpr int value = 1; };
template <class K>
struct min_ctas_of<K, std::void_t<decltype(K::MIN_CTAS)>> { static constexpr int value = K::MIN_CTAS; };

template <class K>
__global__ void __launch_bounds__(K::THREADS, min_ctas_of<K>::value)
fft_kernel_entry(const __grid_constant__ typename K::Params p) {   // grid constant: tensor maps are used in place
    extern __shared__ __align__(128) unsigned char asc_smem[];   // TMA tile boxes land on 128-byte rows
    pdl_prologue();
    DeviceExec ex;
    ex.x_ = (int)blockIdx.x; ex.y_ = (int)blockIdx.y; ex.z_ = (int)blockIdx.z;
    K::run(ex, p, reinterpret_cast<cplx*>(asc_smem));
}
#endif

}  // namespace asc
