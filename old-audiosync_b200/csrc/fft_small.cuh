// fft_small.cuh -- whole-transform-in-one-CTA kernel for short lengths.
//
// For even, 2/3/5-smooth sample_len L = M <= SMALL_MAX_M one CTA per pair does
// the entire path in shared memory: packed forward FFTs of the source and the
// zero-padded sample (runtime radix list from {4,2,3,5}), the real-FFT split,
// conj-multiply and merge (same split_mul_merge as the four-step K_B), the
// inverse FFT and the |r| argmax.  Same in-place DIF / DIT passes and digit
// maps as the static kernels, with runtime strides.  This is what the
// reference's tests/test_cross_correlation.c sizes with smooth lengths (T7, T8:
// L = 1000) run through.
#pragma once

#include "fft_kernels.cuh"

namespace asc {

constexpr int SMALL_MAX_M = 8192;
constexpr int SMALL_MAX_PASSES = 16;
constexpr int SMALL_THREADS = 256;

struct SmallPlan {
    int M;
    int npass;
    int radix[SMALL_MAX_PASSES];
    int stride[SMALL_MAX_PASSES];   // s(p) = M / (r0*...*rp)
};

ASC_HD int small_pos_of_freq(const SmallPlan& pl, int k) {
    int pos = 0;
    for (int p = 0; p < pl.npass; p++) {
        int d = k % pl.radix[p];
        k /= pl.radix[p];
        pos += d * pl.stride[p];
    }
    return pos;
}

// PHAT: the split step whitens the spectra (split_phat_merge); w is wn[k] as for the product.
// WIN: the windowed twin -- only the raw indices Params::win allows compete (ArgmaxAcc::consider_win).
// SHARED_SRC: every pair reads the one source at Params::sources (its pitch is not read).
template <typename InT, bool PHAT = false, bool WIN = false, bool SHARED_SRC = false>
struct SmallXcorrKernel {
    static constexpr int THREADS = SMALL_THREADS;

    struct Params {
        const InT* sources;   // [pair][2M]
        const InT* samples;   // [pair][M]
        PairPeak* peaks;      // [pair]
        const cplx* wm;       // exp(-2*pi*i*t/M),  t < M
        const cplx* wn;       // exp(-2*pi*i*t/2M), t < M
        SmallPlan plan;
        long long src_pitch;  // elements between consecutive pairs; 0 = packed (2M / M)
        long long smp_pitch;
        int vec_src, vec_smp; // one load per packed point (every pair's base is aligned to two elements)
        [[no_unique_address]] std::conditional_t<WIN, RawWindow, NoWindow> win;   // WIN only
    };
    // two rows of M points + 512 bytes of reduction scratch (phase_argmax needs 392)
    static size_t smem_bytes(int M) { return (size_t)2 * M * sizeof(cplx) + 512; }

    // one in-place radix-R pass over `rows` rows; FWD: DIF (twiddle after the
    // butterfly), else DIT inverse (conjugate twiddle before it).
    template <int R, bool FWD, class Ex>
    static ASC_HD void pass(Ex& ex, const Params& p, cplx* __restrict__ buf, int ps, int rows,
                            bool from_global) {
        const int M = p.plan.M;
        const int S = p.plan.stride[ps];
        const int per_row = M / R;
        const int tstep = M / (S * R);
        const int items = per_row * rows;
        const long long pair = ex.bz();
        ex.phase([&](int tid) {
            for (int w = tid; w < items; w += THREADS) {
                const int rr = w / per_row;
                const int bf = w - rr * per_row;
                cplx* __restrict__ row = buf + rr * M;
                const int blk = bf / S;
                const int j = bf - blk * S;
                const int i0 = blk * (S * R) + j;
                cplx v[R];
                if (from_global) {
                    static_for<0, R>([&](auto Q) {
                        constexpr int q = decltype(Q)::value;
                        const long long n = i0 + q * S;
                        if (rr == 0) v[q] = load_packed<InT>(p.sources + (SHARED_SRC ? 0 : pair * (p.src_pitch ? p.src_pitch : 2 * M)), n, p.vec_src != 0);
                        else v[q] = n < M / 2 ? load_packed<InT>(p.samples + pair * (p.smp_pitch ? p.smp_pitch : M), n, p.vec_smp != 0)
                                              : cmake(0.f, 0.f);
                    });
                } else {
                    static_for<0, R>([&](auto Q) {
                        constexpr int q = decltype(Q)::value;
                        cplx x = row[i0 + q * S];
                        if (!FWD && q > 0 && S > 1) x = cmulc(x, ldg(p.wm + (long long)j * q * tstep));
                        v[q] = x;
                    });
                }
                dft_reg<R, FWD ? -1 : +1>(v);
                static_for<0, R>([&](auto K) {
                    constexpr int k = decltype(K)::value;
                    cplx y = v[k];
                    if (FWD && k > 0 && S > 1) y = cmul(y, ldg(p.wm + (long long)j * k * tstep));
                    row[i0 + k * S] = y;
                });
            }
        });
    }

    template <bool FWD, class Ex>
    static ASC_HD void pass_any(Ex& ex, const Params& p, cplx* buf, int ps, int rows, bool from_global) {
        switch (p.plan.radix[ps]) {
            case 2: pass<2, FWD>(ex, p, buf, ps, rows, from_global); break;
            case 3: pass<3, FWD>(ex, p, buf, ps, rows, from_global); break;
            case 4: pass<4, FWD>(ex, p, buf, ps, rows, from_global); break;
            default: pass<5, FWD>(ex, p, buf, ps, rows, from_global); break;
        }
    }

    // grid = (1, 1, pairs)
    template <class Ex>
    static ASC_HD void run(Ex& ex, const Params& p, cplx* __restrict__ buf) {
        const int M = p.plan.M;
        const int np = p.plan.npass;
        const long long pair = ex.bz();
        ex.phase([&](int tid) {
            if (tid == 0) p.peaks[pair] = cleared_peak();
        });
        for (int ps = 0; ps < np; ps++) pass_any<true>(ex, p, buf, ps, 2, ps == 0);
        // split + multiply + merge: bins (k, M-k), k = 0 .. M/2, into row 0
        ex.phase([&](int tid) {
            for (int e = tid; e <= M / 2; e += THREADS) {
                const int pa = small_pos_of_freq(p.plan, e);
                const int pb = small_pos_of_freq(p.plan, e == 0 ? 0 : M - e);
                cplx qk, qmk;
                if constexpr (PHAT) split_phat_merge<1>(buf[pa], buf[pb], buf[M + pa], buf[M + pb], ldg(p.wn + e), qk, qmk);
                else split_mul_merge(buf[pa], buf[pb], buf[M + pa], buf[M + pb], ldg(p.wn + e), qk, qmk);
                buf[pa] = qk;
                if (pa != pb) buf[pb] = qmk;
            }
        });
        for (int ps = np - 1; ps >= 0; ps--) pass_any<false>(ex, p, buf, ps, 1, false);
        // natural order now: packed point n carries r[2n], r[2n+1]
        ex.phase_argmax(
            [&](int tid) -> ArgmaxPair {
                ArgmaxAcc acc;
                for (int n = tid; n < M; n += THREADS) {
                    const cplx v = buf[n];
                    const uint32_t i_re = (uint32_t)(2 * n);
                    if constexpr (WIN) {
                        acc.consider_win(v.x, i_re, p.win, &p.peaks[pair]);
                        acc.consider_win(v.y, i_re + 1u, p.win, &p.peaks[pair]);
                    } else {
                        if (n == 0) acc.consider_seed(v.x, &p.peaks[pair]);
                        else acc.consider(v.x, i_re);
                        acc.consider(v.y, i_re + 1u);
                    }
                }
                return acc.result();
            },
            &p.peaks[pair].key, &p.peaks[pair].second_bits, buf + 2 * M);
    }
};

}  // namespace asc
