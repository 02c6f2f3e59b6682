// audiosync_cuda.cu -- libaudiosync_cuda.so: context, wave scheduler,
// multi-GPU dispatcher and the C ABI of include/audiosync_cuda.h.
//
// Product path only: nothing here (or anywhere in this library) calls the CPU
// oracle, cuFFT, or any host-side arithmetic fallback.  If CUDA is missing or
// a launch fails the entry points fail loudly (-1 / NaN + one stderr line).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <immintrin.h>
#include <sched.h>
#include <limits>
#include <map>
#include <thread>

#include "plan_host.h"
#include "reduce_kernels.cuh"

// The reference defines `volatile int global_debug` in src/audiosync.c:37 and its
// LOG() macro (include/audiosync/audiosync.h:88-94) reads it.  When this library
// is linked into the reference build the symbol resolves to that definition;
// stand-alone (ctypes, tests) it is absent, hence weak.
extern "C" {
extern volatile int global_debug __attribute__((weak));
}

namespace asc {

// ------------------------------------------------------------------ errors
static thread_local char g_last_error[512] = "";
static int g_debug_flag = 0;

void set_last_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_last_error, sizeof(g_last_error), fmt, ap);
    va_end(ap);
    fprintf(stderr, "audiosync: %s\n", g_last_error);
}

// A worker thread's message (its own thread-local buffer) handed to the calling thread.
static std::string take_last_error() { return std::string(g_last_error); }
static void adopt_last_error(const std::string& msg) {
    snprintf(g_last_error, sizeof(g_last_error), "%s", msg.c_str());
}

static bool debug_on() { return g_debug_flag || (&global_debug != nullptr && global_debug); }

const char* kernel_class_name(int k) {
    static const char* names[KC_COUNT] = {
        "synth", "direct_corr", "argmax_f64", "col_fwd", "row_fused",
        "col_inv_argmax", "small_fft", "pearson", "src_spectrum"};
    return (k >= 0 && k < KC_COUNT) ? names[k] : "?";
}

// ----------------------------------------------------------------- buffers
int DevBuf::ensure(size_t need) {
    if (need <= bytes) return 0;
    if (p) { cudaFree(p); p = nullptr; bytes = 0; }
    size_t want = need + need / 8;
    if (cudaMalloc(&p, want) != cudaSuccess) {
        cudaGetLastError();
        want = need;
        ASC_CUDA_OK(cudaMalloc(&p, want));
    }
    bytes = want;
    return 0;
}
void DevBuf::release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }

int PinnedBuf::ensure(size_t need) {
    if (need <= bytes) return 0;
    if (p) { cudaFreeHost(p); p = nullptr; bytes = 0; }
    ASC_CUDA_OK(cudaMallocHost(&p, need));
    bytes = need;
    return 0;
}
void PinnedBuf::release() { if (p) cudaFreeHost(p); p = nullptr; bytes = 0; }

template <typename InT, bool PHAT, bool WIN>
static int run_small_wave(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, const void* src,
                          const void* smp, long long sp, long long mp, PairPeak* peaks, int pairs,
                          cudaStream_t st, const RawWindow* win) {
    auto go = [&](auto KK) -> int {
        using K = decltype(KK);
        // one load per packed point where every pair's base is aligned to two elements
        const size_t al = 2 * sizeof(InT);
        const int vec_src = reinterpret_cast<uintptr_t>(src) % al == 0 && sp % 2 == 0;
        const int vec_smp = reinterpret_cast<uintptr_t>(smp) % al == 0 && mp % 2 == 0;
        typename K::Params p{static_cast<const InT*>(src), static_cast<const InT*>(smp), peaks,
                             static_cast<const cplx*>(plan->wm.p), static_cast<const cplx*>(plan->wn.p),
                             plan->small, sp, mp, vec_src, vec_smp};
        if constexpr (WIN) p.win = *win;
        const size_t smem = K::smem_bytes(plan->small.M);
        const dim3 grid(1, 1, pairs);
        return launch(ctx, d, KC_SMALL_FFT, st, [&] {
            fft_kernel_entry<K><<<grid, K::THREADS, smem, st>>>(p);
        });
    };
    // sp == 0: every pair reads the one source (the shared-source call; the kernel's 0 means packed)
    return sp == 0 ? go(SmallXcorrKernel<InT, PHAT, WIN, true>{}) : go(SmallXcorrKernel<InT, PHAT, WIN>{});
}

static int build_small_plan(FftPlan* plan, long long L) {
    plan->kind = PATH_SMALL_FFT;
    plan->L = L;
    if (!make_small_plan(L, &plan->small)) return -1;
    plan->ws_bytes_per_pair = 0;
    std::string d = "fft L=" + std::to_string(L) + " single-CTA radices=";
    for (int i = 0; i < plan->small.npass; i++) d += (i ? "x" : "") + std::to_string(plan->small.radix[i]);
    d += " fp32";
    plan->desc = d;
    if (upload(plan->wm, build_full_table(L, L)) != 0 || upload(plan->wn, build_full_table(2 * L, L)) != 0)
        return -1;
    const size_t smem = SmallXcorrKernel<float>::smem_bytes((int)L);
    if (smem > 48 * 1024) {
        const int cap = (int)SmallXcorrKernel<float>::smem_bytes(SMALL_MAX_M);
        auto allow = [&](auto KK) -> int {
            ASC_CUDA_OK(cudaFuncSetAttribute(fft_kernel_entry<decltype(KK)>, cudaFuncAttributeMaxDynamicSharedMemorySize, cap));
            return 0;
        };
        auto allow_all = [&](auto PH, auto W) -> int {
            constexpr bool PHAT = decltype(PH)::value, WIN = decltype(W)::value;
            return allow(SmallXcorrKernel<float, PHAT, WIN>{}) | allow(SmallXcorrKernel<double, PHAT, WIN>{}) |
                   allow(SmallXcorrKernel<int16_t, PHAT, WIN>{}) | allow(SmallXcorrKernel<float, PHAT, WIN, true>{}) |
                   allow(SmallXcorrKernel<double, PHAT, WIN, true>{}) | allow(SmallXcorrKernel<int16_t, PHAT, WIN, true>{});
        };
        if ((plan->phat ? allow_all(std::true_type{}, std::false_type{}) | allow_all(std::true_type{}, std::true_type{})
                        : allow_all(std::false_type{}, std::false_type{}) | allow_all(std::false_type{}, std::true_type{})) != 0)
            return -1;
    }
    auto run = [plan](auto PH, auto W, audiosync_cuda_ctx* ctx, DeviceState& d, const void* src, const void* smp, int dtype,
                      long long sp, long long mp, PairPeak* peaks, int pairs, cudaStream_t st, const RawWindow* win) -> int {
        constexpr bool PHAT = decltype(PH)::value, WIN = decltype(W)::value;
        switch (dtype) {
            case AUDIOSYNC_CUDA_F32: return run_small_wave<float, PHAT, WIN>(plan, ctx, d, src, smp, sp, mp, peaks, pairs, st, win);
            case AUDIOSYNC_CUDA_F64: return run_small_wave<double, PHAT, WIN>(plan, ctx, d, src, smp, sp, mp, peaks, pairs, st, win);
            case AUDIOSYNC_CUDA_S16: return run_small_wave<int16_t, PHAT, WIN>(plan, ctx, d, src, smp, sp, mp, peaks, pairs, st, win);
        }
        set_last_error("bad dtype %d", dtype);
        return -1;
    };
    plan->run_wave = [plan, run](audiosync_cuda_ctx* ctx, DeviceState& d, const void* src, const void* smp,
                                 int dtype, long long sp, long long mp, void*, PairPeak* peaks, int pairs,
                                 cudaStream_t st, const RawWindow* win) {
        auto with_phat = [&](auto PH) {
            return win ? run(PH, std::true_type{}, ctx, d, src, smp, dtype, sp, mp, peaks, pairs, st, win)
                       : run(PH, std::false_type{}, ctx, d, src, smp, dtype, sp, mp, peaks, pairs, st, win);
        };
        return plan->phat ? with_phat(std::true_type{}) : with_phat(std::false_type{});
    };
    return 0;
}

template <typename T>
static int build_generic_plan_t(FftPlan* plan) {
    typedef typename GenTraits<T>::C C;
    const GenShape& sh = plan->gen;
    const GenTables<C> tb = gen_build_tables<C>(sh);
    if (upload(plan->g_wcol, tb.wcol) != 0 || upload(plan->g_wrow, tb.wrow) != 0 || upload(plan->g_lo, tb.m_lo) != 0 ||
        upload(plan->g_hi, tb.m_hi) != 0 || upload(plan->g_p2f_col, tb.p2f_col) != 0 ||
        upload(plan->g_wpos, tb.wpos) != 0 || upload(plan->g_f2p_row, tb.f2p_row) != 0)
        return -1;
    const bool small_col = sh.nt_col == GEN_THREADS_SMALL, small_row = sh.nt_row == GEN_THREADS_SMALL;
    // rows on a static row kernel where the plan's M2 has one (fp32 only): its output carries the
    // factor 1/2 of the merge step that the runtime-radix row kernel leaves to peak_scale
    static const bool no_static_rows = getenv("AUDIOSYNC_CUDA_NO_STATIC_ROWS") != nullptr;      // diagnostics / A-B runs
    const bool static_rows = sizeof(T) == 4 && sh.static_rows != 0 && !no_static_rows;
    if (static_rows) plan->peak_scale *= 2.0;
    // PHAT: the split's half-angle tables in the runtime-radix row kernel's position order (a static
    // row kernel uploads its own)
    if (plan->phat && !static_rows &&
        (upload(plan->phat_rev, tb.phat_pos) != 0 || upload(plan->phat_lo, tb.phat_lo) != 0 || upload(plan->phat_hi, tb.phat_hi) != 0))
        return -1;
    if ((small_col ? GenStage<T, GEN_THREADS_SMALL>::prepare_cols(sh) : GenStage<T, GEN_THREADS>::prepare_cols(sh)) != 0 ||
        (static_rows ? static_rows_prepare(plan)
                     : small_row ? GenStage<T, GEN_THREADS_SMALL>::prepare_rows(sh, plan->phat)
                                 : GenStage<T, GEN_THREADS>::prepare_rows(sh, plan->phat)) != 0)
        return -1;
    plan->run_wave = [plan, small_col, small_row, static_rows](audiosync_cuda_ctx* ctx, DeviceState& d, const void* src, const void* smp,
                                                  int dtype, long long sp, long long mp, void* ws, PairPeak* peaks, int pairs,
                                                  cudaStream_t st, const RawWindow* win) {
        using Big = GenStage<T, GEN_THREADS>;
        using Small = GenStage<T, GEN_THREADS_SMALL>;
        if ((small_col ? Small::col_fwd(plan, ctx, d, src, smp, dtype, sp, mp, ws, peaks, pairs, st)
                       : Big::col_fwd(plan, ctx, d, src, smp, dtype, sp, mp, ws, peaks, pairs, st)) != 0) return -1;
        if ((static_rows ? static_rows_launch(plan, ctx, d, ws, pairs, st)
                         : small_row ? Small::rows(plan, ctx, d, ws, pairs, st) : Big::rows(plan, ctx, d, ws, pairs, st)) != 0) return -1;
        return small_col ? Small::col_inv(plan, ctx, d, ws, peaks, pairs, st, win) : Big::col_inv(plan, ctx, d, ws, peaks, pairs, st, win);
    };
    return 0;
}

static int build_generic_plan(FftPlan* plan, long long L, bool precise) {
    plan->kind = PATH_GENERIC_FFT;
    plan->L = L;
    if (!gen_make_shape(L, precise, &plan->gen)) return -1;
    plan->M1 = plan->gen.M1; plan->M2 = plan->gen.M2;
    plan->ws_bytes_per_pair = (size_t)2 * plan->gen.M * (precise ? sizeof(cplxd) : sizeof(cplx));
    plan->peak_scale = gen_peak_scale(plan->gen);
    plan->desc = gen_describe(plan->gen, precise);
    return precise ? build_generic_plan_t<double>(plan) : build_generic_plan_t<float>(plan);
}

template <typename InT>
static int run_direct_wave(long long L, audiosync_cuda_ctx* ctx, DeviceState& d, const void* src,
                           const void* smp, long long sp, long long mp, void* ws, PairPeak* peaks, int pairs,
                           cudaStream_t st, const RawWindow* win) {
    const long long N = 2 * L;
    double* r = static_cast<double*>(ws);
    const dim3 grid((unsigned)((N + DIRECT_TILE - 1) / DIRECT_TILE), pairs);
    if (launch(ctx, d, KC_DIRECT, st, [&] {
            direct_corr_kernel<InT><<<grid, DIRECT_TILE, 0, st>>>(static_cast<const InT*>(src),
                                                                  static_cast<const InT*>(smp), r, L, sp, mp);
        }) != 0) return -1;
    return launch(ctx, d, KC_ARGMAX_F64, st, [&] {
        if (win) argmax_f64_window_kernel<<<pairs, 1024, 0, st>>>(r, N, N, peaks, *win);
        else argmax_f64_kernel<<<pairs, 1024, 0, st>>>(r, N, N, peaks);
    });
}

static int build_direct_plan(FftPlan* plan, long long L) {
    plan->kind = PATH_DIRECT;
    plan->L = L;
    plan->ws_bytes_per_pair = (size_t)2 * L * sizeof(double);
    plan->desc = "direct L=" + std::to_string(L) + " time-domain O(L^2) fp64";
    plan->run_wave = [L](audiosync_cuda_ctx* ctx, DeviceState& d, const void* src, const void* smp,
                         int dtype, long long sp, long long mp, void* ws, PairPeak* peaks, int pairs,
                         cudaStream_t st, const RawWindow* win) {
        switch (dtype) {
            case AUDIOSYNC_CUDA_F32: return run_direct_wave<float>(L, ctx, d, src, smp, sp, mp, ws, peaks, pairs, st, win);
            case AUDIOSYNC_CUDA_F64: return run_direct_wave<double>(L, ctx, d, src, smp, sp, mp, ws, peaks, pairs, st, win);
            case AUDIOSYNC_CUDA_S16: return run_direct_wave<int16_t>(L, ctx, d, src, smp, sp, mp, ws, peaks, pairs, st, win);
        }
        set_last_error("bad dtype %d", dtype);
        return -1;
    };
    return 0;
}

// plans are cached per device and per (L, forced path, precise, weighting)
static FftPlan* get_plan(audiosync_cuda_ctx* ctx, DeviceState& d, long long L) {
    std::lock_guard<std::mutex> plk(d.plan_mu);
    const bool phat = ctx->weighting == AUDIOSYNC_CUDA_WEIGHT_PHAT;
    const size_t key = ((size_t)L * 8 + (size_t)ctx->path * 2 + (ctx->precise ? 1 : 0)) * 2 + (phat ? 1 : 0);
    auto it = d.plans.find(key);
    if (it != d.plans.end()) return it->second.get();
    auto plan = std::make_shared<FftPlan>();
    plan->phat = phat;
    const char* why = nullptr;
    const PathKind kind = phat ? choose_path_phat(L, ctx->path, ctx->precise, &why) : choose_path(L, ctx->path, ctx->precise);
    int rc = -1;
    if (kind == PATH_NONE) {
        if (why) set_last_error("sample_len %lld: %s", L, why);
        else set_last_error("sample_len %lld: no transform plan fits the device and the O(L^2) kernel is not used above %lld frames",
                            L, DIRECT_MAX_L);
        return nullptr;
    }
    if (kind == PATH_STATIC_FFT) {
        for_each_static_plan([&](auto P) {
            using PT = decltype(P);
            if (PT::L == L) rc = build_static_plan<PT>(plan.get());
        });
    } else if (kind == PATH_SMALL_FFT) {
        rc = build_small_plan(plan.get(), L);
    } else if (kind == PATH_GENERIC_FFT) {
        rc = build_generic_plan(plan.get(), L, ctx->precise);
    } else {
        rc = build_direct_plan(plan.get(), L);
    }
    if (rc != 0) {
        if (g_last_error[0] == 0) set_last_error("could not build a plan for sample_len %lld", L);
        return nullptr;
    }
    if (phat) plan->desc += " phat";
    d.plans[key] = plan;
    return plan.get();
}

static int default_wave_pairs(const FftPlan* plan, size_t n_pairs) {
    long long w;
    if (plan->kind == PATH_STATIC_FFT) {
        // Enough pairs per launch that the partial last wave of CTAs and the serialised
        // start/drain of each launch are ~1 % of it (256 pairs at L = 1.44M: ~170 waves of the
        // 3-CTA/SM kernels; measured in the 4,096-pair run: 64 -> 39.0k, 128 -> 39.5k,
        // 256 -> 39.9k pairs/s); the workspace stays at <= 5.9 GB whatever the length and
        // is only as large as the batch needs.
        w = (256LL * 1440000) / plan->L;
        w = std::max(16LL, std::min(1024LL, w));
    } else if (plan->kind == PATH_SMALL_FFT) {
        w = 16384;
    } else if (plan->kind == PATH_GENERIC_FFT) {
        // ~6 GB of planes per wave at most, at least a few hundred CTAs per launch
        w = std::max(1LL, std::min(1024LL, (6LL << 30) / (long long)std::max<size_t>(plan->ws_bytes_per_pair, 1)));
    } else {
        const long long per = (long long)plan->ws_bytes_per_pair;
        w = std::max(1LL, std::min(1024LL, (256LL << 20) / std::max(1LL, per)));
    }
    return (int)std::min<long long>(w, (long long)std::max<size_t>(n_pairs, 1));
}

// The context's lag window at sample_len L: -1 (message set) when no lag of [-L, L - 1] is in it,
// 0 when it holds them all (the unwindowed kernels), 1 with *w set otherwise.
static int lag_window(const audiosync_cuda_ctx* ctx, long long L, RawWindow* w) {
    const int rc = raw_window_of(ctx->lag_lo, ctx->lag_hi, L, w);
    if (rc < 0)
        set_last_error("lag window [%lld, %lld] holds no lag of [%lld, %lld] at sample_len %lld",
                       ctx->lag_lo, ctx->lag_hi, -L, L - 1, L);
    return rc;
}

// Ticket counters of the Pearson kernel: zeroed once, self-resetting afterwards.
static int ensure_tickets(WorkSet& w, size_t n) {
    const size_t need = sizeof(unsigned int) * n;
    if (need <= w.tickets.bytes) return 0;
    ASC_CUDA_OK(cudaDeviceSynchronize());
    if (w.tickets.ensure(need) != 0) return -1;
    ASC_CUDA_OK(cudaMemset(w.tickets.p, 0, w.tickets.bytes));
    return 0;
}

// Enqueue the whole path for device-resident pairs on `st` (no sync).
// src_pitch / smp_pitch: elements between consecutive pairs (0 = packed [pair][2L] / [pair][L]).
// shared_src: every pair reads the one source at `src` (audiosync_cuda_xcorr_shared_source); the
// kernels then get a source pitch of 0, and a static plan transforms the source into work.spec.
// spectrum_ready: an earlier enqueue of the same call, on this work set and stream, already left that
// source's spectrum in work.spec (the chunks of a host-fed call), so it is not computed again.
static int enqueue_batch(audiosync_cuda_ctx* ctx, DeviceState& d, WorkSet& work, const void* src, const void* smp,
                         size_t n_pairs, long long L, int dtype, audiosync_cuda_result* d_results,
                         cudaStream_t st, long long src_pitch = 0, long long smp_pitch = 0, bool shared_src = false,
                         bool spectrum_ready = false) {
    if (n_pairs == 0) return 0;
    if (shared_src) src_pitch = 0;
    else if (src_pitch == 0) src_pitch = 2 * L;
    if (smp_pitch == 0) smp_pitch = L;
    const bool packed = src_pitch == 2 * L && smp_pitch == L;
    if (L <= 0 || L > (1LL << 30)) { set_last_error("unsupported sample_len %lld", L); return -1; }
    const size_t esz = dtype_bytes(dtype);
    if (esz == 0) { set_last_error("bad dtype %d", dtype); return -1; }
    // every kernel reads whole elements: a base between two elements is no array of this dtype
    if (reinterpret_cast<uintptr_t>(src) % esz != 0 || reinterpret_cast<uintptr_t>(smp) % esz != 0) {
        set_last_error("sources / samples base is not aligned to its %zu-byte element", esz);
        return -1;
    }
    RawWindow raw_win;
    const int windowed = lag_window(ctx, L, &raw_win);
    if (windowed < 0) return -1;
    const RawWindow* win = windowed ? &raw_win : nullptr;
    ASC_CUDA_OK(cudaSetDevice(d.device));
    FftPlan* plan = get_plan(ctx, d, L);
    if (!plan) return -1;
    const int in_dtype = dtype == ASC_DTYPE_F32_EXACT ? AUDIOSYNC_CUDA_F32 : dtype;   // what the transform loads
    int wave = ctx->wave_pairs > 0 ? ctx->wave_pairs : default_wave_pairs(plan, n_pairs);
    wave = (int)std::min<size_t>((size_t)wave, n_pairs);
    wave = std::min(wave, 65535);
    const int n_chunks = (int)((L + PEARSON_CHUNK - 1) / PEARSON_CHUNK);
    // The previous user of this scratch set may still be running on another stream: order this
    // batch behind it (same stream: stream order already does).
    if (work.used && work.last_stream != st) ASC_CUDA_OK(cudaStreamWaitEvent(st, work.done, 0));
    if (!work.done) ASC_CUDA_OK(cudaEventCreateWithFlags(&work.done, cudaEventDisableTiming));
    if (work.ws.ensure(plan->ws_bytes_per_pair * (size_t)wave + 256) != 0) return -1;
    if (work.peaks.ensure(sizeof(PairPeak) * (size_t)wave) != 0) return -1;
    if (work.partials.ensure(sizeof(PearsonPartial) * (size_t)wave * n_chunks) != 0) return -1;
    PairPeak* peaks = static_cast<PairPeak*>(work.peaks.p);
    PearsonPartial* partials = static_cast<PearsonPartial*>(work.partials.p);
    if (ensure_tickets(work, (size_t)wave) != 0) return -1;
    unsigned int* tickets = static_cast<unsigned int*>(work.tickets.p);
    // the source's forward rows, once per call, where the plan can reuse them (the static plans);
    // every other plan reads the one source in every pair's transform
    const bool reuse = shared_src && plan->run_shared_wave;
    if (reuse && !spectrum_ready &&
        (work.spec.ensure(sizeof(cplx) * (size_t)L) != 0 || plan->source_spectrum(ctx, d, src, in_dtype, work.spec.p, peaks, st) != 0))
        return -1;
    for (size_t p0 = 0; p0 < n_pairs; p0 += (size_t)wave) {
        const int pairs = (int)std::min<size_t>((size_t)wave, n_pairs - p0);
        const char* s = static_cast<const char*>(src) + p0 * (size_t)src_pitch * esz;
        const char* m = static_cast<const char*>(smp) + p0 * (size_t)smp_pitch * esz;
        if ((reuse ? plan->run_shared_wave(ctx, d, work.spec.p, m, in_dtype, smp_pitch, work.ws.p, peaks, pairs, st, win)
                   : plan->run_wave(ctx, d, s, m, in_dtype, src_pitch, smp_pitch, work.ws.p, peaks, pairs, st, win)) != 0)
            return -1;
        const dim3 grid(n_chunks, pairs);
        int rc;
        if (dtype == AUDIOSYNC_CUDA_F32) {
            rc = launch(ctx, d, KC_PEARSON, st, [&] {
                launch_stage(plan->phat ? pearson_kernel<float, false, true> : pearson_kernel<float, false>, grid, dim3(PEARSON_THREADS), 0, st,
                    reinterpret_cast<const float*>(s), reinterpret_cast<const float*>(m), src_pitch, smp_pitch, L,
                    (const PairPeak*)peaks, 0LL, plan->peak_scale, partials, tickets, n_chunks, d_results + p0);
            });
        } else if (dtype == ASC_DTYPE_F32_EXACT) {
            rc = launch(ctx, d, KC_PEARSON, st, [&] {
                launch_stage(plan->phat ? pearson_kernel<float, true, true> : pearson_kernel<float, true>, grid, dim3(PEARSON_THREADS), 0, st,
                    reinterpret_cast<const float*>(s), reinterpret_cast<const float*>(m), src_pitch, smp_pitch, L,
                    (const PairPeak*)peaks, 0LL, plan->peak_scale, partials, tickets, n_chunks, d_results + p0);
            });
        } else if (dtype == AUDIOSYNC_CUDA_F64) {
            rc = launch(ctx, d, KC_PEARSON, st, [&] {
                launch_stage(plan->phat ? pearson_kernel<double, true, true> : pearson_kernel<double, true>, grid, dim3(PEARSON_THREADS), 0, st,
                    reinterpret_cast<const double*>(s), reinterpret_cast<const double*>(m), src_pitch, smp_pitch, L,
                    (const PairPeak*)peaks, 0LL, plan->peak_scale, partials, tickets, n_chunks, d_results + p0);
            });
        } else {   // S16 (esz above admits nothing else): the f64 path's arithmetic on s * 2^-15
            rc = launch(ctx, d, KC_PEARSON, st, [&] {
                launch_stage(plan->phat ? pearson_kernel<int16_t, true, true> : pearson_kernel<int16_t, true>, grid, dim3(PEARSON_THREADS), 0, st,
                    reinterpret_cast<const int16_t*>(s), reinterpret_cast<const int16_t*>(m), src_pitch, smp_pitch, L,
                    (const PairPeak*)peaks, 0LL, plan->peak_scale, partials, tickets, n_chunks, d_results + p0);
            });
        }
        if (rc != 0) return -1;
    }
    ASC_CUDA_OK(cudaEventRecord(work.done, st));
    work.last_stream = st;
    work.used = true;
    return 0;
}

static int drain_profile(DeviceState& d) {
    ASC_CUDA_OK(cudaSetDevice(d.device));
    ASC_CUDA_OK(cudaDeviceSynchronize());
    for (auto& r : d.prof_pending) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, r.e0, r.e1) == cudaSuccess) {
            d.prof_ms[r.cls] += ms;
            d.prof_launches[r.cls] += 1;
        }
        d.event_pool.push_back(r.e0);
        d.event_pool.push_back(r.e1);
    }
    d.prof_pending.clear();
    return 0;
}

static void destroy_device_state(DeviceState& d) {
    if (d.device < 0) return;
    cudaSetDevice(d.device);
    cudaDeviceSynchronize();
    d.plans.clear();
    d.work.release(); d.results.release();
    for (int i = 0; i < 2; i++) {
        d.in_src[i].release(); d.in_smp[i].release();
        d.in_src32[i].release(); d.in_smp32[i].release();
        if (d.ev_up32[i]) cudaEventDestroy(d.ev_up32[i]);
        if (d.ev_up[i]) cudaEventDestroy(d.ev_up[i]);
        if (d.ev_done[i]) cudaEventDestroy(d.ev_done[i]);
    }
    d.h_results.release();
    d.stage.release();
    for (auto& r : d.prof_pending) { cudaEventDestroy(r.e0); cudaEventDestroy(r.e1); }
    for (auto e : d.event_pool) cudaEventDestroy(e);
    if (d.stream) cudaStreamDestroy(d.stream);
    if (d.copy_stream) cudaStreamDestroy(d.copy_stream);
    if (d.narrow_stream) cudaStreamDestroy(d.narrow_stream);
    for (int k = 0; k < DeviceState::DIRECT_DEPTH; k++)
        if (d.direct_ev[k]) cudaEventDestroy(d.direct_ev[k]);
    d.device = -1;
}

bool narrow_f64_to_f32(float* dst, const double* src, size_t n, bool stream);      // host_simd.cpp

// A few persistent helper threads that split one large host memcpy (pageable input -> pinned
// bounce buffer) or one double -> float narrowing pass into slices: a single core copies ~10 GB/s,
// PCIe takes 55.  One pass at a time (callers would only fight over the same memory bandwidth);
// never torn down.
class CopyPool {
    struct Slice { char* dst; const char* src; size_t n; bool narrow; };   // n: bytes (copy) or elements (narrow)
    void run_slice(const Slice& s) {
        if (!s.narrow) { memcpy(s.dst, s.src, s.n); return; }
        if (!narrow_f64_to_f32(reinterpret_cast<float*>(s.dst), reinterpret_cast<const double*>(s.src), s.n, nt_stores_))
            inexact_.store(true, std::memory_order_relaxed);
    }
    std::vector<std::thread> workers_;
    std::mutex m_, run_mu_;
    std::condition_variable cv_, done_cv_;
    std::vector<Slice> slices_;
    size_t next_ = 0, pending_ = 0;
    std::atomic<bool> inexact_{false};
    bool nt_stores_ = true;
    size_t copy_parts_ = 8;
    void loop() {
        std::unique_lock<std::mutex> lk(m_);
        for (;;) {
            cv_.wait(lk, [&] { return next_ < slices_.size(); });
            const Slice s = slices_[next_++];
            lk.unlock();
            run_slice(s);
            lk.lock();
            if (--pending_ == 0) done_cv_.notify_all();
        }
    }
    // n units of `in_unit` source bytes each become `out_unit` destination bytes (copy: 1 -> 1 with
    // n bytes; narrow: 8 -> 4 with n doubles), split over the workers and the calling thread
    void run(void* dst, const void* src, size_t n, size_t in_unit, size_t out_unit, bool narrow, size_t parts) {
        parts = std::max<size_t>(1, std::min(parts, threads()));
        if (n * in_unit < ((size_t)1 << 20) || parts == 1) {
            run_slice(Slice{static_cast<char*>(dst), static_cast<const char*>(src), n, narrow});
            return;
        }
        const size_t per = ((n + parts - 1) / parts + 63) & ~(size_t)63;
        {
            std::lock_guard<std::mutex> lk(m_);
            slices_.clear(); next_ = 0; pending_ = 0;
            for (size_t o = per; o < n; o += per) {       // slice 0 is the caller's own
                slices_.push_back(Slice{static_cast<char*>(dst) + o * out_unit, static_cast<const char*>(src) + o * in_unit,
                                        std::min(per, n - o), narrow});
                pending_++;
            }
        }
        cv_.notify_all();
        run_slice(Slice{static_cast<char*>(dst), static_cast<const char*>(src), std::min(per, n), narrow});
        std::unique_lock<std::mutex> lk(m_);
        done_cv_.wait(lk, [&] { return pending_ == 0; });
    }
public:
    CopyPool(unsigned n, unsigned copy_parts, bool nt) : nt_stores_(nt), copy_parts_(copy_parts) {
        for (unsigned i = 0; i < n; i++) workers_.emplace_back([this] { loop(); });
        for (auto& t : workers_) t.detach();
    }
    size_t threads() const { return workers_.size() + 1; }
    void copy(void* dst, const void* src, size_t bytes) {
        std::lock_guard<std::mutex> run_lk(run_mu_);
        run(dst, src, bytes, 1, 1, false, copy_parts_);
    }
    // dst[i] = (float)src[i]; true when every conversion was exact
    bool narrow(float* dst, const double* src, size_t n) {
        std::lock_guard<std::mutex> run_lk(run_mu_);
        inexact_.store(false, std::memory_order_relaxed);
        run(dst, src, n, sizeof(double), sizeof(float), true, threads());
        return !inexact_.load(std::memory_order_relaxed);
    }
    // The same on the workers alone, so that the calling thread can keep the copy engine fed in the
    // meantime: narrow_begin(); while (!narrow_done()) { ... }; exact = narrow_end().
    void narrow_begin(float* dst, const double* src, size_t n) {
        run_mu_.lock();
        inexact_.store(false, std::memory_order_relaxed);
        const size_t parts = workers_.size();
        if (parts == 0 || n * sizeof(double) < ((size_t)1 << 20)) {
            run_slice(Slice{reinterpret_cast<char*>(dst), reinterpret_cast<const char*>(src), n, true});
            return;
        }
        const size_t per = ((n + parts - 1) / parts + 63) & ~(size_t)63;
        {
            std::lock_guard<std::mutex> lk(m_);
            slices_.clear(); next_ = 0; pending_ = 0;
            for (size_t o = 0; o < n; o += per) {
                slices_.push_back(Slice{reinterpret_cast<char*>(dst + o), reinterpret_cast<const char*>(src + o), std::min(per, n - o), true});
                pending_++;
            }
        }
        cv_.notify_all();
    }
    bool narrow_done() {
        std::lock_guard<std::mutex> lk(m_);
        return pending_ == 0;
    }
    bool narrow_end() {
        {
            std::unique_lock<std::mutex> lk(m_);
            done_cv_.wait(lk, [&] { return pending_ == 0; });
        }
        const bool exact = !inexact_.load(std::memory_order_relaxed);
        run_mu_.unlock();
        return exact;
    }
};
// Plain copies stop scaling at ~8 threads (measured on the 16-core B200 host: 4 / 8 / 12 threads
// stage pageable doubles at 38 / 52 / 50 GB/s); narrowing keeps gaining up to 12 (45 / 68 / 77 GB/s
// of doubles read).  Default: three quarters of the cores this process may run on, at most 12; a
// launcher that runs several processes per host divides the cores among them through
// AUDIOSYNC_CUDA_COPY_THREADS (bench.py under torchrun does).
static CopyPool& copy_pool() {
    static CopyPool* pool = [] {
        unsigned hw = std::max(1u, std::thread::hardware_concurrency());
        cpu_set_t set;
        if (sched_getaffinity(0, sizeof(set), &set) == 0 && CPU_COUNT(&set) > 0) hw = (unsigned)CPU_COUNT(&set);
        const char* e = getenv("AUDIOSYNC_CUDA_COPY_THREADS");
        unsigned n = e ? (unsigned)std::max(1, atoi(e)) : std::min(12u, std::max(1u, hw * 3 / 4));
        const char* nt = getenv("AUDIOSYNC_CUDA_NT_STORES");
        return new CopyPool(n - 1, std::min(8u, n), !(nt && atoi(nt) == 0));
    }();
    return *pool;
}
// Below this many copy threads the conversion cannot outrun the link it is meant to relieve
// (8 GPUs on a 32-vCPU host, 3 threads per process: 4.96 k pairs/s narrowing page-locked doubles
// vs 5.37 k sending them as they are; pageable inputs need the threads anyway and gain at any count).
static size_t narrow_min_threads() {
    static const size_t n = [] { const char* e = getenv("AUDIOSYNC_CUDA_NARROW_MIN_THREADS"); return (size_t)(e ? std::max(1, atoi(e)) : 8); }();
    return n;
}

// Host -> device copy of `bytes` on `st` from ANY host memory.  Page-locked (cudaMallocHost /
// cudaHostRegister'ed, e.g. this library's fftw_alloc_real) and managed sources go straight to
// the copy engine; pageable ones are staged through the pinned ring.
static bool host_pointer_is_pageable(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return true; }
    return at.type == cudaMemoryTypeUnregistered;
}
static int upload_from_host(void* dst, const void* src, size_t bytes, cudaStream_t st, StageRing& ring,
                            bool pageable) {
    if (bytes == 0) return 0;
    if (!pageable) {
        ASC_CUDA_OK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
        return 0;
    }
    for (size_t o = 0; o < bytes; o += StageRing::PIECE) {
        const size_t m = std::min(StageRing::PIECE, bytes - o);
        const int i = ring.next;
        ring.next = (ring.next + 1) % StageRing::N;
        if (ring.buf[i].ensure(StageRing::PIECE) != 0) return -1;
        if (!ring.ev[i]) ASC_CUDA_OK(cudaEventCreateWithFlags(&ring.ev[i], cudaEventDisableTiming));
        if (ring.pending[i]) ASC_CUDA_OK(cudaEventSynchronize(ring.ev[i]));   // its last DMA has drained
        copy_pool().copy(ring.buf[i].p, static_cast<const char*>(src) + o, m);
        ASC_CUDA_OK(cudaMemcpyAsync(static_cast<char*>(dst) + o, ring.buf[i].p, m, cudaMemcpyHostToDevice, st));
        ASC_CUDA_OK(cudaEventRecord(ring.ev[i], st));
        ring.pending[i] = true;
    }
    return 0;
}

// Host doubles -> device floats: converted on the host into the pinned ring (copy threads), so that
// half the bytes cross PCIe.  Any host memory.  *exact is cleared when a value did not survive the
// conversion unchanged; with stop_on_inexact the upload ends at that piece (the caller redoes it).
// meanwhile: called over and over by this thread while the workers convert a piece (it then takes no
// part in the conversion itself).
static int upload_narrowed(float* dst, const double* src, size_t n, cudaStream_t st, StageRing& ring,
                           bool* exact, bool stop_on_inexact, const std::function<void()>& meanwhile) {
    const size_t piece = StageRing::PIECE / sizeof(float);        // elements per ring buffer (4 / 16 MB pieces: -13 %)
    for (size_t o = 0; o < n; o += piece) {
        const size_t m = std::min(piece, n - o);
        const int i = ring.next;
        ring.next = (ring.next + 1) % StageRing::N;
        if (ring.buf[i].ensure(StageRing::PIECE) != 0) return -1;
        if (!ring.ev[i]) ASC_CUDA_OK(cudaEventCreateWithFlags(&ring.ev[i], cudaEventDisableTiming));
        if (ring.pending[i]) ASC_CUDA_OK(cudaEventSynchronize(ring.ev[i]));
        ring.pending[i] = false;
        bool piece_exact;
        if (meanwhile) {
            // the workers convert; this thread keeps the copy engine fed until they are done
            copy_pool().narrow_begin(static_cast<float*>(ring.buf[i].p), src + o, m);
            while (!copy_pool().narrow_done()) {
                meanwhile();
                for (int k = 0; k < 64; k++) _mm_pause();
            }
            piece_exact = copy_pool().narrow_end();
        } else {
            piece_exact = copy_pool().narrow(static_cast<float*>(ring.buf[i].p), src + o, m);
        }
        if (!piece_exact) {
            *exact = false;
            if (stop_on_inexact) return 0;
        }
        ASC_CUDA_OK(cudaMemcpyAsync(dst + o, ring.buf[i].p, m * sizeof(float), cudaMemcpyHostToDevice, st));
        ASC_CUDA_OK(cudaEventRecord(ring.ev[i], st));
        ring.pending[i] = true;
        if (meanwhile) meanwhile();
    }
    return 0;
}

// Pieces of the staging ring whose upload has not finished yet.
static int ring_backlog(StageRing& ring) {
    int n = 0;
    for (int i = 0; i < StageRing::N; i++) {
        if (!ring.pending[i]) continue;
        if (cudaEventQuery(ring.ev[i]) == cudaSuccess) ring.pending[i] = false;
        else { cudaGetLastError(); n++; }
    }
    return n;
}

// Direct (un-narrowed) uploads of whole pairs that run beside the narrowing threads: how many
// are still in flight.
static int direct_in_flight(DeviceState& d) {
    int n = 0;
    for (int k = 0; k < DeviceState::DIRECT_DEPTH; k++) {
        if (!d.direct_pending[k]) continue;
        if (cudaEventQuery(d.direct_ev[k]) == cudaSuccess) d.direct_pending[k] = false;
        else { cudaGetLastError(); n++; }
    }
    return n;
}

// Host-memory pairs [p0, p1) on one device: chunked, double buffered.
//
// F64 batches with host narrowing on (see include/audiosync_cuda.h): a chunk's pairs are taken from
// both ends.  From the back, the copy threads convert a pair to fp32 into the pinned ring and its
// half-size pieces go up on `narrow_stream`; from the front -- page-locked inputs only -- the copy
// engine takes pairs of doubles straight from the caller's memory on `copy_stream`, in slices of
// 8 MB issued only while the ring's uploads keep up, so that link time the conversion leaves idle
// is used and neither side waits for the other.  The two sub-batches [0, k) (doubles) and [k, n) (exact fp32 images) are
// enqueued separately.  solo: this call drives a single device (several devices of one context
// share the copy threads; each then feeds its device with direct uploads only).
// shared_src: `sources` is one source for every pair; it is uploaded once (into in_src[0]) and only
// the samples are chunked, as they are (host narrowing does not apply).
static int run_host_range(audiosync_cuda_ctx* ctx, DeviceState& d, const char* sources,
                          const char* samples, size_t p0, size_t p1, long long L, int dtype,
                          audiosync_cuda_result* out, bool solo, bool shared_src = false) {
    if (p1 <= p0) return 0;
    std::lock_guard<std::mutex> dlk(d.mu);
    ASC_CUDA_OK(cudaSetDevice(d.device));
    const size_t esz = dtype_bytes(dtype);
    const size_t src_n = (size_t)(2 * L), smp_n = (size_t)L;
    const size_t src_bytes = src_n * esz, smp_bytes = smp_n * esz;
    const bool pageable = host_pointer_is_pageable(sources) || host_pointer_is_pageable(samples);
    int mode = (dtype == AUDIOSYNC_CUDA_F64 && !ctx->precise && !shared_src) ? ctx->narrow_host : AUDIOSYNC_CUDA_NARROW_OFF;
    if (mode == AUDIOSYNC_CUDA_NARROW_LOSSLESS && !pageable && (!solo || copy_pool().threads() < narrow_min_threads()))
        mode = AUDIOSYNC_CUDA_NARROW_OFF;
    static const int feed_depth = [] { const char* e = getenv("AUDIOSYNC_CUDA_FEED_DEPTH");
                                       return e ? std::max(1, std::min(atoi(e), DeviceState::DIRECT_DEPTH)) : 2; }();
    static const int feed_backlog = [] { const char* e = getenv("AUDIOSYNC_CUDA_FEED_BACKLOG"); return e ? std::max(0, atoi(e)) : 1; }();
    static const bool both_ways = [] { const char* e = getenv("AUDIOSYNC_CUDA_FEED_BOTH_WAYS"); return !(e && atoi(e) == 0); }();
    const bool hybrid = mode == AUDIOSYNC_CUDA_NARROW_LOSSLESS && !pageable && both_ways;
    // what narrowed pairs are enqueued as: exact images keep the f64 call's arithmetic, ALWAYS answers as an fp32 batch
    const int narrowed_dtype = mode == AUDIOSYNC_CUDA_NARROW_ALWAYS ? AUDIOSYNC_CUDA_F32 : ASC_DTYPE_F32_EXACT;
    // chunk: about 192 MB of input per buffer (twice that when pairs are fed both ways), at least one pair
    const size_t src_chunk_bytes = shared_src ? 0 : src_bytes;      // source bytes per chunked pair
    size_t chunk = std::max<size_t>(1, ((size_t)(hybrid ? 384u : 192u) << 20) / (src_chunk_bytes + smp_bytes));
    chunk = std::min(chunk, p1 - p0);
    for (int b = 0; b < 2; b++) {
        if (d.in_src[b].ensure(shared_src ? src_bytes : src_bytes * chunk) != 0 || d.in_smp[b].ensure(smp_bytes * chunk) != 0)
            return -1;
        if (mode != AUDIOSYNC_CUDA_NARROW_OFF &&
            (d.in_src32[b].ensure(sizeof(float) * src_n * chunk) != 0 || d.in_smp32[b].ensure(sizeof(float) * smp_n * chunk) != 0))
            return -1;
        if (!d.ev_up[b]) ASC_CUDA_OK(cudaEventCreateWithFlags(&d.ev_up[b], cudaEventDisableTiming));
        if (!d.ev_up32[b]) ASC_CUDA_OK(cudaEventCreateWithFlags(&d.ev_up32[b], cudaEventDisableTiming));
        if (!d.ev_done[b]) ASC_CUDA_OK(cudaEventCreateWithFlags(&d.ev_done[b], cudaEventDisableTiming));
    }
    for (int k = 0; k < DeviceState::DIRECT_DEPTH; k++)
        if (!d.direct_ev[k]) ASC_CUDA_OK(cudaEventCreateWithFlags(&d.direct_ev[k], cudaEventDisableTiming));
    if (mode != AUDIOSYNC_CUDA_NARROW_OFF && !d.narrow_stream)
        ASC_CUDA_OK(cudaStreamCreateWithFlags(&d.narrow_stream, cudaStreamNonBlocking));
    const size_t total = p1 - p0;
    if (d.results.ensure(sizeof(audiosync_cuda_result) * total) != 0) return -1;
    if (d.h_results.ensure(sizeof(audiosync_cuda_result) * total) != 0) return -1;
    audiosync_cuda_result* d_res = static_cast<audiosync_cuda_result*>(d.results.p);
    if (shared_src && upload_from_host(d.in_src[0].p, sources, src_bytes, d.copy_stream, d.stage, pageable) != 0) return -1;
    int it = 0;
    for (size_t c0 = 0; c0 < total; c0 += chunk, it++) {
        const size_t n = std::min(chunk, total - c0);
        const int b = it & 1;
        const char* hs = sources + (shared_src ? 0 : (p0 + c0) * src_bytes);
        const char* hm = samples + (p0 + c0) * smp_bytes;
        if (it >= 2) {
            ASC_CUDA_OK(cudaStreamWaitEvent(d.copy_stream, d.ev_done[b], 0));
            if (mode != AUDIOSYNC_CUDA_NARROW_OFF) ASC_CUDA_OK(cudaStreamWaitEvent(d.narrow_stream, d.ev_done[b], 0));
        }
        // The chunk is fed in UNITS of g consecutive pairs (about 32 MB of doubles; one pair at the
        // headline length, hundreds at short ones, so that the per-unit bookkeeping never shows):
        // units [0, lo) go up as they are (unit lo too, partly, when dir_off > 0); units [hi, nu) narrowed.
        const size_t pair_bytes = src_bytes + smp_bytes;
        const size_t g = std::max<size_t>(1, ((size_t)32 << 20) / pair_bytes);
        const size_t nu = (n + g - 1) / g;
        auto unit_pairs = [&](size_t u) { return std::min(g, n - u * g); };
        size_t lo = 0, hi = nu, dir_off = 0;
        if (mode == AUDIOSYNC_CUDA_NARROW_OFF) {
            if ((!shared_src && upload_from_host(d.in_src[b].p, hs, src_bytes * n, d.copy_stream, d.stage, pageable) != 0) ||
                upload_from_host(d.in_smp[b].p, hm, smp_bytes * n, d.copy_stream, d.stage, pageable) != 0)
                return -1;
            lo = nu;
        }
        // the next slice of unit lo, as doubles, straight from the caller's (page-locked) memory:
        // first the unit's sources, then its samples (both contiguous)
        auto direct_slice = [&]() -> int {
            int k = 0;
            while (k < DeviceState::DIRECT_DEPTH - 1 && d.direct_pending[k]) k++;
            if (d.direct_pending[k]) ASC_CUDA_OK(cudaEventSynchronize(d.direct_ev[k]));
            const size_t up = unit_pairs(lo), usrc = up * src_bytes, usmp = up * smp_bytes;
            const bool in_src = dir_off < usrc;
            const size_t o = in_src ? dir_off : dir_off - usrc;
            const size_t m = std::min(DeviceState::DIRECT_SLICE, (in_src ? usrc : usmp) - o);
            char* dst = static_cast<char*>(in_src ? d.in_src[b].p : d.in_smp[b].p) + lo * g * (in_src ? src_bytes : smp_bytes) + o;
            const char* src = (in_src ? hs : hm) + lo * g * (in_src ? src_bytes : smp_bytes) + o;
            ASC_CUDA_OK(cudaMemcpyAsync(dst, src, m, cudaMemcpyHostToDevice, d.copy_stream));
            ASC_CUDA_OK(cudaEventRecord(d.direct_ev[k], d.copy_stream));
            d.direct_pending[k] = true;
            dir_off += m;
            if (dir_off == usrc + usmp) { lo++; dir_off = 0; }
            return 0;
        };
        // Direct slices only into link time the narrowed stream leaves idle: at most DIRECT_DEPTH
        // in flight, and only while the ring's uploads keep up with the conversion (the narrowed
        // form costs half the link bytes per pair, so it has the right of way; the copy threads,
        // not the link, bound it).  Called over and over while a piece is being narrowed.
        int feed_rc = 0;
        auto feed_direct = [&]() {
            while (feed_rc == 0 && (dir_off > 0 || lo < hi) && direct_in_flight(d) < feed_depth &&
                   ring_backlog(d.stage) <= feed_backlog)
                feed_rc = direct_slice();
        };
        while (lo < hi) {
            if (mode == AUDIOSYNC_CUDA_NARROW_OFF) {
                // narrowing was given up in this chunk: everything that is left goes up as doubles
                while (dir_off > 0)
                    if (direct_slice() != 0) return -1;
                if (lo < hi) {
                    const size_t p_lo = lo * g, p_hi = std::min(n, hi * g);
                    if (upload_from_host(static_cast<char*>(d.in_src[b].p) + p_lo * src_bytes, hs + p_lo * src_bytes, src_bytes * (p_hi - p_lo),
                                         d.copy_stream, d.stage, pageable) != 0 ||
                        upload_from_host(static_cast<char*>(d.in_smp[b].p) + p_lo * smp_bytes, hm + p_lo * smp_bytes, smp_bytes * (p_hi - p_lo),
                                         d.copy_stream, d.stage, pageable) != 0)
                        return -1;
                }
                lo = hi;
                break;
            }
            if (hybrid) feed_direct();
            if (feed_rc != 0) return -1;
            if (lo == hi) break;
            if (hi - 1 == lo && dir_off > 0) {          // only the partly fed unit is left
                while (dir_off > 0)
                    if (direct_slice() != 0) return -1;
                break;
            }
            // the next unit from the back, narrowed
            const size_t j = --hi, up = unit_pairs(j);
            bool exact = true;
            const bool stop = mode == AUDIOSYNC_CUDA_NARROW_LOSSLESS;
            std::function<void()> between;
            if (hybrid) between = feed_direct;
            if (upload_narrowed(static_cast<float*>(d.in_src32[b].p) + j * g * src_n, reinterpret_cast<const double*>(hs) + j * g * src_n,
                                up * src_n, d.narrow_stream, d.stage, &exact, stop, between) != 0)
                return -1;
            if ((exact || !stop) &&
                upload_narrowed(static_cast<float*>(d.in_smp32[b].p) + j * g * smp_n, reinterpret_cast<const double*>(hm) + j * g * smp_n,
                                up * smp_n, d.narrow_stream, d.stage, &exact, stop, between) != 0)
                return -1;
            if (feed_rc != 0) return -1;
            if (!exact && stop) { hi = j + 1; mode = AUDIOSYNC_CUDA_NARROW_OFF; }   // this unit and all later ones go up as doubles
        }
        // pairs [0, n_dbl): doubles (or the caller's fp32); pairs [p_nar, n): narrowed
        const size_t n_dbl = std::min(n, lo * g), p_nar = std::min(n, hi * g);
        if (n_dbl > 0) {
            ASC_CUDA_OK(cudaEventRecord(d.ev_up[b], d.copy_stream));
            ASC_CUDA_OK(cudaStreamWaitEvent(d.stream, d.ev_up[b], 0));
            // shared_src: the first chunk transforms the source, the later ones reuse its spectrum
            if (enqueue_batch(ctx, d, d.work, d.in_src[shared_src ? 0 : b].p, d.in_smp[b].p, n_dbl, L, dtype, d_res + c0, d.stream,
                              0, 0, shared_src, shared_src && c0 > 0) != 0)
                return -1;
        }
        if (p_nar < n) {
            ASC_CUDA_OK(cudaEventRecord(d.ev_up32[b], d.narrow_stream));
            ASC_CUDA_OK(cudaStreamWaitEvent(d.stream, d.ev_up32[b], 0));
            if (enqueue_batch(ctx, d, d.work, static_cast<float*>(d.in_src32[b].p) + p_nar * src_n,
                              static_cast<float*>(d.in_smp32[b].p) + p_nar * smp_n, n - p_nar, L, narrowed_dtype, d_res + c0 + p_nar, d.stream) != 0)
                return -1;
        }
        ASC_CUDA_OK(cudaEventRecord(d.ev_done[b], d.stream));
        if (dtype == AUDIOSYNC_CUDA_F64) { ctx->fed_direct += n_dbl; ctx->fed_narrowed += n - p_nar; }
    }
    ASC_CUDA_OK(cudaMemcpyAsync(d.h_results.p, d_res, sizeof(audiosync_cuda_result) * total,
                                cudaMemcpyDeviceToHost, d.stream));
    ASC_CUDA_OK(cudaStreamSynchronize(d.stream));
    memcpy(out + p0, d.h_results.p, sizeof(audiosync_cuda_result) * total);
    return 0;
}

}  // namespace asc

using namespace asc;

asc::DeviceState* audiosync_cuda_ctx::find(int device) {
    for (auto& d : devs)
        if (d.device == device) return &d;
    return nullptr;
}

// ------------------------------------------------- allocator registry / residency
// Blocks handed out by the FFTW-named allocators below.  cross_correlation() keeps its
// inputs device-resident across the interval schedule only when the source buffer is one of
// them (the reference allocates it with fftw_alloc_real, src/audiosync.c:189); any fftw_free
// bumps the generation and drops the session.
static std::mutex g_alloc_mu;
static std::map<const char*, size_t> g_allocs;          // user pointer -> bytes
static std::atomic<uint64_t> g_alloc_gen{1};
static std::atomic<int> g_residency{-1};                // -1: read AUDIOSYNC_CUDA_RESIDENT on first use
static std::atomic<uint64_t> g_dropin_calls{0}, g_dropin_h2d_bytes{0}, g_dropin_resident_hits{0};
static std::atomic<int> g_dropin_inflight{0}, g_dropin_inflight_max{0};

static bool residency_enabled() {
    int v = g_residency.load();
    if (v < 0) {
        const char* e = getenv("AUDIOSYNC_CUDA_RESIDENT");
        v = (e && atoi(e) != 0) ? 1 : 0;          // opt-in: the reference re-reads the host buffers on every call
        g_residency.store(v);
    }
    return v != 0;
}

// bytes of the library allocation that contains [p, p + need), 0 if none
static size_t library_block_bytes(const void* p, size_t need) {
    std::lock_guard<std::mutex> lk(g_alloc_mu);
    const char* c = static_cast<const char*>(p);
    auto it = g_allocs.upper_bound(c);
    if (it == g_allocs.begin()) return 0;
    --it;
    if (c < it->first || c + need > it->first + it->second) return 0;
    return (size_t)(it->first + it->second - c);
}

static void fingerprint(const double* buf, size_t n, size_t* idx, double* val) {
    for (int k = 0; k < ResidentSession::NFP; k++) {
        // evenly spread, odd offsets so a periodic refill cannot dodge every probe
        const size_t i = n == 0 ? 0 : ((size_t)k * n + (size_t)(37 * k + 11) % (n / ResidentSession::NFP + 1)) /
                                           ResidentSession::NFP;
        idx[k] = i < n ? i : (n ? n - 1 : 0);
        val[k] = n ? buf[idx[k]] : 0.0;
    }
}
static bool fingerprint_matches(const double* buf, const size_t* idx, const double* val) {
    for (int k = 0; k < ResidentSession::NFP; k++)
        if (memcmp(&buf[idx[k]], &val[k], sizeof(double)) != 0) return false;
    return true;
}

// ===========================================================================
// C ABI (the only symbols with default visibility)
// ===========================================================================
#pragma GCC visibility push(default)
extern "C" {

const char* audiosync_cuda_last_error(void) { return g_last_error; }
const char* audiosync_cuda_version(void) { return "audiosync_cuda 0.1 (sm_100a)"; }
void audiosync_cuda_set_debug(int on) { g_debug_flag = on; }
void audiosync_cuda_set_residency(int on) { g_residency.store(on ? 1 : 0); }
void audiosync_cuda_dropin_stats(uint64_t* calls, uint64_t* h2d_bytes, uint64_t* resident_hits) {
    if (calls) *calls = g_dropin_calls.load();
    if (h2d_bytes) *h2d_bytes = g_dropin_h2d_bytes.load();
    if (resident_hits) *resident_hits = g_dropin_resident_hits.load();
}

int audiosync_cuda_dropin_max_inflight(int reset) {
    return reset ? g_dropin_inflight_max.exchange(0) : g_dropin_inflight_max.load();
}

int audiosync_cuda_create(audiosync_cuda_ctx** out, const int* devices, int n_devices) {
    if (!out) return -1;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) {
        cudaGetLastError();
        set_last_error("no CUDA device available (this library has no CPU fallback)");
        return -1;
    }
    std::vector<int> ids;
    if (devices && n_devices > 0) ids.assign(devices, devices + n_devices);
    else for (int i = 0; i < count; i++) ids.push_back(i);
    auto* ctx = new audiosync_cuda_ctx();
    ctx->devs = std::vector<DeviceState>(ids.size());
    for (size_t i = 0; i < ids.size(); i++) {
        DeviceState& d = ctx->devs[i];
        cudaDeviceProp prop;
        if (ids[i] < 0 || ids[i] >= count || cudaSetDevice(ids[i]) != cudaSuccess ||
            cudaGetDeviceProperties(&prop, ids[i]) != cudaSuccess) {
            set_last_error("cannot use CUDA device %d", ids[i]);
            audiosync_cuda_destroy(ctx);
            return -1;
        }
        d.device = ids[i];
        d.sm_count = prop.multiProcessorCount;
        d.smem_optin = prop.sharedMemPerBlockOptin;
        // the only kernel image in this library is sm_100a
        cudaFuncAttributes fa;
        if (cudaFuncGetAttributes(&fa, argmax_f64_kernel) != cudaSuccess) {
            cudaGetLastError();
            set_last_error("device %d (%s, sm_%d%d) cannot run the sm_100a kernels of this library",
                           ids[i], prop.name, prop.major, prop.minor);
            audiosync_cuda_destroy(ctx);
            return -1;
        }
        if (cudaStreamCreateWithFlags(&d.stream, cudaStreamNonBlocking) != cudaSuccess ||
            cudaStreamCreateWithFlags(&d.copy_stream, cudaStreamNonBlocking) != cudaSuccess) {
            set_last_error("cudaStreamCreate failed on device %d", ids[i]);
            audiosync_cuda_destroy(ctx);
            return -1;
        }
    }
    const char* w = getenv("AUDIOSYNC_CUDA_WAVE_PAIRS");
    if (w) ctx->wave_pairs = atoi(w);
    const char* nh = getenv("AUDIOSYNC_CUDA_HOST_NARROWING");
    if (nh && atoi(nh) >= AUDIOSYNC_CUDA_NARROW_OFF && atoi(nh) <= AUDIOSYNC_CUDA_NARROW_ALWAYS) ctx->narrow_host = atoi(nh);
    *out = ctx;
    return 0;
}

void audiosync_cuda_destroy(audiosync_cuda_ctx* ctx) {
    if (!ctx) return;
    for (auto& sl : ctx->slots) {
        if (sl->dev && sl->dev->device >= 0) { cudaSetDevice(sl->dev->device); cudaDeviceSynchronize(); }
        sl->work.release(); sl->in_src.release(); sl->in_smp.release(); sl->d_res.release();
        sl->h_res.release(); sl->stage.release();
        if (sl->stream) cudaStreamDestroy(sl->stream);
    }
    ctx->slots.clear();
    ctx->resident.d_src.release(); ctx->resident.d_smp.release();
    for (auto& d : ctx->devs) destroy_device_state(d);
    delete ctx;
}

int audiosync_cuda_device_count(const audiosync_cuda_ctx* ctx) { return ctx ? (int)ctx->devs.size() : 0; }

int audiosync_cuda_set_path(audiosync_cuda_ctx* ctx, int path) {
    if (!ctx || path < AUDIOSYNC_CUDA_PATH_AUTO || path > AUDIOSYNC_CUDA_PATH_DIRECT) return -1;
    ctx->path = path;
    return 0;
}

int audiosync_cuda_set_precise(audiosync_cuda_ctx* ctx, int on) {
    if (!ctx) return -1;
    ctx->precise = on != 0;
    return 0;
}

int audiosync_cuda_set_weighting(audiosync_cuda_ctx* ctx, int mode) {
    if (!ctx || (mode != AUDIOSYNC_CUDA_WEIGHT_NONE && mode != AUDIOSYNC_CUDA_WEIGHT_PHAT)) {
        set_last_error("unknown weighting %d", mode);
        return -1;
    }
    ctx->weighting = mode;
    return 0;
}

int audiosync_cuda_set_lag_window(audiosync_cuda_ctx* ctx, int64_t lag_lo, int64_t lag_hi) {
    if (!ctx) { set_last_error("null argument"); return -1; }
    if (lag_lo > lag_hi) {
        set_last_error("lag window [%lld, %lld]: lag_lo > lag_hi", (long long)lag_lo, (long long)lag_hi);
        return -1;
    }
    ctx->lag_lo = lag_lo;
    ctx->lag_hi = lag_hi;
    return 0;
}

int audiosync_cuda_set_host_narrowing(audiosync_cuda_ctx* ctx, int mode) {
    if (!ctx || mode < AUDIOSYNC_CUDA_NARROW_OFF || mode > AUDIOSYNC_CUDA_NARROW_ALWAYS) return -1;
    ctx->narrow_host = mode;
    return 0;
}

int audiosync_cuda_copy_threads(void) { return (int)copy_pool().threads(); }

int audiosync_cuda_host_narrow(float* dst, const double* src, size_t n) {
    if (n == 0) return 1;
    if (!dst || !src) return 0;
    return copy_pool().narrow(dst, src, n) ? 1 : 0;
}

int audiosync_cuda_set_wave_pairs(audiosync_cuda_ctx* ctx, int pairs) {
    if (!ctx || pairs < 0) return -1;
    ctx->wave_pairs = pairs;
    return 0;
}

uint64_t audiosync_cuda_launch_count(const audiosync_cuda_ctx* ctx) {
    return ctx ? ctx->launches.load() : 0;
}

int audiosync_cuda_host_feed_stats(audiosync_cuda_ctx* ctx, uint64_t out[2], int reset) {
    if (!ctx || !out) return -1;
    out[0] = reset ? ctx->fed_direct.exchange(0) : ctx->fed_direct.load();
    out[1] = reset ? ctx->fed_narrowed.exchange(0) : ctx->fed_narrowed.load();
    return 0;
}

int audiosync_cuda_describe_plan(audiosync_cuda_ctx* ctx, size_t sample_len, char* buf, size_t buf_len) {
    if (!ctx || !buf || ctx->devs.empty()) return -1;
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceState& d = ctx->devs[0];
    if (cudaSetDevice(d.device) != cudaSuccess) return -1;
    FftPlan* plan = get_plan(ctx, d, (long long)sample_len);
    if (!plan) return -1;
    std::string desc = plan->desc;
    RawWindow w;
    long long lo = 0, hi = 0;
    if (raw_window_of(ctx->lag_lo, ctx->lag_hi, (long long)sample_len, &w, &lo, &hi) > 0)
        desc += " lags=[" + std::to_string(lo) + "," + std::to_string(hi) + "]";
    if (desc.size() + 1 > buf_len) return -1;
    memcpy(buf, desc.c_str(), desc.size() + 1);
    return (int)desc.size();
}

int audiosync_cuda_profile_enable(audiosync_cuda_ctx* ctx, int on) {
    if (!ctx) return -1;
    ctx->profile = on != 0;
    return 0;
}

int audiosync_cuda_profile_reset(audiosync_cuda_ctx* ctx) {
    if (!ctx) return -1;
    for (auto& d : ctx->devs) {
        if (drain_profile(d) != 0) return -1;
        for (int k = 0; k < KC_COUNT; k++) { d.prof_ms[k] = 0; d.prof_launches[k] = 0; }
    }
    return 0;
}

int audiosync_cuda_profile_read(audiosync_cuda_ctx* ctx, int i, char* name, size_t name_len,
                                uint64_t* launches, double* total_ms) {
    if (!ctx) return -1;
    if (i < 0 || i >= KC_COUNT) return KC_COUNT;
    uint64_t n = 0;
    double ms = 0;
    for (auto& d : ctx->devs) {
        if (drain_profile(d) != 0) return -1;
        n += d.prof_launches[i];
        ms += d.prof_ms[i];
    }
    if (name && name_len) snprintf(name, name_len, "%s", kernel_class_name(i));
    if (launches) *launches = n;
    if (total_ms) *total_ms = ms;
    return KC_COUNT;
}

int audiosync_cuda_synchronize(audiosync_cuda_ctx* ctx, int device) {
    if (!ctx) return -1;
    DeviceState* d = ctx->find(device);
    if (!d) { set_last_error("device %d is not part of this context", device); return -1; }
    ASC_CUDA_OK(cudaSetDevice(d->device));
    ASC_CUDA_OK(cudaDeviceSynchronize());
    return 0;
}

int audiosync_cuda_synth_pairs(audiosync_cuda_ctx* ctx, int device, uint64_t seed, uint64_t first_pair,
                               size_t n_pairs, size_t sample_len, int dtype, void* d_sources,
                               void* d_samples, void* stream) {
    if (!ctx || !d_sources || !d_samples) return -1;
    if (dtype != AUDIOSYNC_CUDA_F32 && dtype != AUDIOSYNC_CUDA_F64) { set_last_error("bad dtype"); return -1; }   // F32 / F64 only
    DeviceState* d = ctx->find(device);
    if (!d) { set_last_error("device %d is not part of this context", device); return -1; }
    if (n_pairs == 0) return 0;
    std::lock_guard<std::mutex> lk(d->mu);
    ASC_CUDA_OK(cudaSetDevice(d->device));
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : d->stream;
    const long long L = (long long)sample_len;
    const size_t esz = dtype_bytes(dtype);
    const unsigned bx = (unsigned)std::min<long long>((3 * L + 255) / 256, 4096);
    for (size_t p0 = 0; p0 < n_pairs; p0 += 32768) {
        const unsigned np = (unsigned)std::min<size_t>(32768, n_pairs - p0);
        const dim3 grid(bx, np);
        char* s = static_cast<char*>(d_sources) + p0 * (size_t)(2 * L) * esz;
        char* m = static_cast<char*>(d_samples) + p0 * (size_t)L * esz;
        int rc = -1;
        if (dtype == AUDIOSYNC_CUDA_F32)
            rc = launch(ctx, *d, KC_SYNTH, st, [&] {
                synth_kernel<float><<<grid, 256, 0, st>>>(reinterpret_cast<float*>(s),
                                                          reinterpret_cast<float*>(m), seed, first_pair + p0, L);
            });
        else if (dtype == AUDIOSYNC_CUDA_F64)
            rc = launch(ctx, *d, KC_SYNTH, st, [&] {
                synth_kernel<double><<<grid, 256, 0, st>>>(reinterpret_cast<double*>(s),
                                                           reinterpret_cast<double*>(m), seed, first_pair + p0, L);
            });
        if (rc != 0) return -1;
    }
    return 0;
}

// xcorr_batch_device and xcorr_shared_source_device
static int batch_device(audiosync_cuda_ctx* ctx, int device, const void* d_sources, const void* d_samples, size_t n_pairs,
                        size_t sample_len, int dtype, audiosync_cuda_result* d_results, void* stream, bool shared_src) {
    if (!ctx || !d_sources || !d_samples || !d_results) { set_last_error("null argument"); return -1; }
    if (dtype != AUDIOSYNC_CUDA_F32 && dtype != AUDIOSYNC_CUDA_F64 && dtype != AUDIOSYNC_CUDA_S16) { set_last_error("bad dtype"); return -1; }
    DeviceState* d = ctx->find(device);
    if (!d) { set_last_error("device %d is not part of this context", device); return -1; }
    std::lock_guard<std::mutex> lk(d->mu);      // per device: threads driving different devices do not serialise
    cudaStream_t st = stream ? static_cast<cudaStream_t>(stream) : d->stream;
    return enqueue_batch(ctx, *d, d->work, d_sources, d_samples, n_pairs, (long long)sample_len, dtype, d_results, st,
                         0, 0, shared_src);
}

int audiosync_cuda_xcorr_batch_device(audiosync_cuda_ctx* ctx, int device, const void* d_sources,
                                      const void* d_samples, size_t n_pairs, size_t sample_len,
                                      int dtype, audiosync_cuda_result* d_results, void* stream) {
    return batch_device(ctx, device, d_sources, d_samples, n_pairs, sample_len, dtype, d_results, stream, false);
}

int audiosync_cuda_xcorr_shared_source_device(audiosync_cuda_ctx* ctx, int device, const void* d_source,
                                              const void* d_samples, size_t n_pairs, size_t sample_len,
                                              int dtype, audiosync_cuda_result* d_results, void* stream) {
    return batch_device(ctx, device, d_source, d_samples, n_pairs, sample_len, dtype, d_results, stream, true);
}

// xcorr_batch_results and xcorr_shared_source
static int batch_results(audiosync_cuda_ctx* ctx, const void* sources, const void* samples, size_t n_pairs,
                         size_t sample_len, int dtype, int memspace, audiosync_cuda_result* results, bool shared_src) {
    if (!ctx || !sources || !samples || (!results && n_pairs)) { set_last_error("null argument"); return -1; }
    if (dtype != AUDIOSYNC_CUDA_F32 && dtype != AUDIOSYNC_CUDA_F64 && dtype != AUDIOSYNC_CUDA_S16) { set_last_error("bad dtype"); return -1; }
    if (n_pairs == 0) return 0;
    if (sample_len == 0) { set_last_error("sample_len must be > 0"); return -1; }
    std::lock_guard<std::mutex> lk(ctx->mu);
    const long long L = (long long)sample_len;
    RawWindow win;
    if (lag_window(ctx, L, &win) < 0) return -1;     // before any copy: nothing is written
    int rc = 0;
    if (memspace == AUDIOSYNC_CUDA_DEVICE) {
        cudaPointerAttributes at;
        ASC_CUDA_OK(cudaPointerGetAttributes(&at, sources));
        DeviceState* d = ctx->find(at.device);
        if (at.type != cudaMemoryTypeDevice || !d) {
            set_last_error("device-memspace pointers must live on a device of the context");
            return -1;
        }
        std::lock_guard<std::mutex> dlk(d->mu);
        ASC_CUDA_OK(cudaSetDevice(d->device));
        if (d->results.ensure(sizeof(audiosync_cuda_result) * n_pairs) != 0) return -1;
        auto* d_res = static_cast<audiosync_cuda_result*>(d->results.p);
        if (enqueue_batch(ctx, *d, d->work, sources, samples, n_pairs, L, dtype, d_res, d->stream, 0, 0, shared_src) != 0) return -1;
        ASC_CUDA_OK(cudaMemcpyAsync(results, d_res, sizeof(audiosync_cuda_result) * n_pairs,
                                    cudaMemcpyDeviceToHost, d->stream));
        ASC_CUDA_OK(cudaStreamSynchronize(d->stream));
    } else {
        // contiguous block split over the devices, one host thread per device
        const size_t G = ctx->devs.size();
        std::vector<int> rcs(G, 0);
        std::vector<std::string> errs(G);
        std::vector<std::thread> th;
        const size_t base = n_pairs / G, rem = n_pairs % G;
        const bool solo = G == 1 || n_pairs == 1;      // one device fed by this call: the copy threads are its own
        size_t p0 = 0;
        for (size_t g = 0; g < G; g++) {
            const size_t cnt = base + (g < rem ? 1 : 0);
            const size_t a = p0, b = p0 + cnt;
            p0 = b;
            if (cnt == 0) continue;
            auto work = [&, g, a, b] {
                rcs[g] = run_host_range(ctx, ctx->devs[g], static_cast<const char*>(sources),
                                        static_cast<const char*>(samples), a, b, L, dtype, results, solo, shared_src);
                if (rcs[g] != 0) errs[g] = take_last_error();   // the worker's thread-local message
            };
            if (G == 1) work(); else th.emplace_back(work);
        }
        for (auto& t : th) t.join();
        for (size_t g = 0; g < G; g++)
            if (rcs[g] != 0) {
                if (rc == 0) adopt_last_error(errs[g]);           // first failing device, for audiosync_cuda_last_error()
                rc = -1;
            }
        if (rc != 0) return -1;
    }
    return 0;
}

int audiosync_cuda_xcorr_batch_results(audiosync_cuda_ctx* ctx, const void* sources, const void* samples,
                                       size_t n_pairs, size_t sample_len, int dtype, int memspace,
                                       audiosync_cuda_result* results) {
    return batch_results(ctx, sources, samples, n_pairs, sample_len, dtype, memspace, results, false);
}

int audiosync_cuda_xcorr_shared_source(audiosync_cuda_ctx* ctx, const void* source, const void* samples,
                                       size_t n_pairs, size_t sample_len, int dtype, int memspace,
                                       audiosync_cuda_result* results) {
    return batch_results(ctx, source, samples, n_pairs, sample_len, dtype, memspace, results, true);
}

int audiosync_cuda_xcorr_batch(audiosync_cuda_ctx* ctx, const void* sources, const void* samples,
                               size_t n_pairs, size_t sample_len, int dtype, int memspace, long* lags,
                               double* coefs, int* rets, double* peaks) {
    std::vector<audiosync_cuda_result> res(n_pairs);
    if (audiosync_cuda_xcorr_batch_results(ctx, sources, samples, n_pairs, sample_len, dtype, memspace,
                                           res.data()) != 0)
        return -1;
    for (size_t i = 0; i < n_pairs; i++) {
        if (lags) lags[i] = (long)res[i].lag;
        if (coefs) coefs[i] = res[i].coef;
        if (rets) rets[i] = res[i].ret;
        if (peaks) peaks[i] = res[i].peak;
    }
    return 0;
}


// ------------------------------------------------------------------ session pool
}  // extern "C"
#pragma GCC visibility pop

struct audiosync_cuda_pool {
    audiosync_cuda_ctx* ctx = nullptr;
    asc::DeviceState* dev = nullptr;
    size_t n_slots = 0, max_len = 0;
    long long src_pitch = 0, smp_pitch = 0;      // elements; multiples of 4 (16-byte rows for TMA-staged tiles)
    int dtype = AUDIOSYNC_CUDA_F64;
    asc::DevBuf src, smp;
    // fp32 slots: arriving doubles land in one of two staging buffers (copy stream) and are
    // converted into the slot by a kernel on the pool's own stream, so the H2D copy of piece k + 1
    // overlaps the conversion of piece k
    asc::DevBuf stage[2];
    cudaEvent_t ev_copied[2] = {nullptr, nullptr}, ev_converted[2] = {nullptr, nullptr};
    bool conv_pending[2] = {false, false};
    int next_stage = 0;
    cudaStream_t conv_stream = nullptr;
    cudaEvent_t ev_arrived = nullptr;            // everything appended so far is in the slots
    bool dirty = false;                          // appends enqueued since the last flush / run
    std::vector<size_t> have_src, have_smp;
};

namespace asc {
static int pool_upload(audiosync_cuda_pool* pool, DevBuf& slab, size_t elem_off, const double* host, size_t n) {
    DeviceState& d = *pool->dev;
    if (n == 0) return 0;
    const bool pageable = host_pointer_is_pageable(host);
    pool->dirty = true;
    if (pool->dtype == AUDIOSYNC_CUDA_F64)
        return upload_from_host(static_cast<double*>(slab.p) + elem_off, host, sizeof(double) * n, d.copy_stream, d.stage, pageable);
    const size_t piece = 1u << 20;               // doubles per piece: 8 MB
    for (size_t o = 0; o < n; o += piece) {
        const size_t m = std::min(piece, n - o);
        const int k = pool->next_stage;
        pool->next_stage ^= 1;
        if (pool->stage[k].ensure(sizeof(double) * piece) != 0) return -1;
        if (pool->conv_pending[k]) ASC_CUDA_OK(cudaStreamWaitEvent(d.copy_stream, pool->ev_converted[k], 0));
        if (upload_from_host(pool->stage[k].p, host + o, sizeof(double) * m, d.copy_stream, d.stage, pageable) != 0) return -1;
        ASC_CUDA_OK(cudaEventRecord(pool->ev_copied[k], d.copy_stream));
        ASC_CUDA_OK(cudaStreamWaitEvent(pool->conv_stream, pool->ev_copied[k], 0));
        const unsigned blocks = (unsigned)std::min<size_t>((m + 255) / 256, 2048);
        if (launch(pool->ctx, d, KC_SYNTH, pool->conv_stream, [&] {
                convert_f64_to_f32_kernel<<<blocks, 256, 0, pool->conv_stream>>>(
                    static_cast<const double*>(pool->stage[k].p), static_cast<float*>(slab.p) + elem_off + o, (long long)m);
            }) != 0) return -1;
        ASC_CUDA_OK(cudaEventRecord(pool->ev_converted[k], pool->conv_stream));
        pool->conv_pending[k] = true;
    }
    return 0;
}
// `st` waits until every frame appended so far is in its slot
static int pool_order_after_appends(audiosync_cuda_pool* pool, cudaStream_t st) {
    DeviceState& d = *pool->dev;
    if (!pool->dirty) return 0;
    ASC_CUDA_OK(cudaEventRecord(pool->ev_arrived, d.copy_stream));
    ASC_CUDA_OK(cudaStreamWaitEvent(st, pool->ev_arrived, 0));
    if (pool->dtype == AUDIOSYNC_CUDA_F32) {
        ASC_CUDA_OK(cudaEventRecord(pool->ev_arrived, pool->conv_stream));
        ASC_CUDA_OK(cudaStreamWaitEvent(st, pool->ev_arrived, 0));
    }
    return 0;
}
}  // namespace asc

#pragma GCC visibility push(default)
extern "C" {

int audiosync_cuda_pool_create(audiosync_cuda_ctx* ctx, int device, size_t n_slots, size_t max_sample_len,
                               int dtype, audiosync_cuda_pool** out) {
    if (!ctx || !out || n_slots == 0 || max_sample_len == 0) { set_last_error("pool_create: invalid argument"); return -1; }
    if (dtype != AUDIOSYNC_CUDA_F32 && dtype != AUDIOSYNC_CUDA_F64) { set_last_error("bad dtype"); return -1; }
    *out = nullptr;
    DeviceState* d = ctx->find(device);
    if (!d) { set_last_error("device %d is not part of this context", device); return -1; }
    ASC_CUDA_OK(cudaSetDevice(d->device));
    auto* pool = new audiosync_cuda_pool();
    pool->ctx = ctx; pool->dev = d; pool->n_slots = n_slots; pool->max_len = max_sample_len; pool->dtype = dtype;
    pool->smp_pitch = (long long)((max_sample_len + 3) / 4 * 4);
    pool->src_pitch = 2 * pool->smp_pitch;
    const size_t esz = dtype_bytes(dtype);
    if (pool->src.ensure(esz * (size_t)pool->src_pitch * n_slots) != 0 ||
        pool->smp.ensure(esz * (size_t)pool->smp_pitch * n_slots) != 0) {
        audiosync_cuda_pool_destroy(pool);
        return -1;
    }
    pool->have_src.assign(n_slots, 0);
    pool->have_smp.assign(n_slots, 0);
    bool ok = cudaStreamCreateWithFlags(&pool->conv_stream, cudaStreamNonBlocking) == cudaSuccess &&
              cudaEventCreateWithFlags(&pool->ev_arrived, cudaEventDisableTiming) == cudaSuccess;
    for (int k = 0; k < 2 && ok; k++)
        ok = cudaEventCreateWithFlags(&pool->ev_copied[k], cudaEventDisableTiming) == cudaSuccess &&
             cudaEventCreateWithFlags(&pool->ev_converted[k], cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        set_last_error("pool_create: cannot create streams / events");
        audiosync_cuda_pool_destroy(pool);
        return -1;
    }
    *out = pool;
    return 0;
}

void audiosync_cuda_pool_destroy(audiosync_cuda_pool* pool) {
    if (!pool) return;
    if (pool->dev && pool->dev->device >= 0) { cudaSetDevice(pool->dev->device); cudaDeviceSynchronize(); }
    pool->src.release(); pool->smp.release(); pool->stage[0].release(); pool->stage[1].release();
    for (int k = 0; k < 2; k++) {
        if (pool->ev_copied[k]) cudaEventDestroy(pool->ev_copied[k]);
        if (pool->ev_converted[k]) cudaEventDestroy(pool->ev_converted[k]);
    }
    if (pool->ev_arrived) cudaEventDestroy(pool->ev_arrived);
    if (pool->conv_stream) cudaStreamDestroy(pool->conv_stream);
    delete pool;
}

int audiosync_cuda_pool_reset(audiosync_cuda_pool* pool, size_t slot) {
    if (!pool || slot >= pool->n_slots) { set_last_error("pool_reset: bad slot"); return -1; }
    std::lock_guard<std::mutex> lk(pool->ctx->mu);
    pool->have_src[slot] = 0;
    pool->have_smp[slot] = 0;
    return 0;
}

int audiosync_cuda_pool_fill(const audiosync_cuda_pool* pool, size_t slot, size_t* source_frames, size_t* sample_frames) {
    if (!pool || slot >= pool->n_slots) return -1;
    if (source_frames) *source_frames = pool->have_src[slot];
    if (sample_frames) *sample_frames = pool->have_smp[slot];
    return 0;
}

int audiosync_cuda_pool_append_async(audiosync_cuda_pool* pool, size_t slot, const double* source_frames, size_t n_source,
                                     const double* sample_frames, size_t n_sample) {
    if (!pool || slot >= pool->n_slots || (n_source && !source_frames) || (n_sample && !sample_frames)) {
        set_last_error("pool_append: invalid argument");
        return -1;
    }
    std::lock_guard<std::mutex> lk(pool->ctx->mu);
    if (pool->have_src[slot] + n_source > 2 * pool->max_len || pool->have_smp[slot] + n_sample > pool->max_len) {
        set_last_error("pool_append: slot %zu would exceed its capacity (%zu source / %zu sample frames)", slot,
                       2 * pool->max_len, pool->max_len);
        return -1;
    }
    DeviceState& d = *pool->dev;
    std::lock_guard<std::mutex> dlk(d.mu);
    ASC_CUDA_OK(cudaSetDevice(d.device));
    if (pool_upload(pool, pool->src, slot * (size_t)pool->src_pitch + pool->have_src[slot], source_frames, n_source) != 0 ||
        pool_upload(pool, pool->smp, slot * (size_t)pool->smp_pitch + pool->have_smp[slot], sample_frames, n_sample) != 0)
        return -1;
    pool->have_src[slot] += n_source;
    pool->have_smp[slot] += n_sample;
    return 0;
}

int audiosync_cuda_pool_flush(audiosync_cuda_pool* pool) {
    if (!pool) return -1;
    std::lock_guard<std::mutex> lk(pool->ctx->mu);
    DeviceState& d = *pool->dev;
    std::lock_guard<std::mutex> dlk(d.mu);
    ASC_CUDA_OK(cudaSetDevice(d.device));
    ASC_CUDA_OK(cudaStreamSynchronize(d.copy_stream));
    ASC_CUDA_OK(cudaStreamSynchronize(pool->conv_stream));
    pool->dirty = false;
    return 0;
}

int audiosync_cuda_pool_append(audiosync_cuda_pool* pool, size_t slot, const double* source_frames, size_t n_source,
                               const double* sample_frames, size_t n_sample) {
    if (audiosync_cuda_pool_append_async(pool, slot, source_frames, n_source, sample_frames, n_sample) != 0) return -1;
    return audiosync_cuda_pool_flush(pool);       // the frames are resident when this returns
}

int audiosync_cuda_pool_run(audiosync_cuda_pool* pool, size_t first_slot, size_t n_slots, size_t sample_len,
                            audiosync_cuda_result* results) {
    if (!pool || !results || sample_len == 0 || n_slots == 0 || first_slot + n_slots > pool->n_slots ||
        sample_len > pool->max_len) {
        set_last_error("pool_run: invalid argument");
        return -1;
    }
    std::lock_guard<std::mutex> lk(pool->ctx->mu);
    for (size_t s = first_slot; s < first_slot + n_slots; s++) {
        if (pool->have_src[s] < 2 * sample_len || pool->have_smp[s] < sample_len) {
            set_last_error("pool_run: slot %zu holds %zu / %zu frames, interval %zu needs %zu / %zu", s,
                           pool->have_src[s], pool->have_smp[s], sample_len, 2 * sample_len, sample_len);
            return -1;
        }
    }
    DeviceState& d = *pool->dev;
    std::lock_guard<std::mutex> dlk(d.mu);
    ASC_CUDA_OK(cudaSetDevice(d.device));
    if (d.results.ensure(sizeof(audiosync_cuda_result) * n_slots) != 0 ||
        d.h_results.ensure(sizeof(audiosync_cuda_result) * n_slots) != 0)
        return -1;
    const size_t esz = dtype_bytes(pool->dtype);
    const char* s0 = static_cast<const char*>(pool->src.p) + first_slot * (size_t)pool->src_pitch * esz;
    const char* m0 = static_cast<const char*>(pool->smp.p) + first_slot * (size_t)pool->smp_pitch * esz;
    auto* d_res = static_cast<audiosync_cuda_result*>(d.results.p);
    if (pool_order_after_appends(pool, d.stream) != 0) return -1;
    if (enqueue_batch(pool->ctx, d, d.work, s0, m0, n_slots, (long long)sample_len, pool->dtype, d_res, d.stream,
                      pool->src_pitch, pool->smp_pitch) != 0)
        return -1;
    ASC_CUDA_OK(cudaMemcpyAsync(d.h_results.p, d_res, sizeof(audiosync_cuda_result) * n_slots,
                                cudaMemcpyDeviceToHost, d.stream));
    ASC_CUDA_OK(cudaStreamSynchronize(d.stream));
    pool->dirty = false;                          // d.stream waited for every append
    memcpy(results, d.h_results.p, sizeof(audiosync_cuda_result) * n_slots);
    return 0;
}

// ------------------------------------------------------------ default context
static audiosync_cuda_ctx* g_default_ctx = nullptr;
static std::mutex g_default_mu;

// Devices of the default context: AUDIOSYNC_CUDA_DEVICE=k (one device, default 0) or
// AUDIOSYNC_CUDA_DEVICES=all | i,j,... (concurrent drop-in callers are spread round-robin over
// them).  AUDIOSYNC_CUDA_DROPIN_SLOTS = in-flight calls per device (default 3).
static audiosync_cuda_ctx* default_ctx() {
    std::lock_guard<std::mutex> lk(g_default_mu);
    if (!g_default_ctx) {
        std::vector<int> ids;
        const char* many = getenv("AUDIOSYNC_CUDA_DEVICES");
        if (many && strcmp(many, "all") != 0) {
            for (const char* q = many; *q;) {
                char* end = nullptr;
                const long v = strtol(q, &end, 10);
                if (end == q) break;
                ids.push_back((int)v);
                q = (*end == ',') ? end + 1 : end;
            }
        } else if (!many) {
            const char* e = getenv("AUDIOSYNC_CUDA_DEVICE");
            ids.push_back(e ? atoi(e) : 0);
        }
        audiosync_cuda_ctx* c = nullptr;
        if (audiosync_cuda_create(&c, ids.empty() ? nullptr : ids.data(), (int)ids.size()) != 0) return nullptr;
        const char* p = getenv("AUDIOSYNC_CUDA_PATH");
        if (p && !strcmp(p, "direct")) c->path = AUDIOSYNC_CUDA_PATH_DIRECT;
        const char* pr = getenv("AUDIOSYNC_CUDA_PRECISE");
        if (pr && atoi(pr) != 0) c->precise = true;
        const char* ns = getenv("AUDIOSYNC_CUDA_DROPIN_SLOTS");
        const int per_dev = std::max(1, std::min(16, ns ? atoi(ns) : 3));
        for (int k = 0; k < per_dev; k++)
            for (auto& d : c->devs) {
                auto slot = std::make_unique<DropinSlot>();
                slot->dev = &d;
                if (cudaSetDevice(d.device) != cudaSuccess ||
                    cudaStreamCreateWithFlags(&slot->stream, cudaStreamNonBlocking) != cudaSuccess) {
                    set_last_error("cannot create a stream for drop-in callers on device %d", d.device);
                    audiosync_cuda_destroy(c);
                    return nullptr;
                }
                c->slots.push_back(std::move(slot));
            }
        g_default_ctx = c;
    }
    return g_default_ctx;
}

namespace {
// A free slot, round-robin over the slots (and with them over the devices); waits when all are busy.
struct SlotLease {
    audiosync_cuda_ctx* ctx;
    DropinSlot* slot = nullptr;
    explicit SlotLease(audiosync_cuda_ctx* c) : ctx(c) {
        std::unique_lock<std::mutex> lk(ctx->slot_mu);
        for (;;) {
            const size_t n = ctx->slots.size();
            for (size_t k = 0; k < n; k++) {
                DropinSlot* s = ctx->slots[(ctx->slot_next + k) % n].get();
                if (!s->busy) {
                    s->busy = true;
                    ctx->slot_next = (ctx->slot_next + k + 1) % n;
                    slot = s;
                    const int now = g_dropin_inflight.fetch_add(1) + 1;
                    int seen = g_dropin_inflight_max.load();
                    while (now > seen && !g_dropin_inflight_max.compare_exchange_weak(seen, now)) {}
                    return;
                }
            }
            ctx->slot_cv.wait(lk);
        }
    }
    ~SlotLease() {
        g_dropin_inflight.fetch_sub(1);
        { std::lock_guard<std::mutex> lk(ctx->slot_mu); slot->busy = false; }
        ctx->slot_cv.notify_one();
    }
};
}  // namespace

// The resident form of the call (opt-in, see audiosync_cuda_set_residency): one session, the
// context's own stream and scratch, serialised on the context mutex.
static int cross_correlation_resident(audiosync_cuda_ctx* ctx, size_t block, double* source, double* input_sample,
                                      long long L, audiosync_cuda_result* out) {
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceState& d = ctx->devs[0];
    std::lock_guard<std::mutex> dlk(d.mu);
    ASC_CUDA_OK(cudaSetDevice(d.device));
    if (d.results.ensure(sizeof(audiosync_cuda_result)) != 0 ||
        d.h_results.ensure(sizeof(audiosync_cuda_result)) != 0)
        return -1;
    auto* d_res = static_cast<audiosync_cuda_result*>(d.results.p);
    const size_t src_n = (size_t)(2 * L), smp_n = (size_t)L;
    ResidentSession& s = ctx->resident;
    bool hit = s.src == source && s.smp == input_sample && (size_t)L > s.L && s.L != 0 &&
               s.alloc_gen == g_alloc_gen.load() && s.src_valid <= src_n && s.smp_valid <= smp_n &&
               fingerprint_matches(source, s.fp_idx_src, s.fp_val_src) &&
               fingerprint_matches(input_sample, s.fp_idx_smp, s.fp_val_smp);
    // device mirrors sized for the whole host block, so they never move while a session lives
    const size_t cap_src = std::max(block, src_n * sizeof(double));
    const size_t cap_smp = std::max(block / 2, smp_n * sizeof(double));
    if (cap_src > s.d_src.bytes || cap_smp > s.d_smp.bytes) hit = false;
    if (!hit) {
        s.invalidate();
        if (s.d_src.ensure(cap_src) != 0 || s.d_smp.ensure(cap_smp) != 0) return -1;
    } else {
        g_dropin_resident_hits.fetch_add(1, std::memory_order_relaxed);
    }
    const size_t new_src = src_n - s.src_valid, new_smp = smp_n - s.smp_valid;
    const bool pageable_smp = host_pointer_is_pageable(input_sample);
    ASC_CUDA_OK(cudaMemcpyAsync(static_cast<double*>(s.d_src.p) + s.src_valid, source + s.src_valid,
                                sizeof(double) * new_src, cudaMemcpyHostToDevice, d.stream));
    if (upload_from_host(static_cast<double*>(s.d_smp.p) + s.smp_valid, input_sample + s.smp_valid,
                         sizeof(double) * new_smp, d.stream, d.stage, pageable_smp) != 0) return -1;
    g_dropin_h2d_bytes.fetch_add(sizeof(double) * (new_src + new_smp), std::memory_order_relaxed);
    s.src = source; s.smp = input_sample; s.L = (size_t)L; s.src_valid = src_n; s.smp_valid = smp_n;
    s.alloc_gen = g_alloc_gen.load();
    fingerprint(source, src_n, s.fp_idx_src, s.fp_val_src);
    fingerprint(input_sample, smp_n, s.fp_idx_smp, s.fp_val_smp);
    if (enqueue_batch(ctx, d, d.work, s.d_src.p, s.d_smp.p, 1, L, AUDIOSYNC_CUDA_F64, d_res, d.stream) != 0) {
        ctx->resident.invalidate();
        return -1;
    }
    ASC_CUDA_OK(cudaMemcpyAsync(d.h_results.p, d_res, sizeof(audiosync_cuda_result), cudaMemcpyDeviceToHost, d.stream));
    ASC_CUDA_OK(cudaStreamSynchronize(d.stream));
    *out = *static_cast<audiosync_cuda_result*>(d.h_results.p);
    return 0;
}

// ---- Part 1: drop-in for reference src/cross_correlation.c -----------------
int cross_correlation(double* source, double* input_sample, const size_t sample_len, long* lag,
                      double* coefficient) {
    if (!source || !input_sample || !lag || !coefficient || sample_len == 0) {
        set_last_error("cross_correlation: invalid argument");
        return -1;
    }
    audiosync_cuda_ctx* ctx = default_ctx();
    if (!ctx) return -1;
    const long long L = (long long)sample_len;
    const size_t src_n = (size_t)(2 * L), smp_n = (size_t)L;
    g_dropin_calls.fetch_add(1, std::memory_order_relaxed);
    audiosync_cuda_result r;
    // Residency (SURVEY 8f rank 1, opt-in): the interval loop of src/audiosync.c:226-259 passes the
    // same buffers with a growing sample_len; only the frames that arrived since the last call are
    // uploaded.  Taken only for a source from this library's allocator, a strictly larger
    // sample_len, an unchanged allocator generation and matching fingerprints of both prefixes.
    const size_t block = residency_enabled() ? library_block_bytes(source, src_n * sizeof(double)) : 0;
    if (block != 0) {
        if (cross_correlation_resident(ctx, block, source, input_sample, L, &r) != 0) return -1;
    } else {
        // Default: like the reference, every call reads the host buffers afresh.  Each caller
        // leases a slot (stream + mirrors + scratch), so concurrent callers overlap.
        SlotLease lease(ctx);
        DropinSlot& sl = *lease.slot;
        DeviceState& d = *sl.dev;
        ASC_CUDA_OK(cudaSetDevice(d.device));
        if (sl.in_src.ensure(sizeof(double) * src_n) != 0 || sl.in_smp.ensure(sizeof(double) * smp_n) != 0 ||
            sl.d_res.ensure(sizeof(audiosync_cuda_result)) != 0 || sl.h_res.ensure(sizeof(audiosync_cuda_result)) != 0)
            return -1;
        // snapshot exactly the prefixes the reference reads (src/cross_correlation.c:164, :204-213)
        if (upload_from_host(sl.in_src.p, source, sizeof(double) * src_n, sl.stream, sl.stage,
                             host_pointer_is_pageable(source)) != 0 ||
            upload_from_host(sl.in_smp.p, input_sample, sizeof(double) * smp_n, sl.stream, sl.stage,
                             host_pointer_is_pageable(input_sample)) != 0)
            return -1;
        g_dropin_h2d_bytes.fetch_add(sizeof(double) * (src_n + smp_n), std::memory_order_relaxed);
        auto* d_res = static_cast<audiosync_cuda_result*>(sl.d_res.p);
        if (enqueue_batch(ctx, d, sl.work, sl.in_src.p, sl.in_smp.p, 1, L, AUDIOSYNC_CUDA_F64, d_res, sl.stream) != 0)
            return -1;
        ASC_CUDA_OK(cudaMemcpyAsync(sl.h_res.p, d_res, sizeof(audiosync_cuda_result), cudaMemcpyDeviceToHost, sl.stream));
        ASC_CUDA_OK(cudaStreamSynchronize(sl.stream));
        r = *static_cast<audiosync_cuda_result*>(sl.h_res.p);
    }
    *lag = (long)r.lag;                 // written before the NaN gate, like :259/:272
    *coefficient = r.coef;
    if (r.ret != 0) return -1;          // :276
    if (debug_on())                     // :278, LOG() format of audiosync.h:88-94
        fprintf(stderr, "\x1B[36maudiosync: \x1B[0m%ld frames of delay with a confidence of %f\n",
                *lag, *coefficient);
    return 0;
}

double pearson_coefficient(double* source_start, const double* source_end, double* sample_start,
                           const double* sample_end) {
    const double nan = std::numeric_limits<double>::quiet_NaN();
    if (!source_start || !source_end || !sample_start || !sample_end) return nan;
    const long long n = (long long)(source_end - source_start);
    if (n < 0 || (long long)(sample_end - sample_start) != n) {
        set_last_error("pearson_coefficient: ranges must have equal, non-negative length");
        return nan;
    }
    if (n == 0) return nan;             // 0/0 in the reference
    audiosync_cuda_ctx* ctx = default_ctx();
    if (!ctx) return nan;
    std::lock_guard<std::mutex> lk(ctx->mu);
    DeviceState& d = ctx->devs[0];
    std::lock_guard<std::mutex> dlk(d.mu);
    auto fail = [&]() { return nan; };
    if (cudaSetDevice(d.device) != cudaSuccess) return fail();
    const int n_chunks = (int)((n + PEARSON_CHUNK - 1) / PEARSON_CHUNK);
    if (d.in_src[0].ensure(sizeof(double) * n) != 0 || d.in_smp[0].ensure(sizeof(double) * n) != 0 ||
        d.work.partials.ensure(sizeof(PearsonPartial) * n_chunks) != 0 ||
        d.results.ensure(sizeof(audiosync_cuda_result)) != 0 ||
        d.h_results.ensure(sizeof(audiosync_cuda_result)) != 0)
        return fail();
    cudaStream_t st = d.stream;
    auto* d_res = static_cast<audiosync_cuda_result*>(d.results.p);
    auto* partials = static_cast<PearsonPartial*>(d.work.partials.p);
    if (cudaMemcpyAsync(d.in_src[0].p, source_start, sizeof(double) * n, cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemcpyAsync(d.in_smp[0].p, sample_start, sizeof(double) * n, cudaMemcpyHostToDevice, st) != cudaSuccess) {
        set_last_error("pearson_coefficient: upload failed");
        return fail();
    }
    if (ensure_tickets(d.work, 1) != 0) return fail();
    if (launch(ctx, d, KC_PEARSON, st, [&] {
            pearson_kernel<double, true><<<dim3(n_chunks, 1), PEARSON_THREADS, 0, st>>>(
                static_cast<const double*>(d.in_src[0].p), static_cast<const double*>(d.in_smp[0].p), 0, 0,
                n, nullptr, n, 1.0, partials, static_cast<unsigned int*>(d.work.tickets.p), n_chunks, d_res);
        }) != 0) return fail();
    if (cudaMemcpyAsync(d.h_results.p, d_res, sizeof(audiosync_cuda_result), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
        cudaStreamSynchronize(st) != cudaSuccess) {
        set_last_error("pearson_coefficient: %s", cudaGetErrorString(cudaGetLastError()));
        return fail();
    }
    return static_cast<audiosync_cuda_result*>(d.h_results.p)->coef;
}

// ---- Part 2: FFTW-named allocators (reference src/audiosync.c:189,277) -------
// A small header in front of every block remembers how it was obtained.
struct AllocHeader { uint64_t magic; uint64_t pinned; void* base; uint64_t pad; };
static const uint64_t ALLOC_MAGIC = 0xA5D10C0DAFF7E11AULL;

void* fftw_malloc(size_t n_bytes) {
    const size_t total = n_bytes + 64;
    void* base = nullptr;
    uint64_t pinned = 0;
    int count = 0;
    if (cudaGetDeviceCount(&count) == cudaSuccess && count > 0 &&
        cudaMallocHost(&base, total) == cudaSuccess) {
        pinned = 1;
    } else {
        cudaGetLastError();
        base = nullptr;
        if (posix_memalign(&base, 64, total) != 0) return nullptr;
    }
    AllocHeader* h = reinterpret_cast<AllocHeader*>(static_cast<char*>(base) + 64 - sizeof(AllocHeader));
    h->magic = ALLOC_MAGIC; h->pinned = pinned; h->base = base; h->pad = 0;
    {
        std::lock_guard<std::mutex> lk(g_alloc_mu);
        g_allocs[static_cast<char*>(base) + 64] = n_bytes;
    }
    return static_cast<char*>(base) + 64;
}

double* fftw_alloc_real(size_t n) { return static_cast<double*>(fftw_malloc(n * sizeof(double))); }
void* fftw_alloc_complex(size_t n) { return fftw_malloc(n * 2 * sizeof(double)); }

void fftw_free(void* p) {
    if (!p) return;
    AllocHeader* h = reinterpret_cast<AllocHeader*>(static_cast<char*>(p) - sizeof(AllocHeader));
    if (h->magic != ALLOC_MAGIC) {
        fprintf(stderr, "audiosync: fftw_free of a pointer not obtained from this library\n");
        return;
    }
    h->magic = 0;
    {
        std::lock_guard<std::mutex> lk(g_alloc_mu);
        g_allocs.erase(static_cast<char*>(p));
        g_alloc_gen.fetch_add(1);          // any resident session built on this block is stale
    }
    if (h->pinned) cudaFreeHost(h->base); else free(h->base);
}

}  // extern "C"
#pragma GCC visibility pop
