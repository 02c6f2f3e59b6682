// gen_impl.cuh -- launchers of the runtime-radix kernels, one set per (arithmetic type, CTA size);
// included by gen_f32_*.cu / gen_f64_*.cu, which instantiate GenStage<T, NT> (declared in plan_host.h).
#pragma once

#include "plan_host.h"
#include "reduce_kernels.cuh"

namespace asc {

// The runtime-radix kernels serve plans of many shapes: each is allowed the device's whole opt-in
// shared memory (a per-plan limit would be lowered again by the next, smaller plan of the same kernel).
template <class K>
static int prepare_gen_kernel(size_t smem) {
    int dev = 0, optin = 0;
    ASC_CUDA_OK(cudaGetDevice(&dev));
    ASC_CUDA_OK(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    if (smem > (size_t)optin) {
        set_last_error("plan needs %zu bytes of shared memory per CTA, the device allows %d", smem, optin);
        return -1;
    }
    ASC_CUDA_OK(cudaFuncSetAttribute(gen_kernel_entry<K>, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
    return 0;
}

// the windowed twin of the fp32 inverse column kernel (fp64 plans window in argmax_f64_window_kernel)
template <typename T, int CT, int NT>
static int prepare_col_inv_window(const GenShape& sh) {
    if constexpr (sizeof(T) == 4) return prepare_gen_kernel<GenColInvKernel<T, CT, NT, true>>(GenColInvKernel<T, CT, NT, true>::smem_bytes(sh));
    return 0;
}

// fp32 arithmetic has 16- and 8-column tiles, fp64 only 8
template <typename T, class F>
static int gen_for_tile_width(int ct, F&& f) {
    if constexpr (sizeof(T) == 4) {
        if (ct == 16) return f(IC<16>{});
    }
    return f(IC<8>{});
}

template <typename T, int NT>
int GenStage<T, NT>::prepare_cols(const GenShape& sh) {
    return gen_for_tile_width<T>(sh.ct, [&](auto CTC) -> int {
        constexpr int CT = decltype(CTC)::value;
        return prepare_gen_kernel<GenColFwdKernel<T, float, CT, NT>>(GenColFwdKernel<T, float, CT, NT>::smem_bytes(sh)) != 0 ||
               prepare_gen_kernel<GenColFwdKernel<T, double, CT, NT>>(GenColFwdKernel<T, double, CT, NT>::smem_bytes(sh)) != 0 ||
               prepare_gen_kernel<GenColFwdKernel<T, int16_t, CT, NT>>(GenColFwdKernel<T, int16_t, CT, NT>::smem_bytes(sh)) != 0 ||
               prepare_gen_kernel<GenColInvKernel<T, CT, NT>>(GenColInvKernel<T, CT, NT>::smem_bytes(sh)) != 0 ||
               prepare_col_inv_window<T, CT, NT>(sh) != 0 ? -1 : 0;
    });
}

template <typename T, int NT>
int GenStage<T, NT>::prepare_rows(const GenShape& sh, bool phat) {
    return phat ? prepare_gen_kernel<GenRowFusedKernel<T, NT, true>>(GenRowFusedKernel<T, NT, true>::smem_bytes(sh))
                : prepare_gen_kernel<GenRowFusedKernel<T, NT>>(GenRowFusedKernel<T, NT>::smem_bytes(sh));
}

template <typename T, int NT>
int GenStage<T, NT>::col_fwd(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, const void* src, const void* smp,
                             int dtype, long long sp, long long mp, void* ws, PairPeak* peaks, int pairs, cudaStream_t st) {
    typedef typename GenTraits<T>::C C;
    const GenShape& sh = plan->gen;
    auto go = [&](auto IN) -> int {
        using InT = decltype(IN);
        return gen_for_tile_width<T>(sh.ct, [&](auto CTC) -> int {
            using K = GenColFwdKernel<T, InT, decltype(CTC)::value, NT>;
            // two elements per load where the pairs' bases allow it
            const size_t al = 2 * sizeof(InT);
            const int vec_src = reinterpret_cast<uintptr_t>(src) % al == 0 && sp % 2 == 0;
            const int vec_smp = reinterpret_cast<uintptr_t>(smp) % al == 0 && mp % 2 == 0;
            typename K::Params p{static_cast<const InT*>(src), static_cast<const InT*>(smp), static_cast<C*>(ws), peaks,
                                 static_cast<const C*>(plan->g_wcol.p), static_cast<const C*>(plan->g_lo.p),
                                 static_cast<const C*>(plan->g_hi.p), static_cast<const int*>(plan->g_p2f_col.p),
                                 sh, sp, mp, vec_src, vec_smp};
            const dim3 grid((sh.M2 + K::CT - 1) / K::CT, 2, pairs);
            return launch(ctx, d, KC_COL_FWD, st, [&] {
                launch_stage(gen_kernel_entry<K>, grid, dim3(K::THREADS), K::smem_bytes(sh), st, p);
            });
        });
    };
    switch (dtype) {
        case AUDIOSYNC_CUDA_F32: return go(float{});
        case AUDIOSYNC_CUDA_F64: return go(double{});
        case AUDIOSYNC_CUDA_S16: return go(int16_t{});
    }
    set_last_error("bad dtype %d", dtype);
    return -1;
}

template <typename T, int NT>
int GenStage<T, NT>::rows(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, void* ws, int pairs, cudaStream_t st) {
    typedef typename GenTraits<T>::C C;
    const GenShape& sh = plan->gen;
    auto go = [&](auto KK) -> int {
        using K = decltype(KK);
        typename K::Params p{static_cast<C*>(ws), static_cast<const C*>(plan->g_wrow.p), static_cast<const C*>(plan->g_wpos.p),
                             static_cast<const C*>(plan->g_lo.p), static_cast<const C*>(plan->g_hi.p),
                             static_cast<const int*>(plan->g_f2p_row.p), sh, static_cast<const C*>(plan->phat_rev.p),
                             static_cast<const C*>(plan->phat_lo.p), static_cast<const C*>(plan->phat_hi.p)};
        const dim3 grid(sh.M1 / 2 + 1, 1, pairs);
        return launch(ctx, d, KC_ROW_FUSED, st, [&] {
            launch_stage(gen_kernel_entry<K>, grid, dim3(K::THREADS), K::smem_bytes(sh), st, p);
        });
    };
    return plan->phat ? go(GenRowFusedKernel<T, NT, true>{}) : go(GenRowFusedKernel<T, NT>{});
}

template <typename T, int NT>
int GenStage<T, NT>::col_inv(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, void* ws, PairPeak* peaks, int pairs,
                             cudaStream_t st, const RawWindow* win) {
    typedef typename GenTraits<T>::C C;
    const GenShape& sh = plan->gen;
    C* planes = static_cast<C*>(ws);
    const int rc = gen_for_tile_width<T>(sh.ct, [&](auto CTC) -> int {
        auto go = [&](auto KK, auto fill) -> int {
            using K = decltype(KK);
            typename K::Params p{planes, peaks, static_cast<const C*>(plan->g_wcol.p), static_cast<const int*>(plan->g_p2f_col.p),
                                 sh, reinterpret_cast<T*>(planes)};
            fill(p);
            const dim3 grid(pairs, (sh.M2 + K::CT - 1) / K::CT, 1);
            return launch(ctx, d, KC_COL_INV, st, [&] {
                launch_stage(gen_kernel_entry<K>, grid, dim3(K::THREADS), K::smem_bytes(sh), st, p);
            });
        };
        constexpr int CT = decltype(CTC)::value;
        if constexpr (sizeof(T) == 4) {
            if (win) return go(GenColInvKernel<T, CT, NT, true>{}, [&](auto& p) { p.win = *win; });
        }
        return go(GenColInvKernel<T, CT, NT>{}, [](auto&) {});
    });
    if (rc != 0) return -1;
    if constexpr (sizeof(T) == 8) {
        // fp64: r[0 .. 2L) of pair i sits in its (dead) sample plane; full double keys
        const double* r = reinterpret_cast<const double*>(planes) + 2 * sh.M;
        return launch(ctx, d, KC_ARGMAX_F64, st, [&] {
            if (win) argmax_f64_window_kernel<<<pairs, 1024, 0, st>>>(r, 2 * sh.L, 4 * sh.M, peaks, *win);
            else argmax_f64_kernel<<<pairs, 1024, 0, st>>>(r, 2 * sh.L, 4 * sh.M, peaks);
        });
    }
    return 0;
}

}  // namespace asc
