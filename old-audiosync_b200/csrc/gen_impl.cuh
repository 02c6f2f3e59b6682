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

// the windowed, exporting and runner-up twins of the fp32 inverse column kernel (fp64 plans window in
// argmax_f64_window_kernel, export in corr_gather_kernel and search runner-ups in argmax_f64_runner_up_kernel)
template <typename T, int CT, int NT>
static int prepare_col_inv_window(const GenShape& sh) {
    if constexpr (sizeof(T) == 4)
        return prepare_gen_kernel<GenColInvKernel<T, CT, NT, true>>(GenColInvKernel<T, CT, NT, true>::smem_bytes(sh)) != 0 ||
               prepare_gen_kernel<GenColInvKernel<T, CT, NT, true, true>>(GenColInvKernel<T, CT, NT, true, true>::smem_bytes(sh)) != 0 ||
               prepare_gen_kernel<GenColInvKernel<T, CT, NT, true, false, true>>(
                   GenColInvKernel<T, CT, NT, true, false, true>::smem_bytes(sh)) != 0
                   ? -1 : 0;
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
int GenStage<T, NT>::col_fwd(FftPlan* plan, const Wave& w) {
    typedef typename GenTraits<T>::C C;
    const GenShape& sh = plan->gen;
    return with_input_type(w.dtype, [&](auto IN) -> int {
        using InT = decltype(IN);
        return gen_for_tile_width<T>(sh.ct, [&](auto CTC) -> int {
            using K = GenColFwdKernel<T, InT, decltype(CTC)::value, NT>;
            typename K::Params p{static_cast<const InT*>(w.src), static_cast<const InT*>(w.smp), static_cast<C*>(w.ws), w.peaks,
                                 static_cast<const C*>(plan->g_wcol.p), static_cast<const C*>(plan->g_lo.p),
                                 static_cast<const C*>(plan->g_hi.p), static_cast<const int*>(plan->g_p2f_col.p),
                                 sh, w.src_pitch, w.smp_pitch, vec_loads<InT>(w.src, w.src_pitch),
                                 vec_loads<InT>(w.smp, w.smp_pitch)};
            const dim3 grid((sh.M2 + K::CT - 1) / K::CT, 2, w.pairs);
            return launch(w.ctx, w.d, KC_COL_FWD, w.st, [&] {
                launch_stage(gen_kernel_entry<K>, grid, dim3(K::THREADS), K::smem_bytes(sh), w.st, p);
            });
        });
    });
}

template <typename T, int NT>
int GenStage<T, NT>::rows(FftPlan* plan, const Wave& w) {
    typedef typename GenTraits<T>::C C;
    const GenShape& sh = plan->gen;
    return with_bool(plan->phat, [&](auto PHAT) -> int {
        using K = GenRowFusedKernel<T, NT, decltype(PHAT)::value>;
        typename K::Params p{static_cast<C*>(w.ws), static_cast<const C*>(plan->g_wrow.p), static_cast<const C*>(plan->g_wpos.p),
                             static_cast<const C*>(plan->g_lo.p), static_cast<const C*>(plan->g_hi.p),
                             static_cast<const int*>(plan->g_f2p_row.p), sh, static_cast<const C*>(plan->phat_rev.p),
                             static_cast<const C*>(plan->phat_lo.p), static_cast<const C*>(plan->phat_hi.p)};
        const dim3 grid(sh.M1 / 2 + 1, 1, w.pairs);
        return launch(w.ctx, w.d, KC_ROW_FUSED, w.st, [&] {
            launch_stage(gen_kernel_entry<K>, grid, dim3(K::THREADS), K::smem_bytes(sh), w.st, p);
        });
    });
}

template <typename T, int NT>
int GenStage<T, NT>::col_inv(FftPlan* plan, const Wave& w) {
    typedef typename GenTraits<T>::C C;
    const GenShape& sh = plan->gen;
    C* planes = static_cast<C*>(w.ws);
    const int rc = gen_for_tile_width<T>(sh.ct, [&](auto CTC) -> int {
        auto go = [&](auto KK, auto fill) -> int {
            using K = decltype(KK);
            typename K::Params p{planes, w.peaks, static_cast<const C*>(plan->g_wcol.p), static_cast<const int*>(plan->g_p2f_col.p),
                                 sh, reinterpret_cast<T*>(planes)};
            fill(p);
            const dim3 grid(w.pairs, (sh.M2 + K::CT - 1) / K::CT, 1);
            return launch(w.ctx, w.d, KC_COL_INV, w.st, [&] {
                launch_stage(gen_kernel_entry<K>, grid, dim3(K::THREADS), K::smem_bytes(sh), w.st, p);
            });
        };
        constexpr int CT = decltype(CTC)::value;
        if constexpr (sizeof(T) == 4) {
            // the exporting twin runs the windowed argmax, over all of [0, 2L) when no window is set
            if (w.corr)
                return go(GenColInvKernel<T, CT, NT, true, true>{}, [&](auto& p) {
                    p.win = w.win ? *w.win : full_window(sh.L);
                    p.corr = *w.corr;
                });
            if (w.win) return go(GenColInvKernel<T, CT, NT, true>{}, [&](auto& p) { p.win = *w.win; });
        }
        return go(GenColInvKernel<T, CT, NT>{}, [](auto&) {});
    });
    if (rc != 0) return -1;
    if constexpr (sizeof(T) == 8) {
        // fp64: r[0 .. 2L) of pair i sits in its (dead) sample plane; full double keys
        const double* r = reinterpret_cast<const double*>(planes) + 2 * sh.M;
        if (launch(w.ctx, w.d, KC_ARGMAX_F64, w.st, [&] {
                if (w.win) argmax_f64_window_kernel<<<w.pairs, 1024, 0, w.st>>>(r, 2 * sh.L, 4 * sh.M, w.peaks, *w.win);
                else argmax_f64_kernel<<<w.pairs, 1024, 0, w.st>>>(r, 2 * sh.L, 4 * sh.M, w.peaks);
            }) != 0)
            return -1;
        if (w.corr) return launch_corr_gather(w, r, 4 * sh.M);
    }
    return 0;
}

// The runner-up search of a wave into w.peaks.  fp32: the inverse column kernel's runner-up twin over
// plane 0, which G_C only reads (the rows' static or runtime-radix kernel wrote it, and nothing since);
// fp64: over r in the pairs' sample planes, which nothing writes after G_C.
template <typename T, int NT>
int GenStage<T, NT>::runner_up(FftPlan* plan, const Wave& w) {
    typedef typename GenTraits<T>::C C;
    const GenShape& sh = plan->gen;
    C* planes = static_cast<C*>(w.ws);
    if constexpr (sizeof(T) == 8) {
        const double* r = reinterpret_cast<const double*>(planes) + 2 * sh.M;
        return launch(w.ctx, w.d, KC_RU_ARGMAX, w.st, [&] {
            argmax_f64_runner_up_kernel<<<w.pairs, 1024, 0, w.st>>>(r, 4 * sh.M, w.peaks, *w.ru);
        });
    } else {
        return gen_for_tile_width<T>(sh.ct, [&](auto CTC) -> int {
            using K = GenColInvKernel<T, decltype(CTC)::value, NT, true, false, true>;
            typename K::Params p{};
            static_cast<typename K::PlainParams&>(p) = {planes, w.peaks, static_cast<const C*>(plan->g_wcol.p),
                                                        static_cast<const int*>(plan->g_p2f_col.p), sh, reinterpret_cast<T*>(planes),
                                                        w.win ? *w.win : full_window(sh.L)};
            p.ru = *w.ru;
            const dim3 grid(w.pairs, (sh.M2 + K::CT - 1) / K::CT, 1);
            return launch(w.ctx, w.d, KC_RU_ARGMAX, w.st, [&] {
                launch_stage(gen_kernel_entry<K>, grid, dim3(K::THREADS), K::smem_bytes(sh), w.st, p);
            });
        });
    }
}

}  // namespace asc
