// Static row kernels with a run-time number of rows: the row stage of runtime-radix fp32 plans whose
// row length M2 is one the static kernels exist for (gen_plan.h: gen_static_rows).  The column
// stages of such a plan stay on the runtime-radix kernels (any M1, wrap / zero fill of embedded
// lengths); planes, row order and the four-step twiddle convention are the same in both families.
#include "plan_host.h"

namespace asc {

// PHAT plans run the PHAT twin of the row kernel, its split twiddle from the half-angle tables.
template <class RL, int NT>
struct StaticRows {
    using K = RowFusedKernel<RL, 0, NT>;
    using KP = RowFusedKernel<RL, 0, NT, true>;
    static int prepare(FftPlan* plan) {
        const GenShape& sh = plan->gen;
        std::vector<cplx> m_lo, m_hi;
        build_two_level(sh.M, sh.M - 1, m_lo, m_hi);
        if (upload(plan->row_tw, build_pass_tables(radix_vector<RL>())) != 0 ||
            upload(plan->row_rev, build_row_rev<RL>()) != 0 ||
            upload(plan->row_tab, build_row_tab<RL>(sh.M, sh.M1)) != 0 ||
            upload(plan->m_lo, m_lo) != 0 || upload(plan->m_hi, m_hi) != 0)
            return -1;
        if (!plan->phat) return prepare_kernel<K>(K::SMEM);
        std::vector<cplx> n_lo, n_hi;
        build_two_level(2 * sh.M, sh.M1 / 2, n_lo, n_hi);
        if (upload(plan->phat_rev, build_row_rev_half<RL>()) != 0 || upload(plan->phat_lo, n_lo) != 0 ||
            upload(plan->phat_hi, n_hi) != 0)
            return -1;
        return prepare_kernel<KP>(KP::SMEM);
    }
    template <class KK>
    static int launch_k(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, void* ws, int pairs, cudaStream_t st,
                        const DevBuf& rev, const DevBuf& lo, const DevBuf& hi) {
        const GenShape& sh = plan->gen;
        typename KK::Params p{static_cast<cplx*>(ws), static_cast<const cplx*>(plan->row_tw.p),
                              static_cast<const cplx*>(rev.p), static_cast<const cplx*>(lo.p),
                              static_cast<const cplx*>(hi.p), sh.M, static_cast<const cplx*>(plan->row_tab.p), sh.M1};
        const dim3 grid(sh.M1 / 2 + 1, 1, pairs);
        return launch(ctx, d, KC_ROW_FUSED, st, [&] {
            launch_stage(fft_kernel_entry<KK>, grid, dim3(KK::THREADS), KK::SMEM, st, p);
        });
    }
    static int launch_rows(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, void* ws, int pairs, cudaStream_t st) {
        return plan->phat ? launch_k<KP>(plan, ctx, d, ws, pairs, st, plan->phat_rev, plan->phat_lo, plan->phat_hi)
                          : launch_k<K>(plan, ctx, d, ws, pairs, st, plan->row_rev, plan->m_lo, plan->m_hi);
    }
};

// the row plans of the interval schedule (fft_plan.h)
template <class F>
static int for_static_rows(int M2, F&& f) {
    switch (M2) {
        case 480:  return f(StaticRows<Plan144k::Row, Plan144k::NT_ROW>{});
        case 960:  return f(StaticRows<Plan288k::Row, Plan288k::NT_ROW>{});
        case 1200: return f(StaticRows<Plan720k::Row, Plan720k::NT_ROW>{});
        case 2400: return f(StaticRows<Plan1440k::Row, Plan1440k::NT_ROW>{});
    }
    set_last_error("no static row kernel for M2 = %d", M2);
    return -1;
}

int static_rows_prepare(FftPlan* plan) {
    return for_static_rows(plan->gen.M2, [&](auto S) { return decltype(S)::prepare(plan); });
}

int static_rows_launch(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, void* ws, int pairs, cudaStream_t st) {
    return for_static_rows(plan->gen.M2, [&](auto S) { return decltype(S)::launch_rows(plan, ctx, d, ws, pairs, st); });
}

}  // namespace asc
