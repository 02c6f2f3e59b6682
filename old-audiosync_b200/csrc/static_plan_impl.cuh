// static_plan_impl.cuh -- launches and plan construction of the static four-step kernels; included
// by the per-length translation units (static_*.cu), which instantiate build_static_plan<P>.
#pragma once

#include "plan_host.h"

namespace asc {

template <class P>
static int run_static_wave(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d,
                           const void* src, const void* smp, int dtype, long long src_pitch,
                           long long smp_pitch, void* ws, PairPeak* peaks, int pairs, cudaStream_t st) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    constexpr int M1 = Col::n, M2 = Row::n;
    cplx* planes = static_cast<cplx*>(ws);
    const cplx* col_tw = static_cast<const cplx*>(plan->col_tw.p);
    const cplx* row_tw = static_cast<const cplx*>(plan->row_tw.p);
    const cplx* col_tc = static_cast<const cplx*>(plan->col_tc.p);
    const cplx* row_rev = static_cast<const cplx*>(plan->row_rev.p);
    const cplx* row_tab = static_cast<const cplx*>(plan->row_tab.p);
    const cplx* m_lo = static_cast<const cplx*>(plan->m_lo.p);
    const cplx* m_hi = static_cast<const cplx*>(plan->m_hi.p);
    // K_C always stages its tiles through the TMA unit: its map is encoded before anything is
    // enqueued, so that a failure leaves no partial wave behind
    using KC = ColInvKernel<Col, Row::n, P::NT_COL>;
    typename KC::Params pc{planes, peaks, col_tw, P::L};
    if (make_tile_map(&pc.tm, planes, M2, M1, (size_t)P::L * sizeof(cplx), (size_t)2 * pairs,
                      tile_box_rows(KC::TMA_ROWS)) != 0) {
        set_last_error("L = %lld: cuTensorMapEncodeTiled %s for the workspace planes", P::L,
                       tensor_map_encoder() ? "failed" : "is not exported by the driver");
        return -1;
    }
    const dim3 grid_a(M2 / COL_T, 2, pairs);
    auto col_fwd = [&](auto KK, const typename decltype(KK)::Params& p) -> int {
        using K = decltype(KK);
        return launch(ctx, d, KC_COL_FWD, st, [&] {
            launch_stage(fft_kernel_entry<K>, grid_a, dim3(K::THREADS), K::SMEM, st, p);
        });
    };
    // register path: one load per packed point where every pair's base is aligned to two elements
    // (a view at an odd element offset, e.g. x[1:], is not: two element loads then)
    auto vec_ok = [](const void* p, long long pitch, size_t esz) -> int {
        return reinterpret_cast<uintptr_t>(p) % (2 * esz) == 0 && pitch % 2 == 0;
    };
    if (dtype == AUDIOSYNC_CUDA_F32) {
        // TMA boxes need 16-byte aligned rows: every pair / row offset is a multiple of 16 bytes,
        // so only the base pointers decide.  Other fp32 inputs load through registers.
        const bool aligned = ((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(smp)) & 15u) == 0 &&
                             src_pitch % 4 == 0 && smp_pitch % 4 == 0;
        const float* s_in = static_cast<const float*>(src);
        const float* m_in = static_cast<const float*>(smp);
        using KT = ColFwdKernel<Col, Row::n, P::NT_COL, float, true>;
        using KR = ColFwdKernel<Col, Row::n, P::NT_COL, float, false>;
        typename KT::Params pt{s_in, m_in, planes, peaks, col_tw, col_tc, m_lo, m_hi, P::L, src_pitch, smp_pitch};
        const bool tma = aligned &&
                         make_tile_map(&pt.tm_src, s_in, M2, M1, (size_t)src_pitch * sizeof(float), (size_t)pairs,
                                       tile_box_rows(KT::SRC_ROWS)) == 0 &&
                         make_tile_map(&pt.tm_smp, m_in, M2, M1 / 2, (size_t)smp_pitch * sizeof(float), (size_t)pairs,
                                       tile_box_rows(KT::SMP_ROWS)) == 0;
        if ((tma ? col_fwd(KT{}, pt)
                 : col_fwd(KR{}, {s_in, m_in, planes, peaks, col_tw, col_tc, m_lo, m_hi, P::L, src_pitch, smp_pitch,
                                  vec_ok(src, src_pitch, sizeof(float)), vec_ok(smp, smp_pitch, sizeof(float))})) != 0)
            return -1;
    } else if (dtype == AUDIOSYNC_CUDA_F64) {
        using K = ColFwdKernel<Col, Row::n, P::NT_COL, double, false>;
        if (col_fwd(K{}, {static_cast<const double*>(src), static_cast<const double*>(smp), planes, peaks, col_tw,
                          col_tc, m_lo, m_hi, P::L, src_pitch, smp_pitch, vec_ok(src, src_pitch, sizeof(double)),
                          vec_ok(smp, smp_pitch, sizeof(double))}) != 0) return -1;
    } else if (dtype == AUDIOSYNC_CUDA_S16) {
        const int vec_src = vec_ok(src, src_pitch, sizeof(int16_t));
        const int vec_smp = vec_ok(smp, smp_pitch, sizeof(int16_t));
        using K = ColFwdKernel<Col, Row::n, P::NT_COL, int16_t, false>;
        if (col_fwd(K{}, {static_cast<const int16_t*>(src), static_cast<const int16_t*>(smp), planes, peaks, col_tw,
                          col_tc, m_lo, m_hi, P::L, src_pitch, smp_pitch, vec_src, vec_smp}) != 0) return -1;
    } else {
        set_last_error("bad dtype %d", dtype);
        return -1;
    }
    {
        auto rows = [&](auto KK, const cplx* rev, const cplx* lo, const cplx* hi) -> int {
            using K = decltype(KK);
            typename K::Params p{planes, row_tw, rev, lo, hi, P::L, row_tab};
            const dim3 grid(M1 / 2 + 1, 1, pairs);
            return launch(ctx, d, KC_ROW_FUSED, st, [&] {
                launch_stage(fft_kernel_entry<K>, grid, dim3(K::THREADS), K::SMEM, st, p);
            });
        };
        if ((plan->phat ? rows(RowFusedKernel<Row, Col::n, P::NT_ROW, true>{}, static_cast<const cplx*>(plan->phat_rev.p),
                               static_cast<const cplx*>(plan->phat_lo.p), static_cast<const cplx*>(plan->phat_hi.p))
                        : rows(RowFusedKernel<Row, Col::n, P::NT_ROW>{}, row_rev, m_lo, m_hi)) != 0)
            return -1;
    }
    {
        const dim3 grid(pairs, M2 / COL_T, 1);
        if (launch(ctx, d, KC_COL_INV, st, [&] {
                launch_stage(fft_kernel_entry<KC>, grid, dim3(KC::THREADS), KC::SMEM, st, pc);
            }) != 0) return -1;
    }
    return 0;
}


template <class P>
int build_static_plan(FftPlan* plan) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    plan->kind = PATH_STATIC_FFT;
    plan->L = P::L;
    plan->M1 = Col::n;
    plan->M2 = Row::n;
    plan->ws_bytes_per_pair = (size_t)2 * P::L * sizeof(cplx);
    std::string d = "fft L=" + std::to_string(P::L) + " M1=" + std::to_string(Col::n) +
                    " M2=" + std::to_string(Row::n) + " col=";
    for (int i = 0; i < Col::count; i++) d += (i ? "x" : "") + std::to_string(Col::r(i));
    d += " row=";
    for (int i = 0; i < Row::count; i++) d += (i ? "x" : "") + std::to_string(Row::r(i));
    d += " static four-step fp32";
    plan->desc = d;
    std::vector<cplx> m_lo, m_hi;
    build_two_level(P::L, P::L - 1, m_lo, m_hi);
    if (upload(plan->col_tw, build_pass_tables(radix_vector<Col>())) != 0 ||
        upload(plan->row_tw, build_pass_tables(radix_vector<Row>())) != 0 ||
        upload(plan->col_tc, build_col_tc(P::L, Col::weight(Col::count - 1))) != 0 ||
        upload(plan->row_rev, build_row_rev<Row>()) != 0 ||
        upload(plan->row_tab, build_row_tab<Row>(P::L, Col::n)) != 0 ||
        upload(plan->m_lo, m_lo) != 0 || upload(plan->m_hi, m_hi) != 0)
        return -1;
    if (plan->phat) {
        std::vector<cplx> n_lo, n_hi;
        build_two_level(2 * P::L, Col::n / 2, n_lo, n_hi);
        if (upload(plan->phat_rev, build_row_rev_half<Row>()) != 0 || upload(plan->phat_lo, n_lo) != 0 ||
            upload(plan->phat_hi, n_hi) != 0)
            return -1;
    }
    using KT = ColFwdKernel<Col, Row::n, P::NT_COL, float, true>;
    using KR = ColFwdKernel<Col, Row::n, P::NT_COL, float, false>;
    using KD = ColFwdKernel<Col, Row::n, P::NT_COL, double, false>;
    using KS = ColFwdKernel<Col, Row::n, P::NT_COL, int16_t, false>;
    using KB = RowFusedKernel<Row, Col::n, P::NT_ROW>;
    using KBP = RowFusedKernel<Row, Col::n, P::NT_ROW, true>;
    using KC = ColInvKernel<Col, Row::n, P::NT_COL>;
    if (prepare_kernel<KT>(KT::SMEM) != 0 || prepare_kernel<KR>(KR::SMEM) != 0 || prepare_kernel<KD>(KD::SMEM) != 0 ||
        prepare_kernel<KS>(KS::SMEM) != 0 ||
        (plan->phat ? prepare_kernel<KBP>(KBP::SMEM) : prepare_kernel<KB>(KB::SMEM)) != 0 || prepare_kernel<KC>(KC::SMEM) != 0)
        return -1;
    plan->run_wave = [plan](audiosync_cuda_ctx* ctx, DeviceState& d, const void* src, const void* smp,
                            int dtype, long long sp, long long mp, void* ws, PairPeak* peaks, int pairs,
                            cudaStream_t st) {
        return run_static_wave<P>(plan, ctx, d, src, smp, dtype, sp, mp, ws, peaks, pairs, st);
    };
    return 0;
}


}  // namespace asc
