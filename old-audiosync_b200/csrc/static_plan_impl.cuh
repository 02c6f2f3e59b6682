// static_plan_impl.cuh -- launches and plan construction of the static four-step kernels; included
// by the per-length translation units (static_*.cu), which instantiate build_static_plan<P>.
#pragma once

#include "plan_host.h"

namespace asc {

// K_A over the wave's pairs.  SMP_ONLY: the sample planes alone (a shared-source wave); otherwise
// `signals` = 2 (source and sample) or 1 (the source alone: one pair whose plane 0 is a shared
// source's column pass).
template <class P, bool SMP_ONLY>
static int static_col_fwd(FftPlan* plan, const Wave& w, int signals) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    constexpr int M1 = Col::n, M2 = Row::n;
    cplx* planes = static_cast<cplx*>(w.ws);
    const cplx* col_tw = static_cast<const cplx*>(plan->col_tw.p);
    const cplx* col_tc = static_cast<const cplx*>(plan->col_tc.p);
    const cplx* m_lo = static_cast<const cplx*>(plan->m_lo.p);
    const cplx* m_hi = static_cast<const cplx*>(plan->m_hi.p);
    const dim3 grid_a(M2 / COL_T, SMP_ONLY ? 1 : signals, w.pairs);
    auto col_fwd = [&](auto KK, const typename decltype(KK)::Params& p) -> int {
        using K = decltype(KK);
        return launch(w.ctx, w.d, KC_COL_FWD, w.st, [&] {
            launch_stage(fft_kernel_entry<K>, grid_a, dim3(K::THREADS), K::SMEM, w.st, p);
        });
    };
    return with_input_type(w.dtype, [&](auto IN) -> int {
        using InT = decltype(IN);
        const InT* s_in = static_cast<const InT*>(w.src);
        const InT* m_in = static_cast<const InT*>(w.smp);
        if constexpr (std::is_same<InT, float>::value) {
            // TMA boxes need 16-byte aligned rows: every pair / row offset is a multiple of 16 bytes,
            // so only the base pointers decide.  Other fp32 inputs load through registers.
            const bool src_aligned = SMP_ONLY || ((reinterpret_cast<uintptr_t>(w.src) & 15u) == 0 && w.src_pitch % 4 == 0);
            const bool aligned = src_aligned && (reinterpret_cast<uintptr_t>(w.smp) & 15u) == 0 && w.smp_pitch % 4 == 0;
            using KT = ColFwdKernel<Col, Row::n, P::NT_COL, float, true, SMP_ONLY>;
            typename KT::Params pt{s_in, m_in, planes, w.peaks, col_tw, col_tc, m_lo, m_hi, P::L, w.src_pitch, w.smp_pitch};
            const bool tma = aligned &&
                             (SMP_ONLY || make_tile_map(&pt.tm_src, s_in, M2, M1, (size_t)w.src_pitch * sizeof(float),
                                                        (size_t)w.pairs, tile_box_rows(KT::SRC_ROWS)) == 0) &&
                             make_tile_map(&pt.tm_smp, m_in, M2, M1 / 2, (size_t)w.smp_pitch * sizeof(float), (size_t)w.pairs,
                                           tile_box_rows(KT::SMP_ROWS)) == 0;
            if (tma) return col_fwd(KT{}, pt);
        }
        using K = ColFwdKernel<Col, Row::n, P::NT_COL, InT, false, SMP_ONLY>;
        return col_fwd(K{}, {s_in, m_in, planes, w.peaks, col_tw, col_tc, m_lo, m_hi, P::L, w.src_pitch, w.smp_pitch,
                             vec_loads<InT>(w.src, w.src_pitch), vec_loads<InT>(w.smp, w.smp_pitch)});
    });
}

// K_C's parameters, its tile map encoded: -1 (message set) when the driver cannot encode it.  Encoded
// before a wave's first launch, so that a failure leaves no partial wave behind.
template <class P>
static int static_col_inv_params(FftPlan* plan, const Wave& w, typename ColInvKernel<typename P::Col, P::Row::n, P::NT_COL>::Params* pc) {
    using Col = typename P::Col;
    constexpr int M1 = Col::n, M2 = P::Row::n;
    cplx* planes = static_cast<cplx*>(w.ws);
    *pc = {planes, w.peaks, static_cast<const cplx*>(plan->col_tw.p), P::L};
    if (make_tile_map(&pc->tm, planes, M2, M1, (size_t)P::L * sizeof(cplx), (size_t)2 * w.pairs,
                      tile_box_rows(ColInvKernel<Col, M2, P::NT_COL>::TMA_ROWS)) != 0) {
        set_last_error("L = %lld: cuTensorMapEncodeTiled %s for the workspace planes", P::L,
                       tensor_map_encoder() ? "failed" : "is not exported by the driver");
        return -1;
    }
    return 0;
}

// K_B of one wave in row mode MODE: ROWS_PAIR, ROWS_SHARED_SRC or ROWS_BOTH_SPECTRA (w.spec: the
// source's forward rows for the last two)
template <class P, int MODE>
static int static_rows(FftPlan* plan, const Wave& w) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    cplx* planes = static_cast<cplx*>(w.ws);
    const cplx* row_tw = static_cast<const cplx*>(plan->row_tw.p);
    const cplx* row_tab = static_cast<const cplx*>(plan->row_tab.p);
    auto rows = [&](auto KK, const cplx* rev, const cplx* lo, const cplx* hi) -> int {
        using K = decltype(KK);
        const typename K::PairParams base{planes, row_tw, rev, lo, hi, P::L, row_tab};
        typename K::Params p;
        if constexpr (MODE == ROWS_BOTH_SPECTRA) p = {{base, static_cast<const cplx*>(w.spec)}, w.peaks};
        else if constexpr (MODE == ROWS_SHARED_SRC) p = {base, static_cast<const cplx*>(w.spec)};
        else p = base;
        const dim3 grid(Col::n / 2 + 1, 1, w.pairs);
        return launch(w.ctx, w.d, KC_ROW_FUSED, w.st, [&] {
            launch_stage(fft_kernel_entry<K>, grid, dim3(K::THREADS), K::SMEM, w.st, p);
        });
    };
    return plan->phat ? rows(RowFusedKernel<Row, Col::n, P::NT_ROW, true, MODE>{}, static_cast<const cplx*>(plan->phat_rev.p),
                             static_cast<const cplx*>(plan->phat_lo.p), static_cast<const cplx*>(plan->phat_hi.p))
                      : rows(RowFusedKernel<Row, Col::n, P::NT_ROW, false, MODE>{}, static_cast<const cplx*>(plan->row_rev.p),
                             static_cast<const cplx*>(plan->m_lo.p), static_cast<const cplx*>(plan->m_hi.p));
}

// K_C of one wave: plain, windowed or exporting
template <class P>
static int static_col_inv(const Wave& w, const typename ColInvKernel<typename P::Col, P::Row::n, P::NT_COL>::Params& pc) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    using KC = ColInvKernel<Col, Row::n, P::NT_COL>;
    const dim3 grid(w.pairs, Row::n / COL_T, 1);
    if (w.corr) {
        // the exporting twin runs the windowed argmax, over all of [0, 2L) when no window is set
        using KCO = ColInvKernel<Col, Row::n, P::NT_COL, true, true, true>;
    using KCR = ColInvKernel<Col, Row::n, P::NT_COL, true, true, false, true>;
        typename KCO::Params po{{pc.planes, pc.peaks, pc.tw, P::L, w.win ? *w.win : full_window(P::L), pc.tm}, *w.corr};
        return launch(w.ctx, w.d, KC_COL_INV, w.st, [&] {
            launch_stage(fft_kernel_entry<KCO>, grid, dim3(KCO::THREADS), KCO::SMEM, w.st, po);
        });
    }
    if (w.win) {
        using KCW = ColInvKernel<Col, Row::n, P::NT_COL, true, true>;
        typename KCW::Params pw{pc.planes, pc.peaks, pc.tw, P::L, *w.win, pc.tm};
        return launch(w.ctx, w.d, KC_COL_INV, w.st, [&] {
            launch_stage(fft_kernel_entry<KCW>, grid, dim3(KCW::THREADS), KCW::SMEM, w.st, pw);
        });
    }
    return launch(w.ctx, w.d, KC_COL_INV, w.st, [&] {
        launch_stage(fft_kernel_entry<KC>, grid, dim3(KC::THREADS), KC::SMEM, w.st, pc);
    });
}

// The runner-up search of a wave: K_C's runner-up twin over the planes run_static_wave left (K_C only
// reads them), into w.peaks.
template <class P>
static int static_runner_up(FftPlan* plan, const Wave& w) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    typename ColInvKernel<Col, Row::n, P::NT_COL>::Params pc;
    if (static_col_inv_params<P>(plan, w, &pc) != 0) return -1;
    using KCR = ColInvKernel<Col, Row::n, P::NT_COL, true, true, false, true>;
    typename KCR::Params pr{{pc.planes, pc.peaks, pc.tw, P::L, w.win ? *w.win : full_window(P::L), pc.tm}, *w.ru};
    const dim3 grid(w.pairs, Row::n / COL_T, 1);
    return launch(w.ctx, w.d, KC_RU_ARGMAX, w.st, [&] {
        launch_stage(fft_kernel_entry<KCR>, grid, dim3(KCR::THREADS), KCR::SMEM, w.st, pr);
    });
}

// One wave.  SHARED: the pairs share one source whose forward rows source_spectrum left in w.spec
// (the source itself is not read): K_A on the samples, the shared-source K_B, K_C.
template <class P, bool SHARED>
static int run_static_wave(FftPlan* plan, const Wave& w) {
    typename ColInvKernel<typename P::Col, P::Row::n, P::NT_COL>::Params pc;
    if (static_col_inv_params<P>(plan, w, &pc) != 0) return -1;
    if (static_col_fwd<P, SHARED>(plan, w, 2) != 0) return -1;
    if (static_rows<P, SHARED ? ROWS_SHARED_SRC : ROWS_PAIR>(plan, w) != 0) return -1;
    return static_col_inv<P>(w, pc);
}

// The sample side of a cross wave (sources against samples): K_A on the samples alone, then their
// forward rows in place in plane 1 -- the source-spectrum kernel launched on the planes one plane
// further on, so that its plane 0 of pair i is pair i's plane 1 (the pair pitch stays 2M).
template <class P>
static int static_cross_samples(FftPlan* plan, const Wave& w) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    if (static_col_fwd<P, true>(plan, w, 2) != 0) return -1;
    using K = RowFusedKernel<Row, Col::n, P::NT_ROW, false, ROWS_SRC_SPECTRUM>;
    typename K::Params p{static_cast<cplx*>(w.ws) + P::L, static_cast<const cplx*>(plan->row_tw.p),
                         static_cast<const cplx*>(plan->row_rev.p), static_cast<const cplx*>(plan->m_lo.p),
                         static_cast<const cplx*>(plan->m_hi.p), P::L, static_cast<const cplx*>(plan->row_tab.p)};
    return launch(w.ctx, w.d, KC_SMP_SPECTRUM, w.st, [&] {
        launch_stage(fft_kernel_entry<K>, dim3(Col::n / 2 + 1, 1, w.pairs), dim3(K::THREADS), K::SMEM, w.st, p);
    });
}

// One source (w.spec: its forward rows) against a wave whose samples static_cross_samples transformed:
// K_B from both spectra, which also clears the peak records, then K_C.  Plane 1 is left as it was.
template <class P>
static int static_cross_rows(FftPlan* plan, const Wave& w) {
    typename ColInvKernel<typename P::Col, P::Row::n, P::NT_COL>::Params pc;
    if (static_col_inv_params<P>(plan, w, &pc) != 0) return -1;
    if (static_rows<P, ROWS_BOTH_SPECTRA>(plan, w) != 0) return -1;
    return static_col_inv<P>(w, pc);
}

// The shared source's forward rows, once per call: K_A on the source alone as one pair (plane 0 of
// that pair is `spec`), then the forward passes of its rows in place.
template <class P>
static int static_source_spectrum(FftPlan* plan, const Wave& w, cplx* spec) {
    using Col = typename P::Col;
    using Row = typename P::Row;
    const Wave src_pair{w.ctx, w.d, w.st, w.src, w.src, w.dtype, 2 * P::L, 2 * P::L, false, nullptr, spec, w.peaks, 1, nullptr, nullptr};
    if (static_col_fwd<P, false>(plan, src_pair, 1) != 0) return -1;
    using K = RowFusedKernel<Row, Col::n, P::NT_ROW, false, ROWS_SRC_SPECTRUM>;
    typename K::Params p{spec, static_cast<const cplx*>(plan->row_tw.p), static_cast<const cplx*>(plan->row_rev.p),
                         static_cast<const cplx*>(plan->m_lo.p), static_cast<const cplx*>(plan->m_hi.p), P::L,
                         static_cast<const cplx*>(plan->row_tab.p)};
    return launch(w.ctx, w.d, KC_SRC_SPECTRUM, w.st, [&] {
        launch_stage(fft_kernel_entry<K>, dim3(Col::n / 2 + 1, 1, 1), dim3(K::THREADS), K::SMEM, w.st, p);
    });
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
    using KCW = ColInvKernel<Col, Row::n, P::NT_COL, true, true>;
    using KCO = ColInvKernel<Col, Row::n, P::NT_COL, true, true, true>;
    using KCR = ColInvKernel<Col, Row::n, P::NT_COL, true, true, false, true>;
    // the shared-source path: sample-only K_A, the source-spectrum kernel and the shared K_B
    using KTs = ColFwdKernel<Col, Row::n, P::NT_COL, float, true, true>;
    using KRs = ColFwdKernel<Col, Row::n, P::NT_COL, float, false, true>;
    using KDs = ColFwdKernel<Col, Row::n, P::NT_COL, double, false, true>;
    using KSs = ColFwdKernel<Col, Row::n, P::NT_COL, int16_t, false, true>;
    using KBspec = RowFusedKernel<Row, Col::n, P::NT_ROW, false, ROWS_SRC_SPECTRUM>;
    using KBs = RowFusedKernel<Row, Col::n, P::NT_ROW, false, ROWS_SHARED_SRC>;
    using KBPs = RowFusedKernel<Row, Col::n, P::NT_ROW, true, ROWS_SHARED_SRC>;
    // the cross path: K_B from both spectra (the sample side reuses KSs..KBspec)
    using KBb = RowFusedKernel<Row, Col::n, P::NT_ROW, false, ROWS_BOTH_SPECTRA>;
    using KBPb = RowFusedKernel<Row, Col::n, P::NT_ROW, true, ROWS_BOTH_SPECTRA>;
    if (prepare_kernel<KT>(KT::SMEM) != 0 || prepare_kernel<KR>(KR::SMEM) != 0 || prepare_kernel<KD>(KD::SMEM) != 0 ||
        prepare_kernel<KS>(KS::SMEM) != 0 ||
        (plan->phat ? prepare_kernel<KBP>(KBP::SMEM) : prepare_kernel<KB>(KB::SMEM)) != 0 || prepare_kernel<KC>(KC::SMEM) != 0 ||
        prepare_kernel<KCW>(KCW::SMEM) != 0 || prepare_kernel<KCO>(KCO::SMEM) != 0 || prepare_kernel<KCR>(KCR::SMEM) != 0)
        return -1;
    if (prepare_kernel<KTs>(KTs::SMEM) != 0 || prepare_kernel<KRs>(KRs::SMEM) != 0 || prepare_kernel<KDs>(KDs::SMEM) != 0 ||
        prepare_kernel<KSs>(KSs::SMEM) != 0 || prepare_kernel<KBspec>(KBspec::SMEM) != 0 ||
        (plan->phat ? prepare_kernel<KBPs>(KBPs::SMEM) : prepare_kernel<KBs>(KBs::SMEM)) != 0 ||
        (plan->phat ? prepare_kernel<KBPb>(KBPb::SMEM) : prepare_kernel<KBb>(KBb::SMEM)) != 0)
        return -1;
    plan->run_wave = [plan](const Wave& w) {
        return w.spec ? run_static_wave<P, true>(plan, w) : run_static_wave<P, false>(plan, w);
    };
    plan->source_spectrum = [plan](const Wave& w, void* spec) {
        return static_source_spectrum<P>(plan, w, static_cast<cplx*>(spec));
    };
    plan->cross_samples = [plan](const Wave& w) { return static_cross_samples<P>(plan, w); };
    plan->cross_rows = [plan](const Wave& w) { return static_cross_rows<P>(plan, w); };
    plan->runner_up = [plan](const Wave& w) { return static_runner_up<P>(plan, w); };
    return 0;
}


}  // namespace asc
