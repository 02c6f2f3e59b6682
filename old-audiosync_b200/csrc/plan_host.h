// plan_host.h -- host-side pieces shared by the translation units of libaudiosync_cuda.so:
// the per-length plan record, table upload, launch accounting / event timing, tensor-map
// encoding and the programmatic-dependent-launch wrapper.  The kernels are instantiated in
// several translation units (one per static plan, one per arithmetic type of the runtime-radix
// kernels) so that the library builds in parallel.
#pragma once

#include <cuda_runtime.h>

#include <algorithm>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

#include "context.h"
#include "fft_kernels.cuh"
#include "fft_plan.h"
#include "fft_small.cuh"
#include "gen_plan.h"

namespace asc {

// -------------------------------------------------------------------- plan
struct FftPlan {
    PathKind kind = PATH_DIRECT;
    long long L = 0;
    int M1 = 0, M2 = 0;
    std::string desc;
    size_t ws_bytes_per_pair = 0;
    DevBuf col_tw, col_tc, row_tw, row_rev, row_tab, m_lo, m_hi;   // static four-step
    DevBuf wm, wn;                                   // short-length kernel
    SmallPlan small;
    GenShape gen{};                                  // runtime-radix four-step kernels
    DevBuf g_wcol, g_wrow, g_wpos, g_lo, g_hi, g_p2f_col, g_f2p_row;
    bool phat = false;                               // PHAT weighting in the split step (AUDIOSYNC_CUDA_WEIGHT_PHAT)
    DevBuf phat_rev, phat_lo, phat_hi;               // its twiddle w = W_N^k1 * phat_rev[e] (row kernel's position order)
    double peak_scale = 1.0;                         // r_reference = r_kernel * peak_scale
    // enqueues the transform kernels for `pairs` pairs (planes/r in ws)
    // (src, smp, dtype, src_pitch, smp_pitch [elements between pairs], workspace, peaks, pairs, stream,
    //  lag window: nullptr for the unwindowed kernels, else the windowed twins of the argmax step)
    std::function<int(audiosync_cuda_ctx*, DeviceState&, const void*, const void*, int, long long, long long,
                      void*, PairPeak*, int, cudaStream_t, const RawWindow*)> run_wave;
    // Static plans only: the reuse path of a batch whose pairs share one source.  source_spectrum
    // (ctx, d, src, dtype, spec, peaks, stream) writes the source's forward rows into spec (M complex)
    // once per call; run_shared_wave is run_wave with spec in place of the source and its pitch.
    std::function<int(audiosync_cuda_ctx*, DeviceState&, const void*, int, void*, PairPeak*, cudaStream_t)> source_spectrum;
    std::function<int(audiosync_cuda_ctx*, DeviceState&, const void*, const void*, int, long long,
                      void*, PairPeak*, int, cudaStream_t, const RawWindow*)> run_shared_wave;
    ~FftPlan() {
        col_tw.release(); col_tc.release(); row_tw.release(); row_rev.release(); row_tab.release(); m_lo.release(); m_hi.release();
        wm.release(); wn.release();
        g_wcol.release(); g_wrow.release(); g_lo.release(); g_hi.release();
        g_wpos.release(); g_p2f_col.release(); g_f2p_row.release();
        phat_rev.release(); phat_lo.release(); phat_hi.release();
    }
};

template <class E>
static inline int upload(DevBuf& b, const std::vector<E>& v) {
    if (b.ensure(v.size() * sizeof(E)) != 0) return -1;
    ASC_CUDA_OK(cudaMemcpy(b.p, v.data(), v.size() * sizeof(E), cudaMemcpyHostToDevice));
    return 0;
}

// ------------------------------------------------------------------ launch
template <class F>
static int launch(audiosync_cuda_ctx* ctx, DeviceState& d, int cls, cudaStream_t st, F&& fn) {
    ProfileRecord rec{cls, nullptr, nullptr};
    const bool prof = ctx->profile;
    if (prof) {
        std::lock_guard<std::mutex> lk(d.prof_mu);
        for (cudaEvent_t* e : {&rec.e0, &rec.e1}) {
            if (!d.event_pool.empty()) { *e = d.event_pool.back(); d.event_pool.pop_back(); }
            else ASC_CUDA_OK(cudaEventCreate(e));
        }
        ASC_CUDA_OK(cudaEventRecord(rec.e0, st));
    }
    fn();
    ASC_CUDA_OK(cudaGetLastError());
    if (prof) {
        ASC_CUDA_OK(cudaEventRecord(rec.e1, st));
        std::lock_guard<std::mutex> lk(d.prof_mu);
        d.prof_pending.push_back(rec);
    }
    ctx->launches.fetch_add(1, std::memory_order_relaxed);
    return 0;
}

// ------------------------------------------------------------ tensor maps
// Column tiles are staged by the TMA unit from 3-D views [slice][row][2*M2 floats] of the
// caller's arrays and of the workspace planes.  The descriptors are encoded on the host per
// launch (cuTensorMapEncodeTiled, reached through the runtime: the library does not link
// libcuda) and travel as grid-constant kernel parameters.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static EncodeTiledFn tensor_map_encoder() {
    static const EncodeTiledFn fn = [] {
        void* f = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &f, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess) {
            cudaGetLastError();
            f = nullptr;
        }
        return reinterpret_cast<EncodeTiledFn>(f);
    }();
    return fn;
}
// [slices][rows][2*M2 floats], `slice_pitch_bytes` between slices; box = 32 floats x box_rows x 1.
static int make_tile_map(CUtensorMap* tm, const void* base, int M2, int rows, size_t slice_pitch_bytes,
                         size_t slices, int box_rows) {
    EncodeTiledFn enc = tensor_map_encoder();
    if (!enc) return -1;
    const cuuint64_t gdim[3] = {(cuuint64_t)2 * M2, (cuuint64_t)rows, (cuuint64_t)std::max<size_t>(slices, 1)};
    const cuuint64_t gstride[2] = {(cuuint64_t)M2 * sizeof(cplx), (cuuint64_t)slice_pitch_bytes};
    const cuuint32_t box[3] = {32u, (cuuint32_t)box_rows, 1u};
    const cuuint32_t estride[3] = {1u, 1u, 1u};
    // L2 promotion measured (64 / 128 / 256 B): no gain, 256 B costs K_C 0.25 us/pair
    const CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<void*>(base), gdim, gstride, box, estride,
                           CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                           CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    return r == CUDA_SUCCESS ? 0 : -1;
}

// Stage launches of the static path: programmatic dependent launch (see pdl_prologue).
static bool pdl_enabled() {
    static const bool on = getenv("AUDIOSYNC_CUDA_NO_PDL") == nullptr;   // diagnostic knob: plain stream-ordered launches
    return on;
}
template <class... KArgs, class... Args>
static void launch_stage(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = pdl_enabled() ? 1 : 0;
    cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);   // errors surface through cudaGetLastError in launch()
}

template <class K>
static int prepare_kernel(size_t smem) {
    if (smem > 48 * 1024)
        ASC_CUDA_OK(cudaFuncSetAttribute(fft_kernel_entry<K>,
                                         cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    return 0;
}


// Builders instantiated in their own translation units.
template <class P> int build_static_plan(FftPlan* plan);     // static_plan_impl.cuh: one per interval length
// gen_impl.cuh: launchers of the runtime-radix kernels per (arithmetic type, CTA size)
template <typename T, int NT>
struct GenStage {
    static int prepare_cols(const GenShape& sh);
    static int prepare_rows(const GenShape& sh, bool phat);
    static int col_fwd(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, const void* src, const void* smp, int dtype,
                       long long sp, long long mp, void* ws, PairPeak* peaks, int pairs, cudaStream_t st);
    static int rows(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, void* ws, int pairs, cudaStream_t st);
    static int col_inv(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, void* ws, PairPeak* peaks, int pairs,
                       cudaStream_t st, const RawWindow* win);
};

// static_rows.cu: the rows of a runtime-radix fp32 plan on a static row kernel (RowFusedKernel<RL, 0, NT>)
// when the plan's M2 has one (GenShape::static_rows).  prepare: tables + kernel attributes.
int static_rows_prepare(FftPlan* plan);
int static_rows_launch(FftPlan* plan, audiosync_cuda_ctx* ctx, DeviceState& d, void* ws, int pairs, cudaStream_t st);

}  // namespace asc
