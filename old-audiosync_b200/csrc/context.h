// context.h -- host-side state of libaudiosync_cuda: devices, streams,
// growable device buffers, launch accounting and per-kernel event timing.
#pragma once

#include <cuda_runtime.h>

#include <atomic>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <memory>
#include <mutex>
#include <string>
#include <vector>

#include "common.cuh"

namespace asc {

void set_last_error(const char* fmt, ...);

#define ASC_CUDA_OK(expr)                                                              \
    do {                                                                               \
        cudaError_t _e = (expr);                                                       \
        if (_e != cudaSuccess) {                                                       \
            asc::set_last_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), \
                                __FILE__, __LINE__);                                   \
            return -1;                                                                 \
        }                                                                              \
    } while (0)

// Kernel classes for launch accounting / timing.
enum KernelClass {
    KC_SYNTH = 0,
    KC_DIRECT,
    KC_ARGMAX_F64,
    KC_COL_FWD,      // K_A  forward column pass (source and sample)
    KC_ROW_FUSED,    // K_B  forward rows + split + conj-multiply + merge + inverse rows
    KC_COL_INV,      // K_C  inverse column pass + |r| argmax epilogue
    KC_SMALL_FFT,    // single-CTA transform for short lengths
    KC_PEARSON,      // window statistics + coefficient + result record
    KC_SRC_SPECTRUM, // forward rows of a shared source, once per call (RowFusedKernel ROWS_SRC_SPECTRUM)
    KC_COUNT
};

const char* kernel_class_name(int k);

struct DevBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int ensure(size_t need);      // grows (never shrinks); returns 0 / -1
    void release();
};

struct PinnedBuf {
    void* p = nullptr;
    size_t bytes = 0;
    int ensure(size_t need);
    void release();
};

// Internal input type of enqueue_batch beside the public F32 / F64 / S16: fp32 values that are the
// EXACT images of the caller's doubles (lossless host narrowing).  The transform reads them as any
// fp32 batch; the Pearson step widens them and runs the f64 path's arithmetic, so the result record
// is the f64 call's bit for bit.
constexpr int ASC_DTYPE_F32_EXACT = 100;

// Bytes of one input element of `dtype`; 0 for a value that is not an input type.
inline size_t dtype_bytes(int dtype) {
    switch (dtype) {
        case AUDIOSYNC_CUDA_F32: case ASC_DTYPE_F32_EXACT: return 4;
        case AUDIOSYNC_CUDA_F64: return 8;
        case AUDIOSYNC_CUDA_S16: return 2;
    }
    return 0;
}

// Pinned bounce buffers for PAGEABLE host inputs: the host memcpy of piece k + 1 overlaps the
// DMA of piece k and the stream stays asynchronous (a cudaMemcpyAsync straight from pageable
// memory is staged by the driver and blocks the calling thread for the whole transfer).
struct StageRing {
    static constexpr int N = 6;
    static constexpr size_t PIECE = (size_t)8 << 20;
    PinnedBuf buf[N];
    cudaEvent_t ev[N] = {};
    bool pending[N] = {};
    int next = 0;
    void release() {
        for (int i = 0; i < N; i++) {
            buf[i].release();
            if (ev[i]) cudaEventDestroy(ev[i]);
            ev[i] = nullptr; pending[i] = false;
        }
    }
};

struct ProfileRecord { int cls; cudaEvent_t e0, e1; };

struct FftPlan;   // fft_plan.h

// Scratch of one in-flight batch: everything enqueue_batch writes besides the caller's result
// records.  A set is used by one stream at a time; `done` (recorded after every enqueue) orders a
// later enqueue on a DIFFERENT stream behind the previous one, so stream-ordered callers may mix
// streams on one context without corrupting planes, argmax keys or ticket counters.
struct WorkSet {
    DevBuf ws;            // transform workspace (direct: r[]; fft: A/B planes)
    DevBuf peaks;         // PairPeak per in-flight pair
    DevBuf partials;      // PearsonPartial
    DevBuf tickets;       // per-pair completion counters of the Pearson kernel
    DevBuf spec;          // shared-source calls on a static plan: the source's forward rows (M complex)
    cudaEvent_t done = nullptr;
    cudaStream_t last_stream = nullptr;
    bool used = false;
    void release() {
        ws.release(); peaks.release(); partials.release(); tickets.release(); spec.release();
        if (done) cudaEventDestroy(done);
        done = nullptr; used = false;
    }
};

struct DeviceState {
    int device = -1;
    int sm_count = 0;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr;        // compute
    cudaStream_t copy_stream = nullptr;   // uploads for the host-facing batch call
    cudaStream_t narrow_stream = nullptr; // uploads of host-narrowed (f64 -> fp32) pairs, beside the direct ones
    WorkSet work;         // scratch of the batch entry points (serialised by the context mutex)
    DevBuf results;       // audiosync_cuda_result for host-facing calls
    DevBuf in_src[2], in_smp[2];          // device copies of host inputs (double buffered)
    DevBuf in_src32[2], in_smp32[2];      // the host-narrowed pairs of a chunk (fp32 images of f64 inputs)
    PinnedBuf h_results;
    StageRing stage;                      // bounce buffers for pageable host inputs
    cudaEvent_t ev_up[2] = {nullptr, nullptr};
    cudaEvent_t ev_up32[2] = {nullptr, nullptr};
    cudaEvent_t ev_done[2] = {nullptr, nullptr};
    // direct (un-narrowed) upload slices in flight beside the narrowing threads: at most DIRECT_DEPTH
    static constexpr int DIRECT_DEPTH = 4;
    static constexpr size_t DIRECT_SLICE = (size_t)8 << 20;
    cudaEvent_t direct_ev[DIRECT_DEPTH] = {};
    bool direct_pending[DIRECT_DEPTH] = {};
    std::map<size_t, std::shared_ptr<FftPlan>> plans;   // by sample_len
    std::mutex mu;        // serialises users of `work`, `results`, the input mirrors and the staging ring
    std::mutex plan_mu;   // plans are built once and shared by concurrent callers
    // profiling (prof_mu: launches may come from concurrent drop-in callers)
    std::mutex prof_mu;
    std::vector<ProfileRecord> prof_pending;
    std::vector<cudaEvent_t> event_pool;
    uint64_t prof_launches[KC_COUNT] = {0};
    double prof_ms[KC_COUNT] = {0};
};

// Interval-schedule residency of the drop-in cross_correlation() (SURVEY 8f rank 1):
// reference src/audiosync.c:226-259 calls it with the SAME two buffers and a growing
// sample_len (144,000 -> ... -> 1,440,000) while its reader threads only append.  The device
// keeps the fp64 prefixes it already has; a call uploads just the newly arrived frames.
struct ResidentSession {
    static constexpr int NFP = 64;           // fingerprint samples per buffer
    const double* src = nullptr;             // host buffers the session mirrors
    const double* smp = nullptr;
    size_t L = 0;                            // sample_len of the last call
    size_t src_valid = 0, smp_valid = 0;     // doubles already on the device
    uint64_t alloc_gen = 0;                  // allocator generation at the last call
    size_t fp_idx_src[NFP], fp_idx_smp[NFP];
    double fp_val_src[NFP], fp_val_smp[NFP];
    DevBuf d_src, d_smp;
    void invalidate() { src = smp = nullptr; L = src_valid = smp_valid = 0; }
};

}  // namespace asc

namespace asc {
// One in-flight drop-in cross_correlation() call: its own stream, input mirrors, scratch and
// result buffers, so concurrent callers overlap each other's upload and kernels like the
// reference's callers do (its mutex covers only FFTW planning, src/cross_correlation.c:33-44).
struct DropinSlot {
    DeviceState* dev = nullptr;
    cudaStream_t stream = nullptr;
    WorkSet work;
    DevBuf in_src, in_smp, d_res;
    PinnedBuf h_res;
    StageRing stage;
    bool busy = false;
};
}  // namespace asc

struct audiosync_cuda_ctx {
    std::vector<asc::DeviceState> devs;
    std::mutex mu;
    std::vector<std::unique_ptr<asc::DropinSlot>> slots;   // drop-in callers (default context)
    std::mutex slot_mu;
    std::condition_variable slot_cv;
    size_t slot_next = 0;
    int path = AUDIOSYNC_CUDA_PATH_AUTO;
    int wave_pairs = 0;
    bool precise = false;     // fp64 ARITHMETIC in the transforms (validation mode)
    int weighting = AUDIOSYNC_CUDA_WEIGHT_NONE;   // AUDIOSYNC_CUDA_WEIGHT_*: cross-spectrum weighting of the batch calls
    long long lag_lo = INT64_MIN, lag_hi = INT64_MAX;   // lag window of the batch calls (folded lags, inclusive)
    int narrow_host = 1;      // AUDIOSYNC_CUDA_NARROW_*: f64 HOST batches converted to fp32 on the host while staged
    bool profile = false;
    std::atomic<uint64_t> launches{0};
    std::atomic<uint64_t> fed_direct{0}, fed_narrowed{0};   // F64 host-fed pairs: as doubles / narrowed on the host
    asc::ResidentSession resident;           // drop-in cross_correlation() only (default context)

    asc::DeviceState* find(int device);
};
