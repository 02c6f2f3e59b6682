/*
 * include/audiosync_cuda.h -- C ABI of libaudiosync_cuda.so
 *
 * B200 (sm_100a) replacement for ONE translation unit of vidify/old-audiosync:
 * src/cross_correlation.c.  Plain C types only; no torch / CUDA types in any
 * signature (streams and device pointers travel as void*).
 *
 * Part 1 re-exports, unchanged, the two functions the reference declares in
 * include/audiosync/cross_correlation.h:10-11 and :24-25, so the reference's
 * src/audiosync.c (interval loop, :226-259) and src/bind.c link against this
 * library instead of cross_correlation.c + -lfftw3 with no source change.
 * Part 2 supplies the FFTW-named allocators src/audiosync.c:189,277 calls.
 * Part 3 is new surface: a reusable context and a batched entry point that
 * takes many (source, sample) pairs at once, on host or device memory, and
 * shards them over the GPUs of one box.
 *
 * There is no CPU fallback: every entry point that computes fails (returns
 * -1 / NaN and prints one "audiosync: ..." line on stderr) when no CUDA
 * device or no sm_100 kernel image is available.
 */
#ifndef AUDIOSYNC_CUDA_H
#define AUDIOSYNC_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------
 * Part 1 -- drop-in for reference src/cross_correlation.c
 * ------------------------------------------------------------------------ */

/* Replaces reference src/cross_correlation.c:133-307
 * (decl include/audiosync/cross_correlation.h:24-25).
 *
 * source[0 .. 2*sample_len), input_sample[0 .. sample_len): caller-owned host
 * doubles, never modified; exactly those prefixes are snapshotted to the GPU
 * at call time (the reference's reader threads keep appending behind them).
 * Computes r = c2r(r2c(source) * conj(r2c(zero-padded sample))) (length
 * 2*sample_len, unnormalised), idx = the reference's max_abs_index(r)
 * (:52-67: signed r[0] seed, strict >, first index wins), folds idx into a
 * signed lag (:256-271) and evaluates the Pearson coefficient of the aligned
 * windows of the ORIGINAL double inputs (:74-116, :272-273).
 *
 * Returns 0 on success; -1 if the coefficient is NaN (outputs already
 * written: *lag folded, *coefficient NaN -- :276) or on any CUDA/allocation
 * failure (outputs untouched, one stderr line).  Prints the reference's
 * "%ld frames of delay with a confidence of %f" line (:278) when the
 * reference's global_debug (or audiosync_cuda_set_debug) is on.
 * Thread-safe and reentrant: every caller leases its own stream, input mirrors and
 * scratch on the default context, so concurrent callers overlap each other's upload
 * and kernels (the reference's mutex likewise covers only FFTW planning, :33-44).
 * Pageable buffers are staged through pinned bounce buffers, page-locked ones (e.g.
 * from fftw_alloc_real below) are read by the copy engine in place.
 * Environment: AUDIOSYNC_CUDA_DEVICE=k (default 0) or AUDIOSYNC_CUDA_DEVICES=all|i,j,..
 * (callers are spread round-robin over the devices), AUDIOSYNC_CUDA_DROPIN_SLOTS=n
 * in-flight calls per device (default 3). */
int cross_correlation(double *source, double *input_sample,
                      const size_t sample_len, long *lag, double *coefficient);

/* Replaces reference src/cross_correlation.c:74-116
 * (decl include/audiosync/cross_correlation.h:10-11).  Pointer ranges of equal
 * length on the host; computed on the GPU in fp64.  Identical windows give
 * exactly 1.0, a zero-variance window gives NaN, as the reference's
 * tests/test_pearson_coefficient.c asserts.  NaN on CUDA failure. */
double pearson_coefficient(double *source_start, const double *source_end,
                           double *sample_start, const double *sample_end);

/* ------------------------------------------------------------------------
 * Part 2 -- allocators with FFTW's names (reference src/audiosync.c:189,277
 * calls fftw_alloc_real / fftw_free for the 2,880,000-double source buffer).
 * Memory is page-locked host memory when a CUDA device is present (so the
 * per-interval upload is a straight DMA), otherwise 64-byte aligned malloc.
 * ------------------------------------------------------------------------ */
void   *fftw_malloc(size_t n_bytes);
double *fftw_alloc_real(size_t n);
void   *fftw_alloc_complex(size_t n);        /* n * 2 doubles */
void    fftw_free(void *p);

/* Interval-schedule residency (SURVEY 8f rank 1) -- OPT-IN.  By default every call reads the
 * host buffers afresh, exactly like the reference.  The reference's loop
 * (src/audiosync.c:226-259) calls cross_correlation() with the same two buffers and a growing
 * sample_len while its reader threads only append; a caller with that access pattern may
 * switch residency on (audiosync_cuda_set_residency(1) or env AUDIOSYNC_CUDA_RESIDENT=1): when
 * `source` comes from the allocators above, the library then keeps the fp64 prefixes it has
 * already uploaded on the device and a call transfers only the frames that arrived since the
 * previous one.  A session is reused only if both pointers are unchanged, sample_len grew
 * strictly, nothing was freed through fftw_free in between, and 64 probe values of each cached
 * prefix still match the host buffers; otherwise everything is uploaded again.  The probes are
 * a guard against reuse of the buffers for another recording, NOT a proof: a caller that edits
 * already-submitted frames in place between growing calls must leave residency off. */
void audiosync_cuda_set_residency(int on);
/* Counters of the drop-in cross_correlation() since load: calls, host->device bytes, and
 * calls that reused a resident session.  Any pointer may be NULL. */
void audiosync_cuda_dropin_stats(uint64_t *calls, uint64_t *h2d_bytes, uint64_t *resident_hits);

/* Largest number of drop-in cross_correlation() calls that were in flight on the GPU(s) at the
 * same time since load (or since the last call with reset != 0): > 1 means concurrent callers
 * really overlapped instead of queueing on a lock. */
int audiosync_cuda_dropin_max_inflight(int reset);

/* ------------------------------------------------------------------------
 * Part 3 -- batched / multi-GPU surface (new; not in the reference)
 * ------------------------------------------------------------------------ */

typedef struct audiosync_cuda_ctx audiosync_cuda_ctx;

/* Element type of the batch calls' sources / samples.
 *   F32, F64: float / double samples.
 *   S16: 16-bit signed PCM, little-endian (ffmpeg's s16le), the value of a sample s being
 *        s * 2^-15 = s / 32768.0 -- the scaling ffmpeg/libswresample and libsndfile apply when they
 *        decode s16 to float or double.  Every int16 maps exactly into fp32 and fp64 under it, and
 *        the library widens on the device, in the first transform pass and in the Pearson step: an
 *        S16 call returns, bit for bit in every field of each record, what the same call returns
 *        with dtype F64 on the doubles s / 32768.0 (every path, precise mode included).  A quarter
 *        of the F64 bytes cross the link (8.64 MB per pair at sample_len 1,440,000, against 17.28
 *        MB in F32 and 34.56 MB in F64).  Shapes, layouts and memspaces are those of F32 / F64.
 *        Accepted by audiosync_cuda_xcorr_batch, audiosync_cuda_xcorr_batch_results and
 *        audiosync_cuda_xcorr_batch_device only: the session pool and audiosync_cuda_synth_pairs
 *        refuse it, and host narrowing does not apply to it.
 * In every dtype any base aligned to its element (4, 8 or 2 bytes) is accepted, such as a view at
 * an odd element offset, x[1:]; the kernels then read it one element at a time where they would
 * read two.  A device base that is not aligned to its element is refused with -1 and nothing is
 * launched (host bases are copied into the library's own device buffers first). */
enum { AUDIOSYNC_CUDA_F32 = 0, AUDIOSYNC_CUDA_F64 = 1, AUDIOSYNC_CUDA_S16 = 2 };
enum { AUDIOSYNC_CUDA_HOST = 0, AUDIOSYNC_CUDA_DEVICE = 1 };

/* Which transform path a given sample_len takes.  AUTO: the static four-step kernels for the
 * six lengths of the reference's interval schedule (src/audiosync.c:50-57); the fp64
 * time-domain kernel below 4,096 frames (where the reference's own unit tests live); a
 * single-CTA FFT for short even 2/3/5-smooth lengths; the runtime-radix four-step kernels for
 * EVERY other length -- 2/3/5-smooth lengths at their own size, all others (odd, prime
 * factors > 5) embedded in the next suitable smooth length N' >= 3 * sample_len, which gives the
 * same r[0 .. 2L) -- so that, like the reference's per-call FFTW plans
 * (src/cross_correlation.c:34, :237), every length costs O(N log N).  Lengths for which no plan
 * fits the device (above ~7 million frames) are refused with -1. */
enum {
    AUDIOSYNC_CUDA_PATH_AUTO   = 0,
    AUDIOSYNC_CUDA_PATH_FFT    = 1,  /* a transform wherever one exists (also below 4,096 frames)   */
    AUDIOSYNC_CUDA_PATH_DIRECT = 2   /* O(L^2) time-domain correlation, fp64; up to 65,536 frames   */
};

/* One record per pair, 64 bytes, identical on host and device. */
typedef struct audiosync_cuda_result {
    int64_t lag;        /* folded lag in frames, [-L, L-1]  (cross_correlation.c:256-271)  */
    double  coef;       /* Pearson coefficient or NaN                                      */
    double  peak;       /* r[raw_index], unnormalised (x N) like FFTW's c2r                */
    int32_t ret;        /* 0 / -1 exactly as cross_correlation() would return              */
    int32_t success;    /* ret == 0 && coef >= 0.95   (src/audiosync.c:254)                */
    int64_t raw_index;  /* argmax index before folding, [0, 2L)                            */
    double  second;     /* second peak: largest |r[i]|, i != raw_index (0 if none) -- a    */
                        /* by-product of the argmax reduction                              */
    double  margin;     /* (|peak| - second) / |peak| (0 when peak == 0): the peak is      */
                        /* unique when this is well above the arithmetic's 1e-6            */
    double  ncc;        /* normalised correlation at the peak: peak / (N * sqrt(Sx2*Sy2)), */
                        /* (PHAT weighting: peak / N, see audiosync_cuda_set_weighting)     */
                        /* N = 2*sample_len, Sx2 / Sy2 = sum of squares of the two aligned */
                        /* windows the coefficient is taken over (cross_correlation.c      */
                        /* :256-271); for lag >= 0 the cosine similarity of the windows.   */
                        /* Empty or all-zero window: peak / 0 (+-inf, or NaN when peak is   */
                        /* 0 too).  SURVEY 8f rank 4.                                       */
} audiosync_cuda_result;

/* devices == NULL or n_devices <= 0: use every visible device.
 * Returns 0 and a context, or -1 (no device, no kernel image, out of memory). */
int  audiosync_cuda_create(audiosync_cuda_ctx **ctx, const int *devices, int n_devices);
void audiosync_cuda_destroy(audiosync_cuda_ctx *ctx);
int  audiosync_cuda_device_count(const audiosync_cuda_ctx *ctx);

/* Host-facing batch call.  sources: [n_pairs][2*sample_len], samples:
 * [n_pairs][sample_len], both contiguous, of `dtype`, in `memspace`.
 *   HOST   : pairs are split in contiguous blocks over the context's devices
 *            (one host thread + one stream per device, chunked and double
 *            buffered so uploads overlap the kernels); pinned buffers are
 *            used in place, pageable ones are staged.
 *   DEVICE : all pointers live on one device of the context; no copies.
 * Outputs are host arrays of n_pairs entries; any of lags/coefs/rets/peaks may
 * be NULL.  Returns 0 if every pair was evaluated (per-pair NaN outcomes are
 * reported in rets[], not here), -1 on CUDA failure. */
int audiosync_cuda_xcorr_batch(audiosync_cuda_ctx *ctx,
                               const void *sources, const void *samples,
                               size_t n_pairs, size_t sample_len,
                               int dtype, int memspace,
                               long *lags, double *coefs, int *rets, double *peaks);

/* Same call, whole result records (incl. raw_index and the second peak) instead of
 * separate arrays.  results: host array of n_pairs audiosync_cuda_result. */
int audiosync_cuda_xcorr_batch_results(audiosync_cuda_ctx *ctx,
                                       const void *sources, const void *samples,
                                       size_t n_pairs, size_t sample_len,
                                       int dtype, int memspace,
                                       audiosync_cuda_result *results);

/* Stream-ordered device call: enqueues every kernel for n_pairs device-resident
 * pairs on `stream` (a cudaStream_t passed as void*, NULL = the context's own
 * stream for that device) and returns without synchronising.  d_results is a
 * device array of n_pairs audiosync_cuda_result.  `device` is a CUDA ordinal
 * that belongs to the context. */
int audiosync_cuda_xcorr_batch_device(audiosync_cuda_ctx *ctx, int device,
                                      const void *d_sources, const void *d_samples,
                                      size_t n_pairs, size_t sample_len, int dtype,
                                      audiosync_cuda_result *d_results, void *stream);

/* ------------------------------------------------------------------------
 * Session pool (SURVEY 8f rank 1): many concurrent audiosync sessions on one device.
 * Each slot owns device-resident source / sample buffers that grow as audio arrives
 * (the reference's reader threads append f64le frames, src/ffmpeg_pipe.c:70-81); when
 * the sessions of a slot range have reached an interval of the schedule
 * (src/audiosync.c:50-70), ONE batched call evaluates that interval for all of them.
 * Only new frames ever cross PCIe, and the transform runs at batch throughput.
 *   dtype F64: slots keep the doubles as sent (results identical to cross_correlation()).
 *   dtype F32: frames are converted on the device as they arrive (half the memory, the
 *              fast fp32 staging path; the coefficient then sees fp32-rounded inputs).
 * ------------------------------------------------------------------------ */
typedef struct audiosync_cuda_pool audiosync_cuda_pool;

int  audiosync_cuda_pool_create(audiosync_cuda_ctx *ctx, int device, size_t n_slots,
                                size_t max_sample_len, int dtype, audiosync_cuda_pool **pool);
void audiosync_cuda_pool_destroy(audiosync_cuda_pool *pool);
/* Forget a slot's frames (a new session starts in it). */
int  audiosync_cuda_pool_reset(audiosync_cuda_pool *pool, size_t slot);
/* Append host doubles to a slot; either count may be 0.  The data is on the device when the
 * call returns.  -1 if the slot would exceed 2 * max_sample_len / max_sample_len frames. */
int  audiosync_cuda_pool_append(audiosync_cuda_pool *pool, size_t slot,
                                const double *source_frames, size_t n_source,
                                const double *sample_frames, size_t n_sample);
/* The same, stream-ordered: returns as soon as the copies are enqueued (arriving doubles cross
 * PCIe in 8 MB pieces; for F32 slots the conversion of one piece overlaps the copy of the next).
 * Page-locked host buffers must stay unchanged until audiosync_cuda_pool_flush() or the next
 * audiosync_cuda_pool_run() returns (pageable ones are copied out before the call returns).
 * pool_run orders itself behind every earlier append. */
int  audiosync_cuda_pool_append_async(audiosync_cuda_pool *pool, size_t slot,
                                      const double *source_frames, size_t n_source,
                                      const double *sample_frames, size_t n_sample);
/* Blocks until every appended frame is in its slot. */
int  audiosync_cuda_pool_flush(audiosync_cuda_pool *pool);
/* Frames a slot holds so far. */
int  audiosync_cuda_pool_fill(const audiosync_cuda_pool *pool, size_t slot,
                              size_t *source_frames, size_t *sample_frames);
/* cross_correlation(source[0, 2L), sample[0, L)) for slots first_slot .. first_slot+n_slots-1
 * as one batch; every one of them must hold at least 2L / L frames.  results: host array of
 * n_slots records.  Returns 0 / -1. */
int  audiosync_cuda_pool_run(audiosync_cuda_pool *pool, size_t first_slot, size_t n_slots,
                             size_t sample_len, audiosync_cuda_result *results);

/* Seeded all-integer synthetic pairs written straight into device memory
 * (same generator as oracle/xcorr_oracle.c: bit-identical values).  Pair ids
 * first_pair .. first_pair+n_pairs-1; stream-ordered like the call above. */
int audiosync_cuda_synth_pairs(audiosync_cuda_ctx *ctx, int device, uint64_t seed,
                               uint64_t first_pair, size_t n_pairs, size_t sample_len,
                               int dtype, void *d_sources, void *d_samples, void *stream);

/* Blocks until everything enqueued by this context on `device` is done. */
int audiosync_cuda_synchronize(audiosync_cuda_ctx *ctx, int device);

/* Tuning / test knobs (default behaviour matches the reference's). */
int  audiosync_cuda_set_path(audiosync_cuda_ctx *ctx, int path);          /* AUTO / FFT / DIRECT */
int  audiosync_cuda_set_wave_pairs(audiosync_cuda_ctx *ctx, int pairs);   /* pairs per kernel wave, 0 = auto */
/* Host narrowing for the HOST-memspace batch calls with dtype F64.  The link, not the GPU, bounds
 * host-fed batches (34.56 MB per 1.44M-frame pair at ~55 GB/s), and the transform is fp32 anyway:
 * the library can convert the doubles to fp32 ON THE HOST while it stages them (copy threads,
 * AUDIOSYNC_CUDA_COPY_THREADS), so that half the bytes cross PCIe.
 *   LOSSLESS (default): only where the conversion is exact -- every double of the chunk the image
 *     of its float, which audio decoded from 16/24-bit PCM or float samples always is.  The Pearson
 *     step then widens the floats back and runs its fp64 arithmetic, so every result bit equals the
 *     un-narrowed call's; the first inexact value (NaN included) ends narrowing for the rest of the
 *     call and that chunk is uploaded as doubles.  Page-locked inputs are fed both ways at once:
 *     whole pairs by the copy engine straight from the caller's memory while the copy threads narrow
 *     others, each taking the next pair when it is free.
 *   ALWAYS: every chunk, exact or not; the call then answers for the fp32 batch of the rounded
 *     values (coefficient ~1e-7 relative from the f64 call's; identical windows still give 1.0).
 *   OFF: the doubles cross the link as they are.
 * Env AUDIOSYNC_CUDA_HOST_NARROWING=0/1/2 sets the mode of new contexts.  Ignored in precise mode. */
enum { AUDIOSYNC_CUDA_NARROW_OFF = 0, AUDIOSYNC_CUDA_NARROW_LOSSLESS = 1, AUDIOSYNC_CUDA_NARROW_ALWAYS = 2 };
int  audiosync_cuda_set_host_narrowing(audiosync_cuda_ctx *ctx, int mode);
/* The host-side conversion itself (copy threads, SIMD): dst[i] = (float)src[i], round to nearest
 * even; returns 1 when every value survived unchanged, 0 otherwise.  Needs no GPU. */
int  audiosync_cuda_host_narrow(float *dst, const double *src, size_t n);
/* Copy threads of this process (pageable staging, host narrowing): AUDIOSYNC_CUDA_COPY_THREADS, default
 * three quarters of the cores the process may run on, at most 12.  With fewer than 8, LOSSLESS
 * narrowing leaves page-locked inputs to the copy engine alone (pageable ones are still narrowed). */
int  audiosync_cuda_copy_threads(void);
/* fp64-ARITHMETIC validation mode: every transform runs on the double-precision instantiation
 * of the runtime-radix kernels (the reference computes in double complex throughout,
 * src/cross_correlation.c:187-239) and the argmax on full double keys -- several times slower
 * than the fp32 product path, peak values within 1e-12 of an fp64 FFT.  A second oracle for the
 * fp32 kernels; env AUDIOSYNC_CUDA_PRECISE=1 selects it for the drop-in cross_correlation(). */
int  audiosync_cuda_set_precise(audiosync_cuda_ctx *ctx, int on);
/* Cross-spectrum weighting of the batch calls, per context (default NONE: the reference's plain
 * correlation).  PHAT is the generalised cross-correlation with phase transform (GCC-PHAT), the
 * standard delay estimator for reverberant or spectrally coloured recordings: with N = 2L,
 * X = DFT_N(source[0, 2L)) and Y = DFT_N(zero-padded sample),
 *     W[k]   = X[k] conj(Y[k]) / (|X[k]| |Y[k]|)    (0 where |X[k]|^2 or |Y[k]|^2 is 0 in the arithmetic type)
 *     r_w[j] = sum_k W[k] e^(2 pi i j k / N)        (unnormalised like FFTW's c2r, so |r_w| <= N)
 * and the record is derived from r_w: raw_index by the reference's argmax rule (signed r_w[0] seed,
 * strict >, first index wins), lag by the same fold, peak / second / margin over r_w, and coef, ret,
 * success the Pearson coefficient of the aligned windows of the original inputs at that lag.  ncc
 * becomes peak / N, the phase coherence at the peak: in [-1, 1], 1 for a pure circular shift, 0
 * when the peak is 0.  The peak is a near-delta whatever the spectral colour or level of either
 * signal; scaling an input by a power of two leaves every record field unchanged.
 * PHAT is defined on the N = 2L spectrum and is served wherever the plan transforms at N = 2L: the
 * six static lengths, the single-CTA kernel (short even 2/3/5-smooth lengths; under AUTO also
 * below 4,096 frames, PHAT never takes the time-domain kernel) and the runtime-radix kernels for
 * 2/3/5-smooth lengths of at least 256 frames, in fp32 and in precise mode.  With PHAT on, a call
 * returns -1 with a message (audiosync_cuda_last_error) and writes no output for PATH_DIRECT, for
 * lengths that would be embedded (not 2/3/5-smooth: a weighted N'-point spectrum is a different
 * function) and for lengths without such a plan.  It applies to xcorr_batch, xcorr_batch_results,
 * xcorr_batch_device and pool_run, every dtype, memspace and host-narrowing mode; the drop-in
 * cross_correlation() never weights.  Returns -1 for an unknown value. */
enum { AUDIOSYNC_CUDA_WEIGHT_NONE = 0, AUDIOSYNC_CUDA_WEIGHT_PHAT = 1 };
int  audiosync_cuda_set_weighting(audiosync_cuda_ctx *ctx, int weighting);
void audiosync_cuda_set_debug(int on);                                    /* same effect as global_debug */
/* Describes the plan for a length, e.g.
 * "fft L=1440000 M1=600 M2=2400 col=6x10x10 row=8x10x30 static", followed by " phat" under
 * PHAT weighting. Returns the
 * number of characters written (excluding the NUL), -1 if buf is too small. */
int audiosync_cuda_describe_plan(audiosync_cuda_ctx *ctx, size_t sample_len,
                                 char *buf, size_t buf_len);

/* Launch accounting: number of kernels this context has launched so far. */
uint64_t audiosync_cuda_launch_count(const audiosync_cuda_ctx *ctx);
/* Host-fed F64 batches since the context was created (or the last call with reset != 0): pairs that
 * crossed the link as doubles -> out[0], pairs narrowed to fp32 on the host -> out[1]. */
int audiosync_cuda_host_feed_stats(audiosync_cuda_ctx *ctx, uint64_t out[2], int reset);

/* Per-kernel device timing.  When enabled every launch is bracketed by CUDA
 * events on its own stream; audiosync_cuda_profile_read() synchronises and
 * returns, for kernel class `i`, its name, launch count and total device
 * milliseconds since the last reset.  Returns the number of classes. */
int audiosync_cuda_profile_enable(audiosync_cuda_ctx *ctx, int on);
int audiosync_cuda_profile_reset(audiosync_cuda_ctx *ctx);
int audiosync_cuda_profile_read(audiosync_cuda_ctx *ctx, int i, char *name, size_t name_len,
                                uint64_t *launches, double *total_ms);

/* Last error message of the calling thread ("" if none). */
const char *audiosync_cuda_last_error(void);
const char *audiosync_cuda_version(void);

#ifdef __cplusplus
}
#endif
#endif /* AUDIOSYNC_CUDA_H */
