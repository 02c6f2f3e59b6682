"""Host-side binding of ``libaudiosync_cuda.so`` (ctypes over the C ABI).

This is the Python mirror of the reference's interface for its one hot path:
``cross_correlation`` / ``pearson_coefficient`` keep the names, argument
meaning and error behaviour of reference ``include/audiosync/cross_correlation.h``
(:10-11, :24-25); ``interval_loop`` restates the caller side,
``src/audiosync.c:226-259``, on top of it; ``Context`` exposes the new batched /
multi-GPU surface of ``include/audiosync_cuda.h``.

There is no CPU fallback here or in the library: importing works anywhere,
but every call that computes raises ``AudiosyncCudaError`` when the shared
object or a CUDA device is missing.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Sequence

import numpy as np

__all__ = [
    "AudiosyncCudaError", "lib", "lib_path", "cross_correlation", "pearson_coefficient",
    "interval_loop", "Context", "RESULT_DTYPE", "MIN_CONFIDENCE", "SAMPLE_RATE",
    "INTERV_SAMPLE", "frames_to_ms", "F32", "F64", "S16", "HOST", "DEVICE",
    "PATH_AUTO", "PATH_FFT", "PATH_DIRECT", "WEIGHT_NONE", "WEIGHT_PHAT", "NARROW_OFF", "NARROW_LOSSLESS", "NARROW_ALWAYS", "EXPORTED_SYMBOLS", "shard_pairs", "gather_results", "host_narrow", "copy_threads",
    "cross_correlation_ptr", "RealBuffer", "set_residency", "dropin_stats", "dropin_max_inflight", "SessionPool",
]

F32, F64, S16 = 0, 1, 2          # S16: int16 PCM, value s / 32768 (records == F64 on those doubles, bit for bit)
HOST, DEVICE = 0, 1
PATH_AUTO, PATH_FFT, PATH_DIRECT = 0, 1, 2
WEIGHT_NONE, WEIGHT_PHAT = 0, 1  # cross-spectrum weighting of the batch calls (GCC-PHAT: ncc = peak / N)
NARROW_OFF, NARROW_LOSSLESS, NARROW_ALWAYS = 0, 1, 2

_NP_DTYPES = {np.dtype(np.float32): F32, np.dtype(np.float64): F64, np.dtype(np.int16): S16}

MIN_CONFIDENCE = 0.95                                             # audiosync.h:24
SAMPLE_RATE = 48000                                               # audiosync.h:14
INTERV_SAMPLE = [s * SAMPLE_RATE for s in (3, 6, 10, 15, 20, 30)]  # src/audiosync.c:50-57

# mirrors struct audiosync_cuda_result (64 bytes)
RESULT_DTYPE = np.dtype([("lag", "<i8"), ("coef", "<f8"), ("peak", "<f8"),
                         ("ret", "<i4"), ("success", "<i4"), ("raw_index", "<i8"), ("second", "<f8"),
                         ("margin", "<f8"), ("ncc", "<f8")])
assert RESULT_DTYPE.itemsize == 64

# every symbol include/audiosync_cuda.h declares
EXPORTED_SYMBOLS = [
    "cross_correlation", "pearson_coefficient",
    "fftw_malloc", "fftw_alloc_real", "fftw_alloc_complex", "fftw_free",
    "audiosync_cuda_create", "audiosync_cuda_destroy", "audiosync_cuda_device_count",
    "audiosync_cuda_xcorr_batch", "audiosync_cuda_xcorr_batch_results", "audiosync_cuda_xcorr_batch_device",
    "audiosync_cuda_xcorr_shared_source", "audiosync_cuda_xcorr_shared_source_device",
    "audiosync_cuda_synth_pairs", "audiosync_cuda_synchronize",
    "audiosync_cuda_set_path", "audiosync_cuda_set_wave_pairs", "audiosync_cuda_set_debug", "audiosync_cuda_set_precise", "audiosync_cuda_set_weighting",
    "audiosync_cuda_set_lag_window",
    "audiosync_cuda_set_host_narrowing", "audiosync_cuda_host_narrow", "audiosync_cuda_copy_threads",
    "audiosync_cuda_set_residency", "audiosync_cuda_dropin_stats", "audiosync_cuda_dropin_max_inflight",
    "audiosync_cuda_pool_create", "audiosync_cuda_pool_destroy", "audiosync_cuda_pool_reset",
    "audiosync_cuda_pool_append", "audiosync_cuda_pool_append_async", "audiosync_cuda_pool_flush",
    "audiosync_cuda_pool_fill", "audiosync_cuda_pool_run",
    "audiosync_cuda_describe_plan", "audiosync_cuda_launch_count", "audiosync_cuda_host_feed_stats",
    "audiosync_cuda_profile_enable", "audiosync_cuda_profile_reset",
    "audiosync_cuda_profile_read", "audiosync_cuda_last_error", "audiosync_cuda_version",
]


class AudiosyncCudaError(RuntimeError):
    pass


_PKG_DIR = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_LIB: Optional[C.CDLL] = None


def lib_path() -> str:
    return os.environ.get("AUDIOSYNC_CUDA_LIB", os.path.join(_PKG_DIR, "libaudiosync_cuda.so"))


def lib() -> C.CDLL:
    """Loads the shared object; raises (never falls back) if it is missing."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise AudiosyncCudaError(
            f"{path} not built: run `make -C old-audiosync_b200` or __graft_entry__.build(); "
            "there is no CPU fallback")
    L = C.CDLL(path)
    vp, sz, i32, u64, dbl = C.c_void_p, C.c_size_t, C.c_int, C.c_uint64, C.c_double
    L.cross_correlation.restype = i32
    L.cross_correlation.argtypes = [vp, vp, sz, C.POINTER(C.c_long), C.POINTER(dbl)]
    L.pearson_coefficient.restype = dbl
    L.pearson_coefficient.argtypes = [vp, vp, vp, vp]
    L.fftw_malloc.restype = vp
    L.fftw_malloc.argtypes = [sz]
    L.fftw_alloc_real.restype = vp
    L.fftw_alloc_real.argtypes = [sz]
    L.fftw_alloc_complex.restype = vp
    L.fftw_alloc_complex.argtypes = [sz]
    L.fftw_free.restype = None
    L.fftw_free.argtypes = [vp]
    L.audiosync_cuda_create.restype = i32
    L.audiosync_cuda_create.argtypes = [C.POINTER(vp), C.POINTER(i32), i32]
    L.audiosync_cuda_destroy.restype = None
    L.audiosync_cuda_destroy.argtypes = [vp]
    L.audiosync_cuda_device_count.restype = i32
    L.audiosync_cuda_device_count.argtypes = [vp]
    L.audiosync_cuda_xcorr_batch.restype = i32
    L.audiosync_cuda_xcorr_batch.argtypes = [vp, vp, vp, sz, sz, i32, i32, vp, vp, vp, vp]
    L.audiosync_cuda_xcorr_batch_results.restype = i32
    L.audiosync_cuda_xcorr_batch_results.argtypes = [vp, vp, vp, sz, sz, i32, i32, vp]
    L.audiosync_cuda_xcorr_batch_device.restype = i32
    L.audiosync_cuda_xcorr_batch_device.argtypes = [vp, i32, vp, vp, sz, sz, i32, vp, vp]
    L.audiosync_cuda_xcorr_shared_source.restype = i32
    L.audiosync_cuda_xcorr_shared_source.argtypes = [vp, vp, vp, sz, sz, i32, i32, vp]
    L.audiosync_cuda_xcorr_shared_source_device.restype = i32
    L.audiosync_cuda_xcorr_shared_source_device.argtypes = [vp, i32, vp, vp, sz, sz, i32, vp, vp]
    L.audiosync_cuda_synth_pairs.restype = i32
    L.audiosync_cuda_synth_pairs.argtypes = [vp, i32, u64, u64, sz, sz, i32, vp, vp, vp]
    L.audiosync_cuda_synchronize.restype = i32
    L.audiosync_cuda_synchronize.argtypes = [vp, i32]
    L.audiosync_cuda_set_path.restype = i32
    L.audiosync_cuda_set_path.argtypes = [vp, i32]
    L.audiosync_cuda_set_host_narrowing.restype = i32
    L.audiosync_cuda_set_host_narrowing.argtypes = [vp, i32]
    L.audiosync_cuda_copy_threads.restype = i32
    L.audiosync_cuda_copy_threads.argtypes = []
    L.audiosync_cuda_host_narrow.restype = i32
    L.audiosync_cuda_host_narrow.argtypes = [vp, vp, C.c_size_t]
    L.audiosync_cuda_set_precise.restype = i32
    L.audiosync_cuda_set_precise.argtypes = [vp, i32]
    L.audiosync_cuda_set_weighting.restype = i32
    L.audiosync_cuda_set_weighting.argtypes = [vp, i32]
    L.audiosync_cuda_set_lag_window.restype = i32
    L.audiosync_cuda_set_lag_window.argtypes = [vp, C.c_int64, C.c_int64]
    L.audiosync_cuda_set_wave_pairs.restype = i32
    L.audiosync_cuda_set_wave_pairs.argtypes = [vp, i32]
    L.audiosync_cuda_set_residency.restype = None
    L.audiosync_cuda_set_residency.argtypes = [i32]
    L.audiosync_cuda_dropin_stats.restype = None
    L.audiosync_cuda_dropin_stats.argtypes = [C.POINTER(C.c_uint64)] * 3
    L.audiosync_cuda_dropin_max_inflight.restype = i32
    L.audiosync_cuda_dropin_max_inflight.argtypes = [i32]
    L.audiosync_cuda_pool_create.restype = i32
    L.audiosync_cuda_pool_create.argtypes = [vp, i32, sz, sz, i32, C.POINTER(vp)]
    L.audiosync_cuda_pool_destroy.restype = None
    L.audiosync_cuda_pool_destroy.argtypes = [vp]
    L.audiosync_cuda_pool_reset.restype = i32
    L.audiosync_cuda_pool_reset.argtypes = [vp, sz]
    L.audiosync_cuda_pool_append.restype = i32
    L.audiosync_cuda_pool_append.argtypes = [vp, sz, vp, sz, vp, sz]
    L.audiosync_cuda_pool_append_async.restype = i32
    L.audiosync_cuda_pool_append_async.argtypes = [vp, sz, vp, sz, vp, sz]
    L.audiosync_cuda_pool_flush.restype = i32
    L.audiosync_cuda_pool_flush.argtypes = [vp]
    L.audiosync_cuda_pool_fill.restype = i32
    L.audiosync_cuda_pool_fill.argtypes = [vp, sz, C.POINTER(sz), C.POINTER(sz)]
    L.audiosync_cuda_pool_run.restype = i32
    L.audiosync_cuda_pool_run.argtypes = [vp, sz, sz, sz, vp]
    L.audiosync_cuda_set_debug.restype = None
    L.audiosync_cuda_set_debug.argtypes = [i32]
    L.audiosync_cuda_describe_plan.restype = i32
    L.audiosync_cuda_describe_plan.argtypes = [vp, sz, C.c_char_p, sz]
    L.audiosync_cuda_host_feed_stats.restype = i32
    L.audiosync_cuda_host_feed_stats.argtypes = [vp, C.POINTER(u64), i32]
    L.audiosync_cuda_launch_count.restype = u64
    L.audiosync_cuda_launch_count.argtypes = [vp]
    L.audiosync_cuda_profile_enable.restype = i32
    L.audiosync_cuda_profile_enable.argtypes = [vp, i32]
    L.audiosync_cuda_profile_reset.restype = i32
    L.audiosync_cuda_profile_reset.argtypes = [vp]
    L.audiosync_cuda_profile_read.restype = i32
    L.audiosync_cuda_profile_read.argtypes = [vp, i32, C.c_char_p, sz, C.POINTER(u64), C.POINTER(dbl)]
    L.audiosync_cuda_last_error.restype = C.c_char_p
    L.audiosync_cuda_version.restype = C.c_char_p
    _LIB = L
    return L


def last_error() -> str:
    return lib().audiosync_cuda_last_error().decode(errors="replace")


def frames_to_ms(lag_frames: int) -> int:
    """round(lag * 1000 / 48000), src/audiosync.c:255 with audiosync.h:21."""
    import math
    x = lag_frames * (1000.0 / SAMPLE_RATE)
    return int(math.copysign(math.floor(abs(x) + 0.5), x))   # C round(): half away from zero


# ------------------------------------------------------------ multi-GPU sharding

def shard_pairs(n_pairs: int, world: int, rank: int):
    """Contiguous block split of pair ids over ``world`` devices / ranks.

    Returns ``(first, count)``: ``n_pairs // world`` each, the remainder going to
    the low ranks -- the same split the in-library dispatcher applies to its
    devices (``audiosync_cuda_xcorr_batch``, HOST memspace).  Pairs are
    independent, so there is no data-path collective: every rank works on its
    own block and only the 40-byte result records are gathered on the host.
    """
    if world <= 0 or not 0 <= rank < world or n_pairs < 0:
        raise ValueError("bad shard request")
    base, rem = divmod(n_pairs, world)
    first = rank * base + min(rank, rem)
    return first, base + (1 if rank < rem else 0)


def gather_results(local: np.ndarray, n_pairs: int, dst: int = 0, group=None):
    """Host gather of the per-pair result records (``RESULT_DTYPE``) of every rank.

    ``local`` holds this rank's block, in pair order; rank ``dst`` returns the
    ``n_pairs`` records in global pair order, the others return ``None``.  Works on
    any ``torch.distributed`` backend (the records travel as CPU byte tensors
    through ``gather_object``-free point-to-point ``gather``); with no process
    group it is the identity.
    """
    import torch
    import torch.distributed as dist
    local = np.ascontiguousarray(local, dtype=RESULT_DTYPE)
    if not (dist.is_available() and dist.is_initialized()):
        if local.shape[0] != n_pairs:
            raise ValueError("single process must hold every pair")
        return local
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    first, count = shard_pairs(n_pairs, world, rank)
    if local.shape[0] != count:
        raise ValueError(f"rank {rank} holds {local.shape[0]} records, its shard has {count}")
    # equal-size payloads: pad every block to the largest shard
    width = (n_pairs + world - 1) // world * RESULT_DTYPE.itemsize
    buf = torch.zeros(max(width, 1), dtype=torch.uint8)
    raw = torch.from_numpy(local.view(np.uint8).reshape(-1).copy())
    buf[: raw.numel()] = raw
    backend = dist.get_backend(group)
    if backend == "nccl":                       # NCCL moves device memory only
        dev = torch.device("cuda", torch.cuda.current_device())
        parts = [torch.empty_like(buf, device=dev) for _ in range(world)]
        dist.all_gather(parts, buf.to(dev), group=group)
        parts = [p.cpu() for p in parts] if rank == dst else None
    else:
        parts = [torch.empty_like(buf) for _ in range(world)] if rank == dst else None
        dist.gather(buf, parts, dst=dst, group=group)
    if rank != dst:
        return None
    out = np.empty(n_pairs, dtype=RESULT_DTYPE)
    for r in range(world):
        f, c = shard_pairs(n_pairs, world, r)
        out[f:f + c] = parts[r].numpy()[: c * RESULT_DTYPE.itemsize].view(RESULT_DTYPE)
    return out


# ----------------------------------------------------------- drop-in functions

def cross_correlation(source: np.ndarray, sample: np.ndarray):
    """``int cross_correlation(double*, double*, size_t, long*, double*)``.

    Returns ``(ret, lag, coefficient)``.  ``source`` must hold at least
    ``2 * len(sample)`` doubles; only that prefix is read.  ret == -1 with a NaN
    coefficient means the reference's NaN gate fired (outputs are still valid);
    ret == -1 with ``lag is None`` means the GPU call itself failed.
    """
    source = np.ascontiguousarray(source, dtype=np.float64)
    sample = np.ascontiguousarray(sample, dtype=np.float64)
    n = sample.shape[0]
    if source.shape[0] < 2 * n:
        raise ValueError("source must be at least twice as long as sample")
    lag = C.c_long(-(2 ** 62))
    coef = C.c_double(12345.0)
    ret = lib().cross_correlation(source.ctypes.data, sample.ctypes.data, n, C.byref(lag), C.byref(coef))
    if ret != 0 and lag.value == -(2 ** 62):
        raise AudiosyncCudaError("cross_correlation failed: " + last_error())
    return ret, lag.value, coef.value


def cross_correlation_ptr(source_ptr: int, sample_ptr: int, sample_len: int):
    """The same call on raw host addresses (no NumPy copy): what reference src/audiosync.c:246
    does with its ``fftw_alloc_real`` source and ``malloc`` sample buffers."""
    lag = C.c_long(-(2 ** 62))
    coef = C.c_double(12345.0)
    ret = lib().cross_correlation(source_ptr, sample_ptr, sample_len, C.byref(lag), C.byref(coef))
    if ret != 0 and lag.value == -(2 ** 62):
        raise AudiosyncCudaError("cross_correlation failed: " + last_error())
    return ret, lag.value, coef.value


class RealBuffer:
    """``fftw_alloc_real(n)`` / ``fftw_free`` of this library (pinned host doubles) as a NumPy view.
    A source held in one makes the drop-in call eligible for interval-schedule residency."""

    def __init__(self, n: int):
        self.n = int(n)
        self.ptr = lib().fftw_alloc_real(self.n)
        if not self.ptr:
            raise AudiosyncCudaError("fftw_alloc_real failed")
        self.array = np.ctypeslib.as_array(C.cast(self.ptr, C.POINTER(C.c_double)), shape=(self.n,))

    def free(self):
        if self.ptr:
            self.array = None
            lib().fftw_free(self.ptr)
            self.ptr = None

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.free()


def copy_threads() -> int:
    """Copy threads of this process (pageable staging, host narrowing)."""
    return int(lib().audiosync_cuda_copy_threads())


def host_narrow(x: np.ndarray):
    """(float32 copy of x, exact) through the library's host-side conversion (no GPU needed)."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    out = np.empty(x.shape, np.float32)
    exact = lib().audiosync_cuda_host_narrow(out.ctypes.data, x.ctypes.data, x.size)
    return out, bool(exact)


def set_residency(on: bool) -> None:
    """Interval-schedule residency of the drop-in ``cross_correlation`` (opt-in, default off)."""
    lib().audiosync_cuda_set_residency(1 if on else 0)


def dropin_stats():
    """(calls, host->device bytes, resident-session hits) of the drop-in call since load."""
    a, b, c = C.c_uint64(), C.c_uint64(), C.c_uint64()
    lib().audiosync_cuda_dropin_stats(C.byref(a), C.byref(b), C.byref(c))
    return int(a.value), int(b.value), int(c.value)


def dropin_max_inflight(reset: bool = False) -> int:
    """Largest number of drop-in calls in flight at the same time (see include/audiosync_cuda.h)."""
    return int(lib().audiosync_cuda_dropin_max_inflight(1 if reset else 0))


def pearson_coefficient(x: np.ndarray, y: np.ndarray) -> float:
    """``double pearson_coefficient(start, end, start, end)`` on two equal-length windows."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.ascontiguousarray(y, dtype=np.float64)
    if x.shape != y.shape or x.ndim != 1:
        raise ValueError("windows must be 1-D and of equal length")
    n = x.shape[0]
    return float(lib().pearson_coefficient(x.ctypes.data, x.ctypes.data + 8 * n,
                                           y.ctypes.data, y.ctypes.data + 8 * n))


def interval_loop(source: np.ndarray, sample: np.ndarray, call=None):
    """The caller loop of reference src/audiosync.c:226-259 on complete buffers.

    ``call(L) -> (ret, lag, coef)`` replaces the NumPy drop-in wrapper when given (e.g.
    ``cross_correlation_ptr`` on a ``RealBuffer``, the way the reference holds its source).

    Calls the drop-in ``cross_correlation`` on the six interval prefixes, skips
    failed intervals (:247-249), stops at the first ``coef >= 0.95`` (:254-258)
    and converts that lag to milliseconds (:255).  Returns a dict with the
    per-interval tuples and ``final_ret`` / ``final_lag`` as ``audiosync_run``
    would report them (on failure the last frame lag, unconverted).
    """
    rets, lags, coefs, succ = [], [], [], []
    final_ret, lag = -1, 0
    for L in INTERV_SAMPLE:
        if call is not None:
            ret, lag_i, coef = call(L)
        else:
            ret, lag_i, coef = cross_correlation(source[:2 * L], sample[:L])
        lag = lag_i
        ok = ret == 0 and coef >= MIN_CONFIDENCE
        rets.append(ret); lags.append(lag_i); coefs.append(coef); succ.append(int(ok))
        if ret < 0:
            continue
        if ok:
            lag = frames_to_ms(lag_i)
            final_ret = 0
            break
    return dict(n=len(rets), rets=rets, lags=lags, coefs=coefs, succ=succ,
                final_ret=final_ret, final_lag=lag)


# -------------------------------------------------------------- batched surface

class Context:
    """``audiosync_cuda_ctx``: devices, streams, plans and workspaces."""

    def __init__(self, devices: Optional[Sequence[int]] = None):
        L = lib()
        self._h = C.c_void_p()
        if devices is None:
            rc = L.audiosync_cuda_create(C.byref(self._h), None, 0)
        else:
            arr = (C.c_int * len(devices))(*devices)
            rc = L.audiosync_cuda_create(C.byref(self._h), arr, len(devices))
        if rc != 0:
            self._h = C.c_void_p()
            raise AudiosyncCudaError("audiosync_cuda_create failed: " + last_error())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().audiosync_cuda_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def handle(self):
        return self._h

    def _check(self, rc: int, what: str):
        if rc != 0:
            raise AudiosyncCudaError(f"{what} failed: {last_error()}")

    def device_count(self) -> int:
        return lib().audiosync_cuda_device_count(self._h)

    def set_path(self, path: int):
        self._check(lib().audiosync_cuda_set_path(self._h, path), "set_path")

    def set_precise(self, on: bool):
        """fp64 arithmetic in the transforms (validation mode; see include/audiosync_cuda.h)."""
        self._check(lib().audiosync_cuda_set_precise(self._h, 1 if on else 0), "set_precise")

    def set_weighting(self, mode: int):
        """Cross-spectrum weighting of this context's batch calls: WEIGHT_NONE (the plain correlation)
        or WEIGHT_PHAT (GCC-PHAT, the whitened cross-spectrum; see include/audiosync_cuda.h)."""
        self._check(lib().audiosync_cuda_set_weighting(self._h, int(mode)), "set_weighting")

    def set_lag_window(self, lo: int | None = None, hi: int | None = None):
        """Restrict this context's batch calls to the folded lags [lo, hi] (inclusive); None leaves
        that side unbounded, and set_lag_window() restores the full search (see include/audiosync_cuda.h)."""
        lo = -(1 << 63) if lo is None else int(lo)
        hi = (1 << 63) - 1 if hi is None else int(hi)
        self._check(lib().audiosync_cuda_set_lag_window(self._h, lo, hi), "set_lag_window")

    def set_host_narrowing(self, mode: int):
        """f64 HOST batches converted to fp32 on the host while staged (half the PCIe bytes):
        NARROW_OFF, NARROW_LOSSLESS (default: only where exact, results bit-identical) or NARROW_ALWAYS."""
        self._check(lib().audiosync_cuda_set_host_narrowing(self._h, int(mode)), "set_host_narrowing")

    def set_wave_pairs(self, pairs: int):
        self._check(lib().audiosync_cuda_set_wave_pairs(self._h, pairs), "set_wave_pairs")

    def describe_plan(self, sample_len: int) -> str:
        buf = C.create_string_buffer(512)
        n = lib().audiosync_cuda_describe_plan(self._h, sample_len, buf, 512)
        if n < 0:
            raise AudiosyncCudaError("describe_plan failed: " + last_error())
        return buf.value.decode()

    def host_feed_stats(self, reset: bool = False):
        """(pairs that crossed the link as doubles, pairs narrowed to fp32 on the host) of F64 host batches."""
        out = (C.c_uint64 * 2)()
        self._check(lib().audiosync_cuda_host_feed_stats(self._h, out, 1 if reset else 0), "host_feed_stats")
        return int(out[0]), int(out[1])

    def launch_count(self) -> int:
        return int(lib().audiosync_cuda_launch_count(self._h))

    def synchronize(self, device: int = 0):
        self._check(lib().audiosync_cuda_synchronize(self._h, device), "synchronize")

    # -- host-facing batch call ------------------------------------------------
    def xcorr_batch(self, sources: np.ndarray, samples: np.ndarray):
        """sources [n][2L], samples [n][L], float32, float64 or int16 (16-bit PCM, S16) host arrays.

        Returns a dict of numpy arrays: lags (int64), coefs, rets (int32), peaks.
        """
        if sources.dtype != samples.dtype or sources.dtype not in _NP_DTYPES:
            raise TypeError("sources/samples must both be float32, float64 or int16")
        sources = np.ascontiguousarray(sources)
        samples = np.ascontiguousarray(samples)
        if sources.ndim != 2 or samples.ndim != 2 or sources.shape[0] != samples.shape[0] \
                or sources.shape[1] != 2 * samples.shape[1]:
            raise ValueError("expected sources [n][2L] and samples [n][L]")
        n, L = samples.shape
        lags = np.zeros(n, np.int64); coefs = np.zeros(n, np.float64)
        rets = np.zeros(n, np.int32); peaks = np.zeros(n, np.float64)
        dt = _NP_DTYPES[sources.dtype]
        rc = lib().audiosync_cuda_xcorr_batch(self._h, sources.ctypes.data, samples.ctypes.data, n, L,
                                              dt, HOST, lags.ctypes.data, coefs.ctypes.data,
                                              rets.ctypes.data, peaks.ctypes.data)
        self._check(rc, "xcorr_batch")
        return dict(lags=lags, coefs=coefs, rets=rets, peaks=peaks)

    def xcorr_batch_ptr(self, sources_ptr: int, samples_ptr: int, n_pairs: int, sample_len: int,
                        dtype: int, memspace: int):
        """Same call on raw pointers (pinned host buffers or device memory); dtype F32, F64 or S16."""
        lags = np.zeros(n_pairs, np.int64); coefs = np.zeros(n_pairs, np.float64)
        rets = np.zeros(n_pairs, np.int32); peaks = np.zeros(n_pairs, np.float64)
        rc = lib().audiosync_cuda_xcorr_batch(self._h, sources_ptr, samples_ptr, n_pairs, sample_len,
                                              dtype, memspace, lags.ctypes.data, coefs.ctypes.data,
                                              rets.ctypes.data, peaks.ctypes.data)
        self._check(rc, "xcorr_batch")
        return dict(lags=lags, coefs=coefs, rets=rets, peaks=peaks)

    def xcorr_batch_records(self, sources_ptr: int, samples_ptr: int, n_pairs: int, sample_len: int,
                            dtype: int, memspace: int) -> np.ndarray:
        """Whole result records (``RESULT_DTYPE``: lag, coef, peak, ret, success, raw_index, second, margin, ncc);
        dtype F32, F64 or S16."""
        res = np.zeros(n_pairs, RESULT_DTYPE)
        rc = lib().audiosync_cuda_xcorr_batch_results(self._h, sources_ptr, samples_ptr, n_pairs, sample_len,
                                                      dtype, memspace, res.ctypes.data)
        self._check(rc, "xcorr_batch_results")
        return res

    def xcorr_shared_source(self, source: np.ndarray, samples: np.ndarray) -> np.ndarray:
        """One source against many samples: ``source`` 1-D with at least 2L elements (only [0, 2L) is
        read), ``samples`` [n][L], both float32, float64 or int16 (S16) host arrays.  Record i is, bit
        for bit, the ``xcorr_batch_records`` record of (source, samples[i]) with the source replicated
        (see include/audiosync_cuda.h); the source is uploaded and transformed once per device."""
        if source.dtype != samples.dtype or source.dtype not in _NP_DTYPES:
            raise TypeError("source/samples must both be float32, float64 or int16")
        if source.ndim != 1 or samples.ndim != 2 or source.shape[0] < 2 * samples.shape[1]:
            raise ValueError("expected source [>= 2L] and samples [n][L]")
        n, L = samples.shape
        source = np.ascontiguousarray(source[: 2 * L])
        samples = np.ascontiguousarray(samples)
        res = np.zeros(n, RESULT_DTYPE)
        rc = lib().audiosync_cuda_xcorr_shared_source(self._h, source.ctypes.data, samples.ctypes.data, n, L,
                                                      _NP_DTYPES[source.dtype], HOST, res.ctypes.data)
        self._check(rc, "xcorr_shared_source")
        return res

    def xcorr_shared_source_torch(self, source, samples, out=None, sync: bool = True):
        """``xcorr_shared_source`` on torch CUDA tensors, zero copy: ``source`` 1-D (at least 2L
        elements, [0, 2L) is read) and ``samples`` [n, L] of one dtype on one device of this context,
        enqueued on torch's current stream; ``out`` and ``sync`` as in ``xcorr_batch_torch``."""
        import torch
        if not (source.is_cuda and samples.is_cuda) or source.device != samples.device:
            raise ValueError("source and samples must be CUDA tensors on the same device")
        dts = {torch.float32: F32, torch.float64: F64, torch.int16: S16}
        if source.dtype != samples.dtype or source.dtype not in dts:
            raise TypeError("source/samples must both be float32, float64 or int16")
        if source.dim() != 1 or samples.dim() != 2 or source.shape[0] < 2 * samples.shape[1]:
            raise ValueError("expected source [>= 2L] and samples [n, L]")
        if not (source.is_contiguous() and samples.is_contiguous()):
            raise ValueError("tensors must be contiguous (no hidden copies on this path)")
        n, L = samples.shape
        dev = source.device
        if out is None:
            out = torch.empty(n * RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        elif out.device != dev or out.dtype != torch.uint8 or out.numel() < n * RESULT_DTYPE.itemsize:
            raise ValueError("out must be a uint8 tensor of n * 64 bytes on the same device")
        stream = torch.cuda.current_stream(dev).cuda_stream
        if stream == 0:
            # as in xcorr_batch_torch: a NULL handle selects the library's own stream
            torch.cuda.current_stream(dev).synchronize()
        if n:
            self.xcorr_shared_source_device(dev.index, source.data_ptr(), samples.data_ptr(), n, L, dts[source.dtype],
                                            out.data_ptr(), stream)
        if stream == 0:
            self.synchronize(dev.index)
        if not sync:
            return out
        return out[: n * RESULT_DTYPE.itemsize].cpu().numpy().view(RESULT_DTYPE)

    def xcorr_batch_torch(self, sources, samples, out=None, sync: bool = True):
        """Zero-copy batch call on torch CUDA tensors (SURVEY 8f rank 3).

        ``sources`` [n, 2L] and ``samples`` [n, L]: contiguous float32, float64 or int16 (S16) tensors on one
        device of this context.  The kernels are enqueued on torch's CURRENT stream of that
        device, reading the tensors in place; the 48-byte records land in ``out`` (a uint8
        CUDA tensor of n * 64 bytes, allocated when omitted).  With ``sync`` the records come
        back as a NumPy structured array (``RESULT_DTYPE``); otherwise the device tensor is
        returned and the caller orders later work on the same stream.
        """
        import torch
        if not (sources.is_cuda and samples.is_cuda) or sources.device != samples.device:
            raise ValueError("sources and samples must be CUDA tensors on the same device")
        dts = {torch.float32: F32, torch.float64: F64, torch.int16: S16}
        if sources.dtype != samples.dtype or sources.dtype not in dts:
            raise TypeError("sources/samples must both be float32, float64 or int16")
        if sources.dim() != 2 or samples.dim() != 2 or sources.shape[0] != samples.shape[0] \
                or sources.shape[1] != 2 * samples.shape[1]:
            raise ValueError("expected sources [n, 2L] and samples [n, L]")
        if not (sources.is_contiguous() and samples.is_contiguous()):
            raise ValueError("tensors must be contiguous (no hidden copies on this path)")
        n, L = samples.shape
        dev = sources.device
        if out is None:
            out = torch.empty(n * RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        elif out.device != dev or out.dtype != torch.uint8 or out.numel() < n * RESULT_DTYPE.itemsize:
            raise ValueError("out must be a uint8 tensor of n * 64 bytes on the same device")
        stream = torch.cuda.current_stream(dev).cuda_stream
        if stream == 0:
            # a NULL handle would select the library's own stream: order it after torch's default
            # stream by draining that one first, and synchronise the device afterwards
            torch.cuda.current_stream(dev).synchronize()
        dt = dts[sources.dtype]
        if n:
            self.xcorr_batch_device(dev.index, sources.data_ptr(), samples.data_ptr(), n, L, dt,
                                    out.data_ptr(), stream)
        if stream == 0:
            self.synchronize(dev.index)
        if not sync:
            return out
        return out[: n * RESULT_DTYPE.itemsize].cpu().numpy().view(RESULT_DTYPE)

    # -- stream-ordered device calls --------------------------------------------
    def xcorr_batch_device(self, device: int, d_sources: int, d_samples: int, n_pairs: int,
                           sample_len: int, dtype: int, d_results: int, stream: int = 0):
        """Stream-ordered call on device pointers; dtype F32, F64 or S16."""
        rc = lib().audiosync_cuda_xcorr_batch_device(self._h, device, d_sources, d_samples, n_pairs,
                                                     sample_len, dtype, d_results, stream or None)
        self._check(rc, "xcorr_batch_device")

    def xcorr_shared_source_device(self, device: int, d_source: int, d_samples: int, n_pairs: int,
                                   sample_len: int, dtype: int, d_results: int, stream: int = 0):
        """Stream-ordered shared-source call on device pointers; dtype F32, F64 or S16."""
        rc = lib().audiosync_cuda_xcorr_shared_source_device(self._h, device, d_source, d_samples, n_pairs,
                                                             sample_len, dtype, d_results, stream or None)
        self._check(rc, "xcorr_shared_source_device")

    def synth_pairs(self, device: int, seed: int, first_pair: int, n_pairs: int, sample_len: int,
                    dtype: int, d_sources: int, d_samples: int, stream: int = 0):
        """Seeded synthetic pairs in device memory; dtype F32 or F64 (S16 is refused)."""
        rc = lib().audiosync_cuda_synth_pairs(self._h, device, seed, first_pair, n_pairs, sample_len,
                                              dtype, d_sources, d_samples, stream or None)
        self._check(rc, "synth_pairs")

    # -- per-kernel device timing -----------------------------------------------
    def profile_enable(self, on: bool = True):
        self._check(lib().audiosync_cuda_profile_enable(self._h, int(on)), "profile_enable")

    def profile_reset(self):
        self._check(lib().audiosync_cuda_profile_reset(self._h), "profile_reset")

    def profile_read(self):
        """{kernel class name: (launches, total device ms)} since the last reset."""
        out = {}
        name = C.create_string_buffer(64)
        n = C.c_uint64(); ms = C.c_double()
        count = lib().audiosync_cuda_profile_read(self._h, 0, name, 64, C.byref(n), C.byref(ms))
        if count < 0:
            raise AudiosyncCudaError("profile_read failed: " + last_error())
        for i in range(count):
            lib().audiosync_cuda_profile_read(self._h, i, name, 64, C.byref(n), C.byref(ms))
            out[name.value.decode()] = (int(n.value), float(ms.value))
        return out


class SessionPool:
    """``audiosync_cuda_pool``: many concurrent sessions with device-resident, growing buffers.

    Frames are appended as they arrive (host doubles, the reference's f64le wire format); when a
    range of slots has reached an interval of the schedule, ``run`` evaluates that interval for all
    of them as one batch and returns the ``RESULT_DTYPE`` records.
    """

    def __init__(self, ctx: "Context", device: int, n_slots: int, max_sample_len: int, dtype: int = F64):
        self._ctx = ctx                       # keeps the context alive
        self._h = C.c_void_p()
        self.n_slots, self.max_sample_len, self.dtype = n_slots, max_sample_len, dtype
        rc = lib().audiosync_cuda_pool_create(ctx._h, device, n_slots, max_sample_len, dtype, C.byref(self._h))
        if rc != 0:
            self._h = C.c_void_p()
            raise AudiosyncCudaError("pool_create failed: " + last_error())

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().audiosync_cuda_pool_destroy(self._h)
            self._h = C.c_void_p()

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset(self, slot: int):
        if lib().audiosync_cuda_pool_reset(self._h, slot) != 0:
            raise AudiosyncCudaError("pool_reset failed: " + last_error())

    def append(self, slot: int, source_frames=None, sample_frames=None):
        s = np.ascontiguousarray(source_frames if source_frames is not None else [], np.float64)
        m = np.ascontiguousarray(sample_frames if sample_frames is not None else [], np.float64)
        rc = lib().audiosync_cuda_pool_append(self._h, slot, s.ctypes.data if s.size else None, s.size,
                                              m.ctypes.data if m.size else None, m.size)
        if rc != 0:
            raise AudiosyncCudaError("pool_append failed: " + last_error())

    def append_ptr(self, slot: int, source_ptr: int, n_source: int, sample_ptr: int, n_sample: int, sync: bool = False):
        """Stream-ordered append from raw host addresses (e.g. ``RealBuffer``): returns once the copies
        are enqueued unless ``sync``; ``run`` / ``flush`` order themselves behind it."""
        fn = lib().audiosync_cuda_pool_append if sync else lib().audiosync_cuda_pool_append_async
        if fn(self._h, slot, source_ptr or None, n_source, sample_ptr or None, n_sample) != 0:
            raise AudiosyncCudaError("pool_append failed: " + last_error())

    def flush(self):
        if lib().audiosync_cuda_pool_flush(self._h) != 0:
            raise AudiosyncCudaError("pool_flush failed: " + last_error())

    def fill(self, slot: int):
        a, b = C.c_size_t(), C.c_size_t()
        if lib().audiosync_cuda_pool_fill(self._h, slot, C.byref(a), C.byref(b)) != 0:
            raise AudiosyncCudaError("pool_fill: bad slot")
        return int(a.value), int(b.value)

    def run(self, first_slot: int, n_slots: int, sample_len: int) -> np.ndarray:
        res = np.zeros(n_slots, RESULT_DTYPE)
        rc = lib().audiosync_cuda_pool_run(self._h, first_slot, n_slots, sample_len, res.ctypes.data)
        if rc != 0:
            raise AudiosyncCudaError("pool_run failed: " + last_error())
        return res
