"""NumPy (pocketfft, fp64) restatement of the PHAT-weighted record -- TEST INFRASTRUCTURE.

GCC-PHAT as include/audiosync_cuda.h defines it (audiosync_cuda_set_weighting): with N = 2L,
X = DFT_N(source[0, 2L)) and Y = DFT_N(zero-padded sample),
    W[k]   = X[k] conj(Y[k]) / (|X[k]| |Y[k]|)      (0 where |X[k]|^2 or |Y[k]|^2 is 0)
    r_w[j] = sum_k W[k] e^(2 pi i j k / N)           (irfft * N: unnormalised like FFTW's c2r)
raw_index = max_abs_index(r_w), the reference's fold, Pearson of the aligned windows of the original
inputs, and ncc = peak / N.  Everything but the weighting is oracle/xcorr_numpy.py's.

Also the two input models the tests use: delayed white noise, and AR(1)-coloured noise through a
random decaying room response with additive noise (the reverberant case GCC-PHAT exists for).
"""
from __future__ import annotations

import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle import xcorr_numpy as xn  # noqa: E402


def phat_correlation(source: np.ndarray, sample: np.ndarray) -> np.ndarray:
    """r_w[0 .. 2L), fp64."""
    source = np.asarray(source, np.float64)
    sample = np.asarray(sample, np.float64)
    L = sample.shape[0]
    N = 2 * L
    padded = np.zeros(N, np.float64)
    padded[:L] = sample
    fa = np.fft.rfft(source[:N])
    fb = np.fft.rfft(padded)
    ma, mb = np.abs(fa), np.abs(fb)
    ok = (ma * ma > 0) & (mb * mb > 0)
    w = np.zeros_like(fa)
    w[ok] = fa[ok] * np.conj(fb[ok]) / (ma[ok] * mb[ok])
    return np.fft.irfft(w, n=N) * N


def phat_record(source: np.ndarray, sample: np.ndarray) -> dict:
    """dict(ret, lag, coef, raw_index, peak, second, margin, ncc) of the PHAT-weighted call."""
    source = np.asarray(source, np.float64)
    sample = np.asarray(sample, np.float64)
    L = sample.shape[0]
    N = 2 * L
    r = phat_correlation(source, sample)
    idx = xn.max_abs_index(r)
    mag = np.abs(r).copy()
    mag[idx] = -1.0
    second = float(np.nanmax(mag))
    lag, wx, wy = xn.windows(source, sample, idx)
    coef = xn.pearson(wx, wy)
    peak = float(r[idx])
    ap = abs(peak)
    margin = (ap - second) / ap if ap > 0 else (0.0 if ap == 0 else float("nan"))
    return dict(ret=-1 if coef != coef else 0, lag=int(lag), coef=coef, raw_index=idx, peak=peak,
                second=second, margin=float(margin), ncc=peak / N)


def noise_pair(L: int, seed: int, lag: int | None = None, noise: float = 0.3):
    """White-noise source [2L]; the sample is source[lag:lag + L] plus `noise` white noise."""
    rng = np.random.default_rng(seed)
    lag = int(rng.integers(0, L)) if lag is None else int(lag)
    src = rng.standard_normal(2 * L)
    smp = src[lag:lag + L] + noise * rng.standard_normal(L)
    return src, smp, lag


def coloured_pair(L: int, seed: int, lag: int | None = None, pole: float = 0.995, taps: int = 2400,
                  noise: float = 0.3):
    """AR(1)-coloured source [2L] (pole 0.995: music-like low-frequency weight); the sample is the
    source from `lag` on, through a random decaying `taps`-tap room response (direct path 1,
    reflections of 0.2 RMS decaying over taps / 6), plus `noise` (relative RMS) white noise."""
    from scipy.signal import fftconvolve, lfilter
    rng = np.random.default_rng(seed)
    lag = int(rng.integers(taps, L)) if lag is None else int(lag)
    src = lfilter([1.0], [1.0, -pole], rng.standard_normal(2 * L))
    h = 0.2 * rng.standard_normal(taps) * np.exp(-np.arange(taps) / (taps / 6.0))
    h[0] = 1.0                                       # the direct path, then the reflections
    wet = fftconvolve(src, h)[:2 * L]
    smp = wet[lag:lag + L]
    smp = smp + noise * np.std(smp) * rng.standard_normal(L)
    return src, smp, lag


def shift_probe(L: int, a: int, seed: int, sign: float = 1.0):
    """Closed-form probe: source = sign * circular roll by a of the zero-padded sample, so that
    r_w = sign * N * delta(j - a) wherever no bin of Y is 0."""
    rng = np.random.default_rng(seed)
    smp = rng.standard_normal(L)
    padded = np.zeros(2 * L)
    padded[:L] = smp
    return sign * np.roll(padded, a), smp
