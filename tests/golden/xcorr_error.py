"""Per-lag error of the correlation r against an fp64 or exact reference -- TEST INFRASTRUCTURE.

The records show r only at its peak, so the parity tests bound r there.  This module judges r[j] at
any lag j, read through the lag window and source rotations (tests/test_xcorr_error_*.py):

  - reference(): fp64 r (numpy) of the values the kernel reads: the fp32-rounded values for F32 inputs,
    the doubles for F64, s / 32768 for S16; under GCC-PHAT phat_oracle.phat_correlation's r_w.  Good
    enough to judge fp32 arithmetic, whose error is 1e8 times larger.
  - exact_reference(): r of integer inputs (times 2^-15) exactly, for the fp64 paths (precise mode,
    PATH_DIRECT), whose error is of the same order as a numpy fp64 FFT's.  Each input is split into
    8-bit limbs, each limb pair correlated by a float64 FFT and rounded to integers (the rounding
    distance is checked) and the integer correlations recombined.
  - yardstick(): the same correlation by scipy.fft in float32 (rfft, complex64 product, irfft): the
    error a plain fp32 transform makes on the same input.

Bound.  With u = 2^-24 (fp32 arithmetic) or 2^-53 (fp64), N = 2L, rho = rms(r) over all 2L lags and
R = max|r|, every lag read must satisfy

    |r_kernel[j] - r[j]| <= A u log2(N) rho + B u R

and the rms of the error over the lags read  <= C u sqrt(log2 N) rho + B u R.

The B term is there because the error is not white on a pair with a tall peak: the value at the
peak itself carries about u |peak| of rounding, and coherent errors of the same order sit at fixed
offsets from the peak on the four-step plans.  A bound on rho alone would fail correct kernels there.

GCC-PHAT in fp32 on a spectrum of wide dynamic range (DC offset, brown noise) is ill-conditioned:
the phase of a weak bin carries the rounding of the strong ones, and PHAT lifts every bin to unit
magnitude.  There the kernel's error reaches 1000 u log2(N) rho, and so does a plain float32 FFT's
(the kernel stays within 1.5 times the yardstick's rms), so fp32 PHAT may also err by PHAT_D times
the yardstick's rms error over the same lags (PHAT_DR for the rms bound).

Constants: about twice the largest value measured on a B200 over every plan, input family, dtype
and weighting of tests/test_xcorr_error_gpu.py (MEASURED below; the emulator's host arithmetic
lands inside the same bound).  A wrong bin moves every r[j] by about |X_k Y_k| ~ rho / sqrt(N),
over 1000 times the bound at N = 2.88M, and the sensitivity test of tests/test_xcorr_error_emu.py
shows a single corrupted table entry fails the bound while the record checks still pass.
"""
from __future__ import annotations

import math
import os
import sys
from dataclasses import dataclass

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(_HERE))
for _p in (ROOT, _HERE):
    if _p not in sys.path:
        sys.path.insert(0, _p)
from oracle import xcorr_numpy as xn  # noqa: E402
import phat_oracle as po  # noqa: E402
from probes import Plan, STATIC_PLANS, parse_plan, single_cta_plan  # noqa: E402,F401

U32 = 2.0 ** -24
U64 = 2.0 ** -53

# (A, B, C) of the bound, and the yardstick multiples of fp32 PHAT; see MEASURED
BOUND_F32 = (3.0, 4.5, 3.0)
BOUND_F64 = (3.0, 3.5, 3.0)
PHAT_D, PHAT_DR = 12.0, 3.0

# Measured on one NVIDIA B200 (power limit 1000 W) over the 125 fp32 and 9 fp64 cases of
# tests/test_xcorr_error_gpu.py (512 slots x 64 rotations per case above 24,000 frames, every lag at
# and below).  a_flat, c_flat: max|e| / (u log2 N rho) and rms(e) / (u sqrt(log2 N) rho) on white, DC
# and brown noise; B_needed: the least B that holds every case with A = C = 3 (the PHAT cases with
# the yardstick term); peak_b: max|e| / (u R) where the error is largest at the peak itself;
# yard_max / yard_rms: kernel over float32 yardstick error, max and rms over the lags read, largest
# over the plan's cases.
MEASURED = {
    "f32": dict(a_flat=1.52, c_flat=1.34, B_needed=2.14,
                phat_ill_conditioned=dict(emax_over_yard_rms=5.8, rms_over_yard_rms=1.41)),
    "f64": dict(a_flat=1.25, c_flat=1.14, peak_b=1.06, phat_b=1.67),
    "yard_max/yard_rms": {
        "static-144000": (1.44, 1.41), "static-288000": (1.34, 1.18), "static-480000": (1.29, 1.42),
        "static-720000": (3.60, 1.52), "static-960000": (1.97, 1.36), "static-1440000": (4.93, 2.53),
        "single_cta-4096": (1.43, 1.21), "single_cta-6000": (2.15, 0.93),
        "radix-24000": (1.50, 1.01), "radix-9600 (64-thread CTAs)": (1.20, 1.06), "radix-48000": (1.24, 0.94),
        "radix-192000": (1.02, 1.01), "radix-100001": (0.61, 0.55), "radix-1440002": (0.64, 0.59),
        "radix-1000000": (1.30, 1.03),
    },
}

S16_SCALE = 1.0 / 32768.0


# ----------------------------------------------------------------------------- references
def reference(src: np.ndarray, smp: np.ndarray, phat: bool = False) -> np.ndarray:
    """fp64 r[0 .. 2L) (scaled by N like FFTW's unnormalised c2r) of the given values."""
    src = np.asarray(src, np.float64)
    smp = np.asarray(smp, np.float64)
    return po.phat_correlation(src, smp) if phat else xn.correlation(src, smp)


def _limbs(v: np.ndarray):
    """v = hi * 256 + lo, lo in [0, 256), hi in [-128, 128) for int16-range integers."""
    v = np.asarray(v, np.int64)
    assert v.min() >= -32768 and v.max() <= 32767
    lo = v & 255
    return ((v - lo) >> 8, lo)


def exact_correlation(src_int: np.ndarray, smp_int: np.ndarray) -> np.ndarray:
    """Exact integer correlation R[j] = sum_m src[(m + j) mod 2L] smp[m] (int64) of int16-range inputs."""
    L = smp_int.shape[0]
    N = 2 * L
    out = np.zeros(N, np.int64)
    fa = [np.fft.rfft(x.astype(np.float64)) for x in _limbs(src_int[:N])]
    fb = []
    for y in _limbs(smp_int):
        p = np.zeros(N)
        p[:L] = y
        fb.append(np.conj(np.fft.rfft(p)))
    for i, (wa, a) in enumerate(zip((256, 1), fa)):
        for k, (wb, b) in enumerate(zip((256, 1), fb)):
            r = np.fft.irfft(a * b, n=N)
            R = np.rint(r)
            d = float(np.max(np.abs(r - R)))
            assert d < 0.05, "limb correlation too far from integers to round (%g)" % d
            out += wa * wb * R.astype(np.int64)
    return out


def exact_reference(src_int: np.ndarray, smp_int: np.ndarray, scale: float = S16_SCALE) -> np.ndarray:
    """r of the values src_int * scale, smp_int * scale, exact up to its one final fp64 rounding."""
    N = 2 * smp_int.shape[0]
    return exact_correlation(src_int, smp_int).astype(np.float64) * (float(N) * scale * scale)


def yardstick(src: np.ndarray, smp: np.ndarray, phat: bool = False) -> np.ndarray:
    """r by scipy.fft in float32 throughout (float64 result of the float32 values)."""
    import scipy.fft as sf
    L = smp.shape[0]
    N = 2 * L
    pad = np.zeros(N, np.float32)
    pad[:L] = np.asarray(smp, np.float32)
    fa = sf.rfft(np.asarray(src[:N], np.float32))
    fb = sf.rfft(pad)
    w = fa * np.conj(fb)
    if phat:
        ma, mb = np.abs(fa), np.abs(fb)
        ok = (ma > 0) & (mb > 0)
        w = np.where(ok, w / np.where(ok, ma * mb, np.float32(1)), np.complex64(0)).astype(np.complex64)
    return sf.irfft(w, n=N).astype(np.float64) * N


# ----------------------------------------------------------------------------- input families
@dataclass
class Pair:
    """One base pair: float64 values the kernel reads (fp32-exact unless the family says otherwise),
    and for integer families the int16-range integers (values = ints * 2^-15)."""
    family: str
    src: np.ndarray
    smp: np.ndarray
    src_int: np.ndarray | None = None
    smp_int: np.ndarray | None = None
    lag: int = -1                 # designed peak lag (delayed families), else -1

    @property
    def L(self):
        return self.smp.shape[0]


FAMILIES = ("white", "delayed", "dc", "brown", "transient", "silent_half", "s16", "f64")
INT_FAMILIES = ("s16", "s16_white")


def _f32(x):
    return np.asarray(x, np.float64).astype(np.float32).astype(np.float64)


def _quantise(x, peak=32767):
    """int16-range integers of x at full scale."""
    return np.clip(np.rint(x / np.max(np.abs(x)) * peak), -32768, 32767).astype(np.int64)


def make_pair(family: str, L: int, seed: int) -> Pair:
    rng = np.random.default_rng([seed, L, FAMILIES.index(family) if family in FAMILIES else 99])
    N = 2 * L
    lag = int(rng.integers(0, L))
    if family == "white":
        return Pair(family, _f32(rng.standard_normal(N)), _f32(rng.standard_normal(L)))
    if family == "delayed":
        src = rng.standard_normal(N)
        return Pair(family, _f32(src), _f32(src[lag:lag + L] + 0.3 * rng.standard_normal(L)), lag=lag)
    if family == "dc":
        src = 10.0 + rng.standard_normal(N)
        return Pair(family, _f32(src), _f32(10.0 + rng.standard_normal(L)))
    if family == "brown":
        src = np.cumsum(rng.standard_normal(N))
        smp = np.cumsum(rng.standard_normal(L))
        return Pair(family, _f32(src / np.std(src)), _f32(smp / np.std(smp)))
    if family == "transient":
        # a burst 1e4 times the floor in the source, copied into the sample: the floor is 1e-4
        src = 1e-4 * rng.standard_normal(N)
        lag = int(rng.integers(0, L // 2))
        at = lag + int(rng.integers(0, L // 2))
        n = max(16, L // 100)
        src[at:at + n] += rng.standard_normal(n)
        return Pair(family, _f32(src), _f32(src[lag:lag + L] + 1e-4 * rng.standard_normal(L)), lag=lag)
    if family == "silent_half":
        src = rng.standard_normal(N)
        src[L:] = 0.0
        return Pair(family, _f32(src), _f32(src[lag:lag + L] + 0.3 * rng.standard_normal(L)), lag=lag)
    if family == "s16":
        # full-scale quantised delayed pair: values s / 32768
        x = rng.integers(-32768, 32768, N)
        y = np.clip((x[lag:lag + L] * 3) // 4 + rng.integers(-6000, 6001, L), -32768, 32767)
        return Pair(family, x * S16_SCALE, y * S16_SCALE, x, y, lag=lag)
    if family == "s16_white":
        x = rng.integers(-32768, 32768, N)
        y = rng.integers(-32768, 32768, L)
        return Pair(family, x * S16_SCALE, y * S16_SCALE, x, y)
    if family == "f64":
        # doubles that fp32 cannot hold: the F64 call must read them as given
        src = rng.standard_normal(N)
        return Pair(family, src, src[lag:lag + L] + 0.3 * rng.standard_normal(L), lag=lag)
    raise ValueError(family)


def quantised(p: Pair) -> Pair:
    """The integer (S16-valued) version of a pair, for the exact reference."""
    if p.src_int is not None:
        return p
    x, y = _quantise(p.src), _quantise(p.smp)
    return Pair(p.family + "_q", x * S16_SCALE, y * S16_SCALE, x, y, lag=p.lag)


def fp32_exact(p: Pair) -> bool:
    return bool(np.array_equal(_f32(p.src), p.src) and np.array_equal(_f32(p.smp), p.smp))


# ----------------------------------------------------------------------------- slots and lags
def fold_slots(L: int) -> list:
    """Raw slots at the edges of the fold: 0, 1, L-1, L, L+1, 2L-1."""
    return [0, 1, L - 1, L, L + 1, 2 * L - 1]


def layout_slots(plan: Plan) -> list:
    """First and last output positions of the four-step layout: rows 0, 1, M1/2, M1-1 crossed with
    the first and last column of the first, second and last column tile, both points of a packed
    pair (output j = 2 (n1 M2 + n2) + odd); for the single-CTA plan (M1 = 1) its positions."""
    L, M1, M2, ct = plan.L, plan.M1, plan.M2, max(plan.ct, 1)
    ntiles = (M2 + ct - 1) // ct
    cols = {0, ct - 1, ct, 2 * ct - 1, (ntiles - 1) * ct, M2 - 1, M2 // 2}
    rows = {0, 1, M1 // 2, M1 - 1} if M1 > 1 else {0}
    out = set()
    for n1 in rows:
        for n2 in cols:
            if 0 <= n2 < M2:
                for odd in (0, 1):
                    j = 2 * (n1 * M2 + n2) + odd
                    if j < 2 * L:
                        out.add(j)
    return sorted(out)


def slots(plan: Plan, n: int, seed: int) -> list:
    """Fold edges, layout positions, then seeded random slots up to n in all (or every slot when
    n >= 2L)."""
    N = 2 * plan.L
    if n >= N:
        return list(range(N))
    base = list(dict.fromkeys(fold_slots(plan.L) + layout_slots(plan)))
    rng = np.random.default_rng([seed, plan.L, 7])
    have = set(base)
    while len(base) < n:
        k = int(rng.integers(0, N))
        if k not in have:
            have.add(k)
            base.append(k)
    return base


def structured_lags(peak: int, L: int) -> list:
    """+-64 around the peak, and the peak's offsets by multiples of 2L/12 (with their neighbours)."""
    N = 2 * L
    out = [(peak + d) % N for d in range(-64, 65)]
    for m in range(1, 12):
        c = peak + round(m * N / 12)
        out += [(c + d) % N for d in (-1, 0, 1)]
    return list(dict.fromkeys(out))


def assign_lags(slot_list: list, per_slot: int, L: int, peak: int, seed: int, every: bool = False):
    """{slot: lags} with per_slot lags for each slot: the structured lags spread over the slots first,
    then seeded random lags.  every: each lag of [0, 2L) read at least once (slot k always reads k
    itself, the rest in order)."""
    N = 2 * L
    rng = np.random.default_rng([seed, L, 11])
    todo = structured_lags(peak, L)
    if every:
        todo = list(range(N))
    out = {}
    it = 0
    for k in slot_list:
        lags = [k] if every else []
        while len(lags) < per_slot:
            if it < len(todo):
                lags.append(todo[it])
                it += 1
            else:
                lags.append(int(rng.integers(0, N)))
        out[k] = lags
    assert it >= len(todo) or not every, "too few readings to cover every lag"
    return out


# ----------------------------------------------------------------------------- the bound
def bound(N: int, rho: float, rmax: float, fp64: bool = False) -> float:
    a, b, _ = BOUND_F64 if fp64 else BOUND_F32
    u = U64 if fp64 else U32
    return a * u * math.log2(N) * rho + b * u * rmax


def rms_bound(N: int, rho: float, rmax: float, fp64: bool = False) -> float:
    _, b, c = BOUND_F64 if fp64 else BOUND_F32
    u = U64 if fp64 else U32
    return c * u * math.sqrt(math.log2(N)) * rho + b * u * rmax


def judge(lags, got, r: np.ndarray, fp64: bool = False, yard: np.ndarray | None = None, phat: bool = False) -> dict:
    """Errors of the kernel values `got` at `lags` against the reference r (all 2L lags).  Returns the
    measured ratios, ok (both bounds hold) and a message naming the worst lag.  phat: r is the
    GCC-PHAT r_w, and an fp32 kernel may also err by PHAT_D (PHAT_DR for the rms) times the rms error
    of the float32 yardstick `yard` over the same lags."""
    lags = np.asarray(lags, np.int64)
    got = np.asarray(got, np.float64)
    N = r.shape[0]
    rho = float(np.sqrt(np.mean(r * r)))
    rmax = float(np.max(np.abs(r)))
    u = U64 if fp64 else U32
    e = np.abs(got - r[lags])
    e = np.where(np.isnan(e), np.inf, e)
    emax = float(e.max()) if e.size else 0.0
    erms = float(np.sqrt(np.mean(e * e))) if e.size else 0.0
    worst = int(lags[int(np.argmax(e))]) if e.size else -1
    peak = xn.max_abs_index(r)
    out = dict(N=N, n=int(e.size), rho=rho, rmax=rmax, emax=emax, erms=erms, worst_lag=worst,
               worst_offset=int((worst - peak) % N),
               a=emax / (u * math.log2(N) * rho), b=emax / (u * rmax),
               c=erms / (u * math.sqrt(math.log2(N)) * rho))
    if yard is not None:
        ey = np.abs(yard[lags] - r[lags])
        out["yard_max"] = emax / max(float(ey.max()), 1e-300)
        out["yard_rms"] = erms / max(float(np.sqrt(np.mean(ey * ey))), 1e-300)
    lim, lim_rms = bound(N, rho, rmax, fp64), rms_bound(N, rho, rmax, fp64)
    if phat and not fp64:
        # fp32 GCC-PHAT: the yardstick's own rms error over the same lags sets the conditioning
        assert yard is not None, "fp32 PHAT is judged against the float32 yardstick"
        yerms = float(np.sqrt(np.mean(ey * ey)))
        lim += PHAT_D * yerms
        lim_rms += PHAT_DR * yerms
    out["ok"] = bool(emax <= lim and erms <= lim_rms)
    out["msg"] = ("max err %.3e at lag %d (peak %+d) vs bound %.3e; rms %.3e vs %.3e; rho %.4g, max|r| %.4g"
                  % (emax, worst, out["worst_offset"], lim, erms, lim_rms, rho, rmax))
    return out
