"""Pairs whose every Pearson and record sum is exact -- TEST INFRASTRUCTURE.

Every element is an integer a with 1 <= |a| <= 15 times 2^-15: exact in fp32 and fp64, and the same
integer as 16-bit PCM (S16 stands for s * 2^-15).  On such inputs every sum the Pearson step forms is
exact, on every path and in every reduction order:
  - the pivot px = (sum of 32 window values) / 32 is m * 2^-20 with |m| <= 480, exact in fp32;
  - dx = x - px = (32a - m) * 2^-20 with |32a - m| <= 960, exact in fp32;
  - dx * dy <= 960^2 * 2^-40, and a 16-term fp32 partial sum stays below 2^24 units, so both are exact;
  - the fp64 totals are integers times 2^-40 far below 2^53.
So a record's coef differs from the exact rational coefficient only by the last few fp64 operations of
the finishing step (a few 1e-16), and any path that reads the same values computes the same bits.  A
kernel that drops, repeats or shifts one window element moves coef by far more than that: the builder
checks that every such change moves the exact coefficient by at least SENSITIVITY.

Pair layout: the sample is dense random; the source holds sign * sample + noise at the positions
(m + raw) mod 2L, m < L, and dense random values elsewhere.  So r[raw] = sum_m source[(m + raw) mod 2L]
* sample[m] is the correlation's peak for any raw index, and every window the fold can produce (n = L
at raw < L, n = raw - L at raw >= L, down to n = 0) is dense.

The exact record comes from integers: the correlation R[j] (of the integer arrays) by a float64 rfft
rounded to the nearest integer (its error is far below 0.5, checked), the peak and second peak confirmed
by int64 dot products, the Pearson coefficient from integer sums in 50-digit decimal arithmetic.
"""
from __future__ import annotations

import os
import sys
from dataclasses import dataclass, field
from decimal import Decimal, getcontext

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from oracle.xcorr_numpy import MIN_CONFIDENCE  # noqa: E402

getcontext().prec = 50

EXP = -15                    # element value = a * 2^EXP
SCALE = 2.0 ** EXP
MARGIN_MIN = 0.05            # exact (|peak| - second) / |peak| of every pair
THRESHOLD_GAP = 1e-9         # exact coef at least this far from MIN_CONFIDENCE: success is never a rounding question
SENSITIVITY = 1e-11          # least change of the exact coef under a dropped or shifted window element
# negative-lag windows: every chunk, fp32 group and last-CTA lane boundary of the Pearson step
WINDOW_NS = (0, 1, 2, 3, 4, 5, 31, 32, 33, 1023, 1024, 1025, 4095, 4096, 4097, 16383, 16384, 16385, 16386,
             524287, 524288, 524289)
NOISE = (2, 4, 6)            # noise amplitudes: exact coefs near 0.99, 0.96, 0.93


def positive_raws(L: int, full: bool = True) -> list:
    """Raw indices < L (window n = L at lag = raw): every class mod 4, 0 and L - 1."""
    m = L // 3
    raws = [0, 1, 2, 3, L - 1] + ([m, m + 1, m + 2, m + 3, L - 4, L - 3, L - 2] if full else [])
    return sorted({r for r in raws if 0 <= r < L})


def negative_raws(L: int, ns=WINDOW_NS) -> list:
    """Raw indices >= L whose windows have the n of `ns` (n < L) and n = L - 1: raw = L + n."""
    return sorted({L + n for n in list(ns) + [L - 1] if 0 <= n < L})


def fold(raw: int, L: int):
    """(lag, xoff, yoff, n) of reference src/cross_correlation.c:256-271."""
    if raw >= L:
        lag = raw % L - L
        return lag, 0, -lag, L + lag
    return raw, raw, 0, L


def _coef_float(C, VX, VY):
    """C / sqrt(VX * VY) elementwise in float64 from exact integer (or int64) sums; NaN where 0/0."""
    with np.errstate(all="ignore"):
        return np.asarray(C, np.float64) / (np.sqrt(np.asarray(VX, np.float64)) * np.sqrt(np.asarray(VY, np.float64)))


def exact_coef(X: np.ndarray, Y: np.ndarray):
    """Exact Pearson coefficient of integer windows as a Decimal (NaN for 0/0), plus the integer sums."""
    n = int(X.shape[0])
    X = X.astype(np.int64); Y = Y.astype(np.int64)
    SX, SY = int(X.sum()), int(Y.sum())
    SXX, SYY, SXY = int(np.dot(X, X)), int(np.dot(Y, Y)), int(np.dot(X, Y))
    C = n * SXY - SX * SY
    VX = n * SXX - SX * SX
    VY = n * SYY - SY * SY
    if VX == 0 or VY == 0:
        return Decimal("NaN"), (SXX, SYY)
    return Decimal(C) / (Decimal(VX) * Decimal(VY)).sqrt(), (SXX, SYY)


def sensitivity(X: np.ndarray, Y: np.ndarray, coef: float) -> float:
    """Least |change| of the coefficient over: removing any one window element, and pairing the
    windows one element out of step (x[i + 1] with y[i] or x[i] with y[i + 1], n - 1 pairs).  The
    fold's windows always end where one of the arrays ends, so a window cannot be extended by a pair
    of elements; reading one element too many or too few is one of these changes.  A NaN on one side
    only counts as a change of infinity."""
    n = X.shape[0]
    X = X.astype(np.int64); Y = Y.astype(np.int64)
    SX, SY, SXX, SYY, SXY = X.sum(), Y.sum(), np.dot(X, X), np.dot(Y, Y), np.dot(X, Y)
    m = n - 1
    sx, sy = SX - X, SY - Y
    C = m * (SXY - X * Y) - sx * sy
    VX = m * (SXX - X * X) - sx * sx
    VY = m * (SYY - Y * Y) - sy * sy
    cands = [_coef_float(C, VX, VY)]
    for a, b in ((X[1:], Y[:-1]), (X[:-1], Y[1:])):
        if m >= 1:
            c, _ = exact_coef(a, b)
            cands.append(np.array([float(c)]))
    d = np.concatenate(cands) - coef
    one_nan = np.isnan(d) & ~np.isnan(coef)
    d = np.where(one_nan, np.inf, np.abs(d))
    return float(np.min(d)) if d.size else float("inf")


@dataclass
class ExactPair:
    L: int
    raw: int                 # designed (and exact) raw index
    seed: int
    noise: int
    sign: int
    src: np.ndarray = field(repr=False)   # int16 [2L]
    smp: np.ndarray = field(repr=False)   # int16 [L]
    exp: dict = field(default_factory=dict, repr=False)

    @property
    def name(self):
        return "L=%d raw=%d (lag %d, n %d) noise=%d sign=%+d" % (self.L, self.raw, self.exp["lag"], self.exp["n"],
                                                                self.noise, self.sign)

    def values(self, dtype):
        """(source, sample) as the element values a * 2^-15 in `dtype` (np.int16: the integers, S16)."""
        if np.dtype(dtype) == np.int16:
            return self.src.copy(), self.smp.copy()
        s = np.asarray(SCALE, dtype)
        return self.src.astype(dtype) * s, self.smp.astype(dtype) * s


def _nonzero(rng, n):
    return (rng.integers(1, 16, n) * rng.choice(np.array([-1, 1]), n)).astype(np.int64)


def _arrays(L, raw, seed, noise, sign):
    rng = np.random.default_rng(seed)
    smp = _nonzero(rng, L)
    src = _nonzero(rng, 2 * L)
    c = np.clip(sign * smp + rng.integers(-noise, noise + 1, L), -15, 15)
    c = np.where(c == 0, sign * smp, c)
    src[(np.arange(L) + raw) % (2 * L)] = c
    return src, smp


def exact_record(src: np.ndarray, smp: np.ndarray) -> dict:
    """The exact record of an integer pair (values a * 2^-15): raw_index, lag, window, peak, second,
    margin (float and exact fraction), coef (float nearest the exact Decimal, NaN for 0/0), ret,
    success, window energies ex / ey (exact doubles) and the fp32 error scale N * |src| * |smp|."""
    L = smp.shape[0]
    N = 2 * L
    a = src.astype(np.int64); b = smp.astype(np.int64)
    bp = np.zeros(N); bp[:L] = b
    r = np.fft.irfft(np.fft.rfft(a.astype(np.float64)) * np.conj(np.fft.rfft(bp)), n=N)
    R = np.rint(r)
    assert float(np.max(np.abs(r - R))) < 0.05, "rfft error too large to round"
    R = R.astype(np.int64)
    # reference rule: signed R[0] seed, strict '>' on |R[i]|, first index wins
    mag = np.abs(R[1:])
    j = int(np.argmax(mag)) + 1
    raw = j if mag[j - 1] > R[0] else 0
    rest = np.abs(R).copy(); rest[raw] = -1
    s_idx = int(np.argmax(rest))
    dot = lambda k: int(np.dot(np.take(a, (np.arange(L) + k) % N), b))   # noqa: E731
    assert dot(raw) == int(R[raw]) and dot(s_idx) == int(R[s_idx]), "rfft-rounded correlation disagrees with int64 dots"
    Rp, S = int(R[raw]), int(abs(R[s_idx]))
    lag, xoff, yoff, n = fold(raw, L)
    X, Y = a[xoff:xoff + n], b[yoff:yoff + n]
    coef_d, (SXX, SYY) = exact_coef(X, Y)
    coef = float(coef_d)
    unit = SCALE * SCALE
    peak = float(N) * Rp * unit
    ret = -1 if coef != coef else 0
    return dict(raw_index=raw, lag=lag, xoff=xoff, yoff=yoff, n=n, R=Rp, S=S,
                peak=peak, second=float(N) * S * unit,
                margin=(abs(Rp) - S) / abs(Rp) if Rp else 0.0,
                coef=coef, coef_dec=coef_d, ret=ret,
                success=int(ret == 0 and coef_d >= Decimal(str(MIN_CONFIDENCE))),
                ex=SXX * unit, ey=SYY * unit,
                scale=float(N) * np.sqrt(float(np.dot(a, a))) * np.sqrt(float(np.dot(b, b))) * unit)


def self_check(p: ExactPair) -> list:
    """The problems of a built pair (empty when it passes): designed raw index, margin, distance of
    coef from the threshold, and sensitivity of coef to one dropped or shifted element."""
    e = p.exp
    bad = []
    if e["raw_index"] != p.raw:
        bad.append("raw index %d != designed %d" % (e["raw_index"], p.raw))
    if not e["margin"] >= MARGIN_MIN:
        bad.append("margin %.4f < %.2f" % (e["margin"], MARGIN_MIN))
    if e["n"] >= 2:
        c = e["coef_dec"]
        if c.is_nan():
            bad.append("0/0 coefficient at n = %d" % e["n"])
        else:
            if abs(c - Decimal(str(MIN_CONFIDENCE))) < Decimal(THRESHOLD_GAP):
                bad.append("coef %s within %g of the threshold" % (c, THRESHOLD_GAP))
            a, b = p.src.astype(np.int64), p.smp.astype(np.int64)
            X, Y = a[e["xoff"]:e["xoff"] + e["n"]], b[e["yoff"]:e["yoff"] + e["n"]]
            s = sensitivity(X, Y, e["coef"])
            if not s >= SENSITIVITY:
                bad.append("one-element change moves coef by only %.3g" % s)
    return bad


def build(L: int, raw: int, seed: int, noise: int = None, sign: int = None, tries: int = 20) -> ExactPair:
    """A pair of sample length L whose exact raw index is `raw` and which passes self_check (the seed
    advances until it does).  noise / sign default to a choice from the seed; raw 0 is always positive
    (a negative r[0] never wins under the reference's signed seed)."""
    noise = NOISE[seed % len(NOISE)] if noise is None else noise
    if sign is None:
        sign = -1 if (raw != 0 and seed % 3 == 1) else 1
    for t in range(tries):
        s = seed + 7919 * t
        src, smp = _arrays(L, raw, s, noise, sign)
        p = ExactPair(L, raw, s, noise, sign, src.astype(np.int16), smp.astype(np.int16))
        p.exp = exact_record(src, smp)
        if not self_check(p):
            return p
    raise AssertionError("no pair passes the self-checks: L=%d raw=%d: %s" % (L, raw, self_check(p)))


def shapes(L: int, full: bool = True, short_ns=(0, 1, 2, 5, 33, 4097)) -> list:
    """Raw indices of one length: `full` -- every positive-lag class and every window of WINDOW_NS;
    otherwise the positive-lag classes plus a few short windows and n = L - 1."""
    if full:
        return positive_raws(L) + negative_raws(L)
    return positive_raws(L, full=False) + negative_raws(L, short_ns)


def build_set(L: int, full: bool = True, seed: int = 0, short_ns=(0, 1, 2, 5, 33, 4097)) -> list:
    return [build(L, raw, seed + 1000 * i + L) for i, raw in enumerate(shapes(L, full, short_ns))]
