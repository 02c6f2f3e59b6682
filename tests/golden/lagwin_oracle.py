"""fp64 restatement of the lag-windowed record (audiosync_cuda_set_lag_window) -- TEST INFRASTRUCTURE.

The correlation is oracle/xcorr_numpy.correlation (or phat_oracle.phat_correlation under PHAT); the
window restricts the argmax and the second peak to the raw indices of the folded lags [lo, hi]:
raw = lag for lag >= 0, lag + 2L below.  Over them, in ascending raw order, r[0] is the signed seed
only when the window holds lag 0, strict > with the first index winning ties, a NaN never wins, and
when no allowed value is a number the lowest allowed index is the answer.  second is the largest |r|
over the allowed indices other than the peak.  Fold, Pearson, margin and ncc are the unwindowed
record's functions of raw_index.
"""
from __future__ import annotations

import os
import sys

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(_HERE)))
sys.path.insert(0, _HERE)
from oracle import xcorr_numpy as xn  # noqa: E402
import phat_oracle as po  # noqa: E402

INT64_MIN, INT64_MAX = -(1 << 63), (1 << 63) - 1


def effective(lo: int, hi: int, L: int):
    """(lo', hi') = (max(lo, -L), min(hi, L - 1)), or None when empty."""
    lo, hi = max(lo, -L), min(hi, L - 1)
    return None if lo > hi else (lo, hi)


def allowed_raw(lo: int, hi: int, L: int) -> np.ndarray:
    """Allowed raw indices in ascending order."""
    lags = np.arange(lo, hi + 1, dtype=np.int64)
    return np.sort(np.where(lags >= 0, lags, lags + 2 * L))


def windowed_argmax(r: np.ndarray, raw: np.ndarray):
    """(raw_index, second) of r restricted to the ascending raw indices `raw`."""
    vals = r[raw]
    mag = np.abs(vals)
    key = np.where(np.isnan(mag), -np.inf, mag)
    seeded = raw[0] == 0
    if seeded:
        seed = vals[0]
        key = key.copy()
        key[0] = np.inf if np.isnan(seed) else seed
    best = 0
    for j in range(1, len(raw)):          # strict >, ascending: the first index wins ties
        if key[j] > key[best]:
            best = j
    others = np.delete(mag, best)
    others = others[~np.isnan(others)]
    second = float(others.max()) if others.size else 0.0
    return int(raw[best]), second


def record(source: np.ndarray, sample: np.ndarray, lo: int, hi: int, phat: bool = False) -> dict:
    """The windowed record of one pair: raw_index, lag, peak, second, margin, coef, ret, ncc."""
    source = np.asarray(source, np.float64)
    sample = np.asarray(sample, np.float64)
    L = sample.shape[0]
    eff = effective(lo, hi, L)
    assert eff is not None, "empty window"
    r = po.phat_correlation(source, sample) if phat else xn.correlation(source, sample)
    idx, second = windowed_argmax(r, allowed_raw(eff[0], eff[1], L))
    lag, wx, wy = xn.windows(source, sample, idx)
    coef = xn.pearson(wx, wy)
    peak = float(r[idx])
    out = dict(raw_index=idx, lag=int(lag), peak=peak, second=second, coef=coef, ret=-1 if coef != coef else 0,
               rmax=float(np.nanmax(np.abs(r))))       # scale of the transform's rounding
    q = xn.peak_quality(source, sample, idx, peak, second)
    out["margin"] = q["margin"]
    out["ncc"] = peak / (2.0 * L) if phat else q["ncc"]
    return out
