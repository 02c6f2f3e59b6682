"""The exact-sum pairs of tests/golden/exact_pairs.py and their exact records -- runs without a GPU.

tests/test_exact_records_gpu.py holds the device records of these pairs to 1e-13 in coef and to the
bit across paths.  That rests on the claims checked here: the builder's pairs have their peak at the
designed raw index with a clear margin, a coef away from the 0.95 threshold and sensitive to every
one-element change of the window; the sums the Pearson step forms on them are exact in its fp32
arithmetic (a float32 model of the pivots and 16-element partials); and the exact record agrees with
the NumPy and C restatements of the reference and with the fp64 PHAT restatement.
"""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
import exact_pairs as ep  # noqa: E402
import phat_oracle as po  # noqa: E402

from oracle import xcorr_numpy as xn  # noqa: E402

SMALL = (1000, 4096, 6000, 24000)
_SETS = {}


def pair_set(L, full=True):
    key = (L, full)
    if key not in _SETS:
        _SETS[key] = ep.build_set(L, full=full)
    return _SETS[key]


@pytest.mark.parametrize("L", SMALL + (144000, 1440000))
def test_builder_self_checks(L):
    """Every shape: designed raw index, margin >= 0.05, |coef - 0.95| >= 1e-9 and every dropped or
    shifted element moving coef by >= 1e-11; positive lags of every class mod 4 and 0, L - 1; every
    window length of the list below L."""
    pairs = pair_set(L)
    for p in pairs:
        assert not ep.self_check(p), (p.name, ep.self_check(p))
        assert p.exp["raw_index"] == p.raw
        assert np.all((np.abs(p.src) >= 1) & (np.abs(p.src) <= 15)) and np.all((np.abs(p.smp) >= 1) & (np.abs(p.smp) <= 15))
    raws = {p.raw for p in pairs}
    assert {0, L - 1} <= raws and {r % 4 for r in raws if r < L} == {0, 1, 2, 3}
    assert {p.exp["n"] for p in pairs if p.raw >= L} == {n for n in ep.WINDOW_NS if n < L} | {L - 1}
    # both outcomes of success and both signs of the peak
    assert {p.exp["success"] for p in pairs} == {0, 1}
    assert {int(np.sign(p.exp["peak"])) for p in pairs} == {-1, 1}


def test_sensitivity_sees_one_element():
    """The sensitivity measure itself: removing an element or shifting the windows changes coef."""
    p = pair_set(4096)[0]
    e = p.exp
    X, Y = p.src[e["xoff"]:e["xoff"] + e["n"]].astype(np.int64), p.smp[:e["n"]].astype(np.int64)
    s = ep.sensitivity(X, Y, e["coef"])
    assert ep.SENSITIVITY <= s < 1e-3
    drop = float(ep.exact_coef(X[:-1], Y[:-1])[0])
    assert abs(drop - e["coef"]) >= s
    shift = float(ep.exact_coef(X[1:], Y[:-1])[0])
    assert abs(shift - e["coef"]) >= s


def _fp32_pearson_model(x32, y32):
    """float32 model of the Pearson step's fp32 path: pivots from 32 evenly spaced elements rounded to
    float32, shifted values and 16-element partials in float32 (asserted exact), totals in float64."""
    n = x32.shape[0]
    k = (np.arange(32, dtype=np.int64) * n) >> 5
    px = x32[k].astype(np.float64).sum() / 32.0
    py = y32[k].astype(np.float64).sum() / 32.0
    pxf, pyf = np.float32(px), np.float32(py)
    assert float(pxf) == px and float(pyf) == py               # the pivots are exact in fp32
    dx, dy = x32 - pxf, y32 - pyf
    assert np.array_equal(dx.astype(np.float64), x32.astype(np.float64) - px)
    assert np.array_equal(dy.astype(np.float64), y32.astype(np.float64) - py)
    m = n - n % 16
    for a, b in ((dx, dy), (dx, dx), (dy, dy)):
        acc = np.zeros(m // 16, np.float32)
        prods = (a[:m] * b[:m]).reshape(-1, 16)
        for j in range(16):
            acc = acc + prods[:, j]
        exact = (a[:m].astype(np.float64) * b[:m].astype(np.float64)).reshape(-1, 16).sum(1)
        assert np.array_equal(acc.astype(np.float64), exact)
    d64x, d64y = dx.astype(np.float64), dy.astype(np.float64)
    s = [d64x.sum(), d64y.sum(), (d64x * d64x).sum(), (d64y * d64y).sum(), (d64x * d64y).sum()]
    nn = float(n)
    cov = s[4] - s[0] * s[1] / nn
    vx = s[2] - s[0] * s[0] / nn
    vy = s[3] - s[1] * s[1] / nn
    return cov / np.sqrt(vx * vy)


@pytest.mark.parametrize("L", [4096, 1440000])
def test_fp32_pearson_sums_are_exact(L):
    """On every window of the builder, the fp32 path's shifted values and partial sums are exact and
    its finishing arithmetic lands within 1e-13 of the exact coefficient."""
    for p in pair_set(L):
        e = p.exp
        if e["n"] < 2:
            continue
        s, m = p.values(np.float32)
        coef = _fp32_pearson_model(s[e["xoff"]:e["xoff"] + e["n"]], m[e["yoff"]:e["yoff"] + e["n"]])
        assert abs(coef - e["coef"]) <= 1e-13, (p.name, coef, e["coef"])


@pytest.mark.parametrize("L", SMALL + (144000,))
def test_exact_record_matches_restatements(L):
    """The exact record against oracle/xcorr_numpy.py (fold, windows, raw index, peak, second, Pearson
    within 1e-13) and, where it is built, the C restatement oracle/capi."""
    capi = None
    if os.path.exists(os.path.join(ROOT, "oracle", "liboracle.so")):
        from oracle import capi
    for p in pair_set(L, full=L != 144000):
        e = p.exp
        s, m = p.values(np.float64)
        o = xn.cross_correlation(s, m)
        assert (o["raw_index"], o["lag"]) == (e["raw_index"], e["lag"]), p.name
        assert abs(o["peak"] - e["peak"]) <= 1e-12 * e["scale"]
        assert abs(o["second"] - e["second"]) <= 1e-12 * e["scale"]
        lag, wx, wy = xn.windows(s, m, e["raw_index"])
        assert lag == e["lag"] and wx.shape[0] == wy.shape[0] == e["n"]
        assert np.array_equal(wx, s[e["xoff"]:e["xoff"] + e["n"]]) and np.array_equal(wy, m[e["yoff"]:e["yoff"] + e["n"]])
        ref = xn.pearson(wx, wy)
        if e["coef"] != e["coef"]:
            assert ref != ref and e["n"] <= 1
        else:
            assert abs(ref - e["coef"]) <= 1e-13, (p.name, ref, e["coef"])
        if capi is not None:
            # the C restatement is the reference's two-pass loop: sequential fp64 sums, whose rounding
            # grows with n (7.7e-13 at n = 144,000) where NumPy's pairwise sums stay within 1e-13
            c = capi.pearson(wx, wy)
            tol = max(1e-13, e["n"] * 2.0 ** -52)
            assert (c != c) if e["coef"] != e["coef"] else abs(c - e["coef"]) <= tol, (p.name, c, e["coef"])
        with np.errstate(divide="ignore", invalid="ignore"):
            assert e["ex"] == float(np.dot(wx, wx)) and e["ey"] == float(np.dot(wy, wy))


@pytest.mark.parametrize("L", SMALL + (144000,))
def test_phat_peak_at_designed_index(L):
    """The GPU suite expects the whitened correlation's peak at the designed raw index too: the fp64
    PHAT restatement puts it there with a clear margin."""
    for p in pair_set(L, full=L != 144000):
        s, m = p.values(np.float64)
        o = po.phat_record(s, m)
        assert o["raw_index"] == p.raw and o["margin"] >= 0.2, (p.name, o["raw_index"], o["margin"])


@pytest.mark.parametrize("n", [0, 1, 2, 3, 33, 3 * 16384 + 5])
def test_exact_coef_of_explicit_windows(n):
    """The explicit windows of the GPU suite's pearson_coefficient check: 0/0 below two elements, the
    NumPy restatement within 1e-13 above."""
    p = pair_set(1000)[0]
    if n > p.L:
        p = pair_set(144000, full=False)[0]
    c = float(ep.exact_coef(p.src[:n], p.smp[:n])[0])
    s, m = p.values(np.float64)
    ref = xn.pearson(s[:n], m[:n])
    assert (c != c and ref != ref) if n < 2 else abs(c - ref) <= 1e-13
