"""Correlation export through the CPU emulation of the kernel bodies -- runs without a GPU.

tests/emu/emu_corr.cu runs one pair, on f64 inputs, unweighted or PHAT, through the static plan at
144,000, the single-CTA kernel or the runtime-radix fp32 kernels (smooth, static-row and embedded
plans), and ends it with either the inverse kernel the library runs without export or its exporting
twin.  The twin must leave the packed peak record unchanged; the reference argmax rule
(lagwin_oracle.windowed_argmax) over the exported values must give the record's raw_index, peak and
second exactly; every exported lag must be within tests/golden/xcorr_error.py's bound; and every export
range must be the matching slice of the full one, bit for bit.
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import emu_build  # noqa: E402
import lagwin_oracle as lo  # noqa: E402
import xcorr_error as xe  # noqa: E402

STATIC, SMALL, GEN32 = 0, 1, 2
STATIC_ROWS, EMBEDDED = 1, 2
# runtime-radix lengths: smooth with runtime-radix rows, smooth with static rows, embedded
CASES = [(STATIC, 144000), (SMALL, 4096), (SMALL, 6000), (GEN32, 24000), (GEN32, 48000), (GEN32, 10007)]
IDS = ["static-144000", "single_cta-4096", "single_cta-6000", "radix-24000", "radix-48000", "radix-10007"]


class Rec(C.Structure):
    _fields_ = [("raw_index", C.c_longlong), ("peak", C.c_double), ("second", C.c_double),
                ("key", C.c_ulonglong), ("second_bits", C.c_uint), ("seed_bits", C.c_uint), ("scale", C.c_double)]


@pytest.fixture(scope="module")
def emu():
    E = C.CDLL(emu_build.build("emu_corr.cu"))
    E.emuc_run.argtypes = [C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int,
                           C.c_longlong, C.c_longlong, C.c_longlong, C.c_longlong, C.c_void_p, C.POINTER(Rec),
                           C.POINTER(C.c_int)]
    return E


def run(E, kind, phat, src, smp, out=False, window=None, rng=None):
    """(record, exported row or None, info)."""
    src = np.ascontiguousarray(src, np.float64)
    smp = np.ascontiguousarray(smp, np.float64)
    L = len(smp)
    clo, chi = rng if rng else (-L, L - 1)
    corr = np.full(chi - clo + 1, 12345.0)
    rec, info = Rec(), C.c_int()
    wlo, whi = window if window else (0, 0)
    rc = E.emuc_run(kind, 1 if phat else 0, src.ctypes.data, smp.ctypes.data, L, 1 if out else 0, 1 if window else 0,
                    wlo, whi, clo, chi, corr.ctypes.data, C.byref(rec), C.byref(info))
    assert rc == 0, rc
    assert rec.key != 12345                      # the kernels cleared the planted peak key
    return rec, (corr if out else None), info.value


def raw_order(corr, L):
    """The full export [-L, L - 1] by raw index."""
    r = np.empty(2 * L)
    lags = np.arange(-L, L)
    r[np.where(lags >= 0, lags, lags + 2 * L)] = corr
    return r


def same_record(a, b):
    assert (a.key, a.second_bits, a.seed_bits) == (b.key, b.second_bits, b.seed_bits), \
        ((a.key, a.second_bits, a.seed_bits), (b.key, b.second_bits, b.seed_bits))


def self_consistent(rec, r, raw):
    """The reference argmax rule over the kernel's own values gives the record exactly."""
    idx, second = lo.windowed_argmax(r, raw)
    assert idx == rec.raw_index, (idx, rec.raw_index)
    assert np.array_equal(r[idx], rec.peak, equal_nan=True), (r[idx], rec.peak)
    assert second == rec.second, (second, rec.second)


def test_plan_kinds_covered(emu):
    """The runtime-radix lengths reach each of the three plan shapes."""
    got = {}
    for kind, L in CASES:
        if kind == GEN32:
            p = xe.make_pair("white", L, 1)
            got[L] = run(emu, kind, False, p.src, p.smp)[2]
    assert got[24000] == 0 and got[48000] == STATIC_ROWS and got[10007] & EMBEDDED, got


@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("kind,L", CASES, ids=IDS)
def test_full_export(emu, kind, L, phat):
    if phat and (kind, L) == (GEN32, 10007):
        pytest.skip("PHAT is not served on embedded lengths")
    p = xe.make_pair("delayed", L, 3)
    plain = run(emu, kind, phat, p.src, p.smp)[0]
    rec, corr, _ = run(emu, kind, phat, p.src, p.smp, out=True)
    same_record(rec, plain)
    r = raw_order(corr, L)
    self_consistent(rec, r, lo.allowed_raw(-L, L - 1, L))
    ref = xe.reference(p.src, p.smp, phat=phat)
    res = xe.judge(np.arange(2 * L), r, ref, yard=xe.yardstick(p.src, p.smp, phat=phat), phat=phat)
    assert res["ok"], res["msg"]


@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("kind,L", CASES, ids=IDS)
def test_windowed_export_and_ranges(emu, kind, L, phat):
    if phat and (kind, L) == (GEN32, 10007):
        pytest.skip("PHAT is not served on embedded lengths")
    p = xe.make_pair("delayed", L, 5)
    full = run(emu, kind, phat, p.src, p.smp, out=True)[1]
    a = p.lag
    for window in ((a - 200, a + 200), (-L // 4, -3), (-50, 60)):
        plain = run(emu, kind, phat, p.src, p.smp, window=window)[0]
        rec, corr, _ = run(emu, kind, phat, p.src, p.smp, out=True, window=window)
        same_record(rec, plain)
        assert np.array_equal(corr, full)        # the range does not depend on the window
        self_consistent(rec, raw_order(corr, L), lo.allowed_raw(*lo.effective(*window, L), L))
    # sub-ranges: all positive, all negative, across 0, one lag, the ends, and one disjoint from the window
    for rng, window in (((5, 900), None), ((-900, -5), None), ((-300, 300), None), ((17, 17), None),
                        ((-L, -L + 10), None), ((L - 11, L - 1), None), ((L // 2, L // 2 + 64), (-40, 40))):
        corr = run(emu, kind, phat, p.src, p.smp, out=True, window=window, rng=rng)[1]
        assert np.array_equal(corr, full[rng[0] + L: rng[1] + L + 1]), rng
