"""Lag-windowed argmax kernels through the CPU emulation of the kernel bodies -- runs without a GPU.

tests/emu/emu_lagwin.cu runs the windowed twins of the static K_C, the runtime-radix inverse column
kernel (fp32; fp64 plans through the restated argmax_f64_window_kernel rule) and the single-CTA kernel
on f64 inputs; this module compiles it (g++, no GPU) into a temporary directory.  The probes put a
one-hot sample at 0, so r[j] = N source[j] in closed form, and set each case of the windowed rule
exactly.  Bounds as in tests/test_phat_emu.py: raw_index exact; peak / N and second / N within 1e-6
(fp32 arithmetic) or 1e-12 (fp64).
"""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
import lagwin_oracle as lo  # noqa: E402

STATIC, SMALL, GEN32, GEN64 = 0, 1, 2, 3
CASES = [(STATIC, L) for L in (144000, 288000, 480000, 720000, 960000, 1440000)] + \
        [(SMALL, 4096), (SMALL, 6000)] + \
        [(k, L) for k in (GEN32, GEN64) for L in (24000, 48000, 65536, 100001)]
IDS = ["%s-%d" % ({STATIC: "static", SMALL: "single_cta", GEN32: "radix_fp32", GEN64: "radix_fp64"}[k], L)
       for k, L in CASES]
TOL = {STATIC: 1e-6, SMALL: 1e-6, GEN32: 1e-6, GEN64: 1e-12}


class Rec(C.Structure):
    _fields_ = [("raw_index", C.c_longlong), ("peak", C.c_double), ("second", C.c_double),
                ("key", C.c_ulonglong), ("second_bits", C.c_uint), ("seed_bits", C.c_uint)]


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_lagwin") / "libasc_emu_lagwin.so")
    cuda_inc = os.environ.get("CUDA_INC", "/usr/local/cuda/include")
    subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-fPIC", "-shared", "-x", "c++",
                    "-I" + cuda_inc, "-I" + os.path.join(ROOT, "old-audiosync_b200", "csrc"),
                    "-o", out, os.path.join(HERE, "emu", "emu_lagwin.cu")], check=True)
    E = C.CDLL(out)
    E.emulw_window.argtypes = [C.c_longlong, C.c_longlong, C.c_longlong, C.POINTER(C.c_uint)]
    E.emulw_run.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_int,
                            C.POINTER(Rec)]
    return E


def run(E, kind, src, smp, window=None):
    """window None: the unwindowed kernels; (lo, hi): the windowed twins."""
    src = np.ascontiguousarray(src, np.float64); smp = np.ascontiguousarray(smp, np.float64)
    r = Rec()
    lo_, hi_ = window if window else (0, 0)
    assert E.emulw_run(kind, src.ctypes.data, smp.ctypes.data, len(smp), lo_, hi_, 1 if window else 0, C.byref(r)) == 0
    if kind != GEN64:
        assert r.key != 12345                    # the kernels cleared the planted peak key
    return r


def probe(L, spikes):
    """source with the given {index: value} spikes, sample one-hot at 0: r[j] = N source[j]."""
    src = np.zeros(2 * L)
    for j, v in spikes.items():
        src[j] = v
    smp = np.zeros(L)
    smp[0] = 1.0
    return src, smp


def expect(r, L, raw, peak, second, tol):
    N = 2 * L
    assert r.raw_index == raw, (r.raw_index, raw)
    if np.isnan(peak):
        assert np.isnan(r.peak)
    else:
        assert abs(r.peak / N - peak) <= tol * max(1.0, abs(peak)), (r.peak / N, peak)
    assert abs(r.second / N - second) <= tol * max(1.0, second), (r.second / N, second)


def test_raw_ranges(emu):
    w = (C.c_uint * 4)()
    L = 1000
    assert emu.emulw_window(lo.INT64_MIN, lo.INT64_MAX, L, w) == 0
    assert emu.emulw_window(-10 * L, 10 * L, L, w) == 0
    assert emu.emulw_window(L, lo.INT64_MAX, L, w) == -1
    assert emu.emulw_window(lo.INT64_MIN, -L - 1, L, w) == -1
    assert emu.emulw_window(5, 9, L, w) == 1 and list(w) == [5, 5, 0, 0]
    assert emu.emulw_window(-9, -5, L, w) == 1 and list(w) == [2 * L - 9, 5, 0, 0]
    assert emu.emulw_window(-3, 4, L, w) == 1 and list(w) == [0, 5, 2 * L - 3, 3]
    assert emu.emulw_window(-L, -L, L, w) == 1 and list(w) == [L, 1, 0, 0]
    for lo_, hi_ in ((5, 9), (-9, -5), (-3, 4), (-L, -L)):
        emu.emulw_window(lo_, hi_, L, w)
        raw = sorted(list(range(w[0], w[0] + w[1])) + list(range(w[2], w[2] + w[3])))
        assert raw == lo.allowed_raw(lo_, hi_, L).tolist()


@pytest.mark.parametrize("kind,L", CASES, ids=IDS)
def test_windowed_rule(emu, kind, L):
    tol = TOL[kind]
    N = 2 * L
    a = L // 4
    # the global max and a larger value just past each end lie outside the window: the in-window
    # maximum is reported and neither outside value reaches `second`
    src, smp = probe(L, {a - 1: 40.0, a + 5: 3.0, a + 9: -2.0, a + 41: 30.0, 0: -50.0})
    expect(run(emu, kind, src, smp, (a, a + 40)), L, a + 5, 3.0, 2.0, tol)
    # window holding 0: a negative r[0] of the largest magnitude loses but joins `second`;
    # a positive one wins at raw 0
    src, smp = probe(L, {0: -50.0, 7: 3.0, 2 * L - 11: -1.0, a: 99.0})
    expect(run(emu, kind, src, smp, (-20, 20)), L, 7, 3.0, 50.0, tol)
    src[0] = 50.0
    expect(run(emu, kind, src, smp, (-20, 20)), L, 0, 50.0, 3.0, tol)
    # window without 0: a huge |r[0]| is neither the peak nor in `second`
    src, smp = probe(L, {0: -50.0, 9: 3.0, 12: -1.0})
    r = run(emu, kind, src, smp, (5, 40))
    expect(r, L, 9, 3.0, 1.0, tol)
    if kind != GEN64:
        assert r.seed_bits == 0                  # r[0] is never read as the seed
    # only negative lags: raw = lag + 2L, in ascending raw order
    src, smp = probe(L, {2 * L - 30: -4.0, 2 * L - 10: 2.5, 10: 9.0})
    expect(run(emu, kind, src, smp, (-40, -5)), L, 2 * L - 30, -4.0, 2.5, tol)
    # equal |r| at the two ends of a window around 0 (r[0] = 0): the positive lag, the lower raw
    # index, wins at equal |r|; the negative one only if rounding made its |r| strictly larger
    w = 25
    src, smp = probe(L, {w: 2.0, 2 * L - w: -2.0})
    r = run(emu, kind, src, smp, (-w, w))
    assert r.raw_index in (w, 2 * L - w)
    assert abs(abs(r.peak) / N - 2.0) <= tol * 2 and abs(r.second / N - 2.0) <= tol * 2
    assert abs(r.peak) > r.second if r.raw_index != w else abs(r.peak) >= r.second


@pytest.mark.parametrize("kind,L", CASES, ids=IDS)
def test_one_lag_windows_and_nan(emu, kind, L):
    tol = TOL[kind]
    src, smp = probe(L, {0: 5.0, L - 1: -3.0, L: 7.0, 100: 11.0})
    expect(run(emu, kind, src, smp, (-L, -L)), L, L, 7.0, 0.0, tol)          # lag -L: raw L
    expect(run(emu, kind, src, smp, (L - 1, L - 1)), L, L - 1, -3.0, 0.0, tol)
    expect(run(emu, kind, src, smp, (0, 0)), L, 0, 5.0, 0.0, tol)
    # every allowed value NaN: the lowest allowed raw index with its NaN value
    src, smp = probe(L, {3: 1.0})
    src[1] = np.nan
    for window, raw in (((5, 40), 5), ((-40, -5), 2 * L - 40), ((-40, 40), 0)):
        r = run(emu, kind, src, smp, window)
        assert r.raw_index == raw and np.isnan(r.peak), (window, r.raw_index, r.peak)


@pytest.mark.parametrize("kind,L", [c for c in CASES if c[0] != STATIC or c[1] <= 288000],
                         ids=[i for c, i in zip(CASES, IDS) if c[0] != STATIC or c[1] <= 288000])
def test_noise_pair_against_oracle(emu, kind, L):
    """A delayed noise pair: windows around the true lag, excluding it, and around 0 against the
    fp64 oracle (a near-tie within the fp32 rounding may resolve to an index of equal |r|)."""
    rng = np.random.default_rng(L)
    lag = L // 3
    src = rng.standard_normal(2 * L)
    smp = src[lag:lag + L] + 0.3 * rng.standard_normal(L)
    for window in ((lag - 500, lag + 500), (lag + 3, lag + 900), (-300, 300)):
        r = run(emu, kind, src, smp, window)
        o = lo.record(src, smp, *window)
        tol = TOL[kind] * o["rmax"]
        if r.raw_index != o["raw_index"]:
            assert kind != GEN64
            alt = lo.record(src, smp, *(2 * [r.raw_index if r.raw_index < L else r.raw_index - 2 * L]))
            assert abs(abs(alt["peak"]) - abs(o["peak"])) <= tol
            continue
        assert abs(r.peak - o["peak"]) <= tol and abs(r.second - o["second"]) <= tol, (window, r.peak, o)


@pytest.mark.parametrize("kind,L", [(STATIC, 144000), (SMALL, 4096), (GEN32, 24000), (GEN32, 100001)],
                         ids=["static-144000", "single_cta-4096", "radix_fp32-24000", "radix_fp32-100001"])
def test_all_allowing_twin_equals_unwindowed(emu, kind, L):
    """The twins with a window that allows every raw index of [0, 2L) but starts past 0 are not
    called by the library (it runs the unwindowed kernels then); with the window [0, L - 1] they
    must give the unwindowed kernels' key whenever the unwindowed answer lies in it."""
    src, smp = probe(L, {0: 1.0, 17: -6.0, 2 * L - 3: 4.0})
    a, b = run(emu, kind, src, smp), run(emu, kind, src, smp, (0, L - 1))
    assert a.raw_index == b.raw_index == 17
    assert a.key == b.key and a.peak == b.peak
