"""Runner-up search kernels through the CPU emulation of the kernel bodies -- runs without a GPU.

tests/emu/emu_runner_up.cu runs the runner-up twins of the static K_C, the runtime-radix inverse column
kernel (fp32; fp64 plans through the restated argmax_f64_runner_up_kernel rule) and the single-CTA
kernel on f64 inputs, with the centre taken from a batch record as on the device.  The probes put a
one-hot sample at 0, so r[j] = N source[j] in closed form.  Bounds as in tests/test_lag_window_emu.py:
raw_index exact; peak / N and second / N within 1e-6 (fp32 arithmetic) or 1e-12 (fp64).  The range
builder (centre, D, lag window -> at most three raw ranges) is checked exhaustively at small L against
the set it stands for.
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
def emu():
    E = C.CDLL(emu_build.build("emu_runner_up.cu"))
    E.emuru_window.argtypes = [C.c_longlong] * 5 + [C.POINTER(C.c_uint)]
    E.emuru_run.argtypes = [C.c_int, C.c_void_p, C.c_void_p] + [C.c_longlong] * 5 + [C.POINTER(Rec)]
    return E


def allowed(p, lo_, hi_, D, L):
    lags = np.arange(lo_, hi_ + 1, dtype=np.int64)
    lags = lags[np.abs(lags - p) >= D]
    return np.sort(np.where(lags >= 0, lags, lags + 2 * L))


def raw_of(lag, L):
    return lag if lag >= 0 else lag + 2 * L


def test_range_builder_exhaustive(emu):
    w = (C.c_uint * 6)()
    for L in (1, 2, 3, 5, 8):
        for lo_ in range(-L, L):
            for hi_ in range(lo_, L):
                for p in range(-L, L):
                    for D in list(range(1, 2 * L + 2)) + [1 << 40]:
                        emu.emuru_window(p, lo_, hi_, D, L, w)
                        got = []
                        for k in range(3):
                            got += list(range(w[2 * k], w[2 * k] + w[2 * k + 1]))
                        want = allowed(p, lo_, hi_, D, L).tolist()
                        assert got == want, (L, lo_, hi_, p, D, list(w))
                        assert (w[1] == 0) == (len(want) == 0)
                        if want:
                            assert w[0] == want[0]
                        else:
                            assert w[0] == 0xFFFFFFFF


def probe(L, spikes):
    """source with the given {lag: value} spikes, sample one-hot at 0: r[raw] = N source[raw]."""
    src = np.zeros(2 * L)
    for lag, v in spikes.items():
        src[raw_of(lag, L)] = v
    smp = np.zeros(L)
    smp[0] = 1.0
    return src, smp


def run(E, kind, src, smp, centre, D, window=None):
    L = len(smp)
    lo_, hi_ = window if window else (-L, L - 1)
    r = Rec()
    assert E.emuru_run(kind, np.ascontiguousarray(src).ctypes.data, np.ascontiguousarray(smp).ctypes.data, L, lo_, hi_,
                       raw_of(centre, L), D, C.byref(r)) == 0
    return r


def expect(r, L, lag, peak, second, tol):
    N = 2 * L
    assert r.raw_index == raw_of(lag, L), (r.raw_index, raw_of(lag, L))
    if np.isnan(peak):
        assert np.isnan(r.peak)
    else:
        assert abs(r.peak / N - peak) <= tol * max(1.0, abs(peak)), (r.peak / N, peak)
    assert abs(r.second / N - second) <= tol * max(1.0, second), (r.second / N, second)


@pytest.mark.parametrize("kind,L", CASES, ids=IDS)
def test_runner_up_rule(emu, kind, L):
    tol = TOL[kind]
    a = L // 4
    # a zone that cuts lag 0 out: the huge negative r[0] and its neighbours are excluded, so nothing
    # is seeded and |r| decides
    src, smp = probe(L, {0: -50.0, 3: 40.0, -4: 30.0, 20: 6.0, -30: -7.0, a: 5.0})
    expect(run(emu, kind, src, smp, 0, 10), L, -30, -7.0, 6.0, tol)
    # a zone at the low end of [-L, L-1]: the centre -L excludes [-L, -L + D)
    src, smp = probe(L, {-L: 9.0, -L + 3: 8.0, -L + 5: 4.0, 1: 3.0})
    expect(run(emu, kind, src, smp, -L, 5), L, -L + 5, 4.0, 3.0, tol)
    # a zone at the high end
    src, smp = probe(L, {L - 1: 9.0, L - 4: 8.0, L - 7: -4.5, 2: 3.0})
    expect(run(emu, kind, src, smp, L - 1, 6), L, L - 7, -4.5, 3.0, tol)
    # a zone crossing the fold (the centre at -L excludes lags -L.. and L-1.. only by plain distance:
    # no wrap-around, so L - 1 stays allowed)
    src, smp = probe(L, {-L + 1: 9.0, L - 1: 7.0, 5: 2.0})
    expect(run(emu, kind, src, smp, -L, 3), L, L - 1, 7.0, 2.0, tol)
    # lag 0 allowed and the seed: a positive r[0] wins over larger |r| elsewhere only by the rule's seed
    src, smp = probe(L, {0: 6.0, a - 5: -5.0, a + 2: 30.0})
    expect(run(emu, kind, src, smp, a + 2, 3, window=(-L, L - 1)), L, 0, 6.0, 5.0, tol)
    # a negative r[0] seed loses to every |r|, but joins `second`
    src[raw_of(0, L)] = -8.0
    expect(run(emu, kind, src, smp, a + 2, 3), L, a - 5, -5.0, 8.0, tol)
    # a tie across the zone boundary: the two allowed ends around the zone have equal |r|; the lower
    # raw index (the positive lag) wins
    src, smp = probe(L, {a - 10: 3.0, a + 10: -3.0, a: 50.0})
    r = run(emu, kind, src, smp, a, 10)
    expect(r, L, a - 10, 3.0, 3.0, tol) if r.raw_index == a - 10 else expect(r, L, a + 10, -3.0, 3.0, tol)


@pytest.mark.parametrize("kind,L", CASES, ids=IDS)
def test_nan_empty_and_window(emu, kind, L):
    tol = TOL[kind]
    # every allowed value NaN: the lowest allowed raw index, with its NaN value
    src, smp = probe(L, {})
    src[:] = np.nan
    src[raw_of(100, L)] = 1.0
    r = run(emu, kind, src, smp, 100, 1, window=(90, 110))
    assert r.raw_index == 90 and np.isnan(r.peak)
    # an empty set: nothing competes (the fp32 kernels leave the cleared key), fp64 reports -1
    src, smp = probe(L, {5: 1.0})
    r = run(emu, kind, src, smp, 0, 50, window=(-20, 20))
    if kind == GEN64:
        assert r.raw_index == -1
    else:
        assert r.key == 0 and r.seed_bits == 0 and r.second == 0.0
    # inside a lag window: three raw ranges around a window holding 0 and a zone right of it
    src, smp = probe(L, {-40: 2.0, -41: 30.0, 3: -2.5, 12: 20.0, 15: 1.0, 30: 1.5, 31: 40.0})
    expect(run(emu, kind, src, smp, 12, 4, window=(-40, 30)), L, 3, -2.5, 2.0, tol)
