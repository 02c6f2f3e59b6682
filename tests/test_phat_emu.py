"""PHAT-weighted correlation through the CPU emulation of the kernel bodies -- runs without a GPU.

tests/emu/emu_phat.cu runs the PHAT twins of the row kernels and of the single-CTA kernel, with the
unweighted column kernels around them, on f64 inputs; this module compiles it (g++, no GPU) into a
temporary directory and compares with the fp64 NumPy restatement in tests/golden/phat_oracle.py.
Bounds: raw_index exact; peak / N and second / N within 1e-6 (fp32 arithmetic) or 1e-12 (fp64).
"""
import ctypes as C
import os
import re
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))
import phat_oracle as po  # noqa: E402
from oracle import xcorr_numpy as xn  # noqa: E402

STATIC_LENGTHS = (144000, 288000, 480000, 720000, 960000, 1440000)
# runtime-radix plans: smooth (24,000), static rows (48,000), power of two (65,536)
GENERIC_LENGTHS = (24000, 48000, 65536)
SMALL_LENGTHS = (4096, 6000)
PATH_STATIC, PATH_SMALL, PATH_GENERIC = 0, 1, 3
COL_T = 16
ROW_LEN = {144000: 480, 288000: 960, 480000: 1200, 720000: 1200, 960000: 2400, 1440000: 2400}
TOL = {False: 1e-6, True: 1e-12}


class Rec(C.Structure):
    _fields_ = [("raw_index", C.c_longlong), ("peak", C.c_double), ("second", C.c_double),
                ("key", C.c_ulonglong), ("second_bits", C.c_uint), ("seed_bits", C.c_uint)]


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_phat") / "libasc_emu_phat.so")
    cuda_inc = os.environ.get("CUDA_INC", "/usr/local/cuda/include")
    subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-fPIC", "-shared", "-x", "c++",
                    "-I" + cuda_inc, "-I" + os.path.join(ROOT, "old-audiosync_b200", "csrc"),
                    "-o", out, os.path.join(HERE, "emu", "emu_phat.cu")], check=True)
    E = C.CDLL(out)
    E.emuphat_xcorr.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.POINTER(Rec), C.POINTER(C.c_int)]
    E.emuphat_generic.argtypes = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.POINTER(Rec), C.POINTER(C.c_int)]
    E.emuphat_path.argtypes = [C.c_longlong, C.c_int, C.c_int]
    return E


def run_auto(E, src, smp, path):
    src = np.ascontiguousarray(src, np.float64); smp = np.ascontiguousarray(smp, np.float64)
    r, p = Rec(), C.c_int()
    assert E.emuphat_xcorr(src.ctypes.data, smp.ctypes.data, len(smp), C.byref(r), C.byref(p)) == 0
    assert p.value == path
    assert r.key != 12345                        # the kernels cleared the planted peak key
    return r


def run_generic(E, src, smp, precise):
    src = np.ascontiguousarray(src, np.float64); smp = np.ascontiguousarray(smp, np.float64)
    r, sr = Rec(), C.c_int()
    assert E.emuphat_generic(src.ctypes.data, smp.ctypes.data, len(smp), int(precise), C.byref(r), C.byref(sr)) == 0
    return r, sr.value


def check(r, o, L, precise=False):
    """Against the oracle; returns the largest error of peak / N and second / N."""
    N = 2 * L
    assert r.raw_index == o["raw_index"]
    err = max(abs(r.peak - o["peak"]) / N, abs(r.second - o["second"]) / N)
    assert err <= TOL[precise], (r.raw_index, r.peak / N, o["peak"] / N, r.second / N, o["second"] / N)
    return err


def probe_shifts(L, m2=None):
    a = {0, 1, L - 1, L, 2 * L - 1, 2 * COL_T - 1, 2 * COL_T}     # column-tile edge: packed column 16
    if m2:
        a |= {2 * m2 - 1, 2 * m2, 2 * m2 * 3 + 2 * COL_T}        # row edge: packed row 1
    return sorted(x for x in a if 0 <= x < 2 * L)


def check_probes(runner, L, m2=None, precise=False):
    """Closed-form shift probes: raw_index = a, peak / N = ncc = 1, second / N ~ 0."""
    N = 2 * L
    for a in probe_shifts(L, m2):
        src, smp = po.shift_probe(L, a, seed=a + 7)
        r = runner(src, smp)
        assert r.raw_index == a, (a, r.raw_index)
        assert abs(r.peak / N - 1.0) <= TOL[precise] and r.second / N <= TOL[precise], (a, r.peak / N, r.second / N)
    # polarity inverted at a = 0: r_w[0] = -N is the signed seed, which any |r_w[i]| beats
    src, smp = po.shift_probe(L, 0, seed=5, sign=-1.0)
    r = runner(src, smp)
    assert r.raw_index != 0
    assert abs(r.second / N - 1.0) <= TOL[precise]
    margin = (abs(r.peak) - r.second) / abs(r.peak)
    assert margin < 0
    # all-zero sample: W = 0, r_w = 0 -- the unweighted record's index, peak and second peak
    r = runner(src, np.zeros(L))
    assert (r.raw_index, r.peak, r.second) == (0, 0.0, 0.0)


def test_header_weighting_matches_binding():
    import audiosync_cuda as ac
    hdr = open(os.path.join(ROOT, "include", "audiosync_cuda.h")).read()
    for name, val in (("NONE", ac.WEIGHT_NONE), ("PHAT", ac.WEIGHT_PHAT)):
        m = re.search(r"AUDIOSYNC_CUDA_WEIGHT_%s\s*=\s*(\d+)" % name, hdr)
        assert m and int(m.group(1)) == val
        assert "WEIGHT_" + name in ac.__all__
    assert "audiosync_cuda_set_weighting" in hdr and "audiosync_cuda_set_weighting" in ac.EXPORTED_SYMBOLS


def test_path_choice(emu):
    """AUTO never takes the time-domain kernel; embedded lengths and PATH_DIRECT are refused."""
    AUTO, FFT, DIRECT = 0, 1, 2
    assert emu.emuphat_path(1000, AUTO, 0) == PATH_SMALL
    assert emu.emuphat_path(4096, AUTO, 0) == PATH_SMALL
    assert emu.emuphat_path(144000, AUTO, 0) == PATH_STATIC
    assert emu.emuphat_path(24000, AUTO, 0) == PATH_GENERIC
    assert emu.emuphat_path(1000, AUTO, 1) == PATH_GENERIC          # precise: fp64 runtime-radix kernels
    assert emu.emuphat_path(144000, AUTO, 1) == PATH_GENERIC
    for L in (100001, 1440002):
        assert emu.emuphat_path(L, AUTO, 0) == -1 and emu.emuphat_path(L, AUTO, 1) == -1
    assert emu.emuphat_path(144000, DIRECT, 0) == -1
    assert emu.emuphat_path(101, FFT, 0) == -1                       # odd and short: no plan at N = 2L


@pytest.mark.parametrize("L", STATIC_LENGTHS)
def test_static_kernels(emu, L):
    src, smp, lag = po.noise_pair(L, seed=L)
    r = run_auto(emu, src, smp, PATH_STATIC)
    check(r, po.phat_record(src, smp), L)
    assert r.raw_index == lag
    check_probes(lambda s, m: run_auto(emu, s, m, PATH_STATIC), L, ROW_LEN[L])


@pytest.mark.parametrize("L", SMALL_LENGTHS)
def test_single_cta_kernel(emu, L):
    src, smp, lag = po.noise_pair(L, seed=L + 1)
    r = run_auto(emu, src, smp, PATH_SMALL)
    check(r, po.phat_record(src, smp), L)
    assert r.raw_index == lag
    check_probes(lambda s, m: run_auto(emu, s, m, PATH_SMALL), L)


@pytest.mark.parametrize("precise", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("L", GENERIC_LENGTHS)
def test_generic_kernels(emu, L, precise):
    src, smp, lag = po.noise_pair(L, seed=L + 2)
    r, static_rows = run_generic(emu, src, smp, precise)
    assert static_rows == (1 if (L == 48000 and not precise) else 0)
    check(r, po.phat_record(src, smp), L, precise)
    assert r.raw_index == lag
    check_probes(lambda s, m: run_generic(emu, s, m, precise)[0], L, precise=precise)


@pytest.mark.parametrize("L,runner", [(144000, "auto"), (48000, "generic")])
def test_coloured_reverberant_pair(emu, L, runner):
    """AR(1)-coloured noise through a decaying room response plus noise: the plain correlation's
    broad peak misses the injected lag (oracle), PHAT finds it, and the kernels agree with the oracle."""
    src, smp, lag = po.coloured_pair(L, seed=1)
    plain = xn.cross_correlation(src, smp)
    assert plain["lag"] != lag and plain["margin"] < 1e-3
    o = po.phat_record(src, smp)
    assert o["lag"] == lag and o["margin"] > 0.1
    r = run_auto(emu, src, smp, PATH_STATIC) if runner == "auto" else run_generic(emu, src, smp, False)[0]
    check(r, o, L)
