"""16-bit PCM (S16) inputs through the CPU emulation of the kernel bodies -- runs without a GPU.

An S16 sample s stands for the value s / 32768 (= s * 2^-15, exact in fp32 and fp64).  The kernels
instantiated for int16_t must therefore produce exactly what their f64-input instantiation produces
on the doubles s / 32768: the same packed peak key, second-peak bits and seed bits on the fp32-argmax
paths, the same resolved index / peak / second peak in fp64 arithmetic.  The same runners also check
the element-load branch that fp32 / fp64 bases at an odd element offset take.  tests/emu/emu_s16.cu
holds the runners; this module compiles it (g++, no GPU) into a temporary directory.
"""
import ctypes as C
import os
import re
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)

STATIC_LENGTHS = (144000, 288000, 480000, 720000, 960000, 1440000)
# runtime-radix plans: smooth (24,000), static rows (48,000), power of two (65,536), embedded odd (100,001)
GENERIC_LENGTHS = (24000, 48000, 65536, 100001)
SMALL_LENGTHS = (4096, 6000)
PATH_FFT = 1
PATH_STATIC, PATH_SMALL, PATH_GENERIC = 0, 1, 3


class Rec(C.Structure):
    _fields_ = [("raw_index", C.c_longlong), ("peak", C.c_double), ("second", C.c_double),
                ("key", C.c_ulonglong), ("second_bits", C.c_uint), ("seed_bits", C.c_uint)]

    def tuple(self):
        return tuple(getattr(self, f) for f, _ in self._fields_)


@pytest.fixture(scope="module")
def emu16(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_s16") / "libasc_emu_s16.so")
    cuda_inc = os.environ.get("CUDA_INC", "/usr/local/cuda/include")
    subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-fPIC", "-shared", "-x", "c++",
                    "-I" + cuda_inc, "-I" + os.path.join(ROOT, "old-audiosync_b200", "csrc"),
                    "-I" + os.path.join(HERE, "emu"), "-o", out, os.path.join(HERE, "emu", "emu_s16.cu")], check=True)
    E = C.CDLL(out)
    xsig = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.POINTER(Rec), C.POINTER(C.c_int)]
    E.emu16_xcorr_s16.argtypes = xsig
    E.emu16_xcorr_f64.argtypes = xsig
    gsig = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.POINTER(Rec)]
    E.emu16_generic_s16.argtypes = gsig
    E.emu16_generic_f64.argtypes = gsig
    vsig = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.c_int, C.POINTER(Rec), C.POINTER(C.c_int)]
    E.emu16_xcorr_vec_f32.argtypes = vsig
    E.emu16_xcorr_vec_f64.argtypes = vsig
    return E


def pcm_pair(L, seed, lag=None, edges=True):
    """int16 source [2L] and sample [L]: the sample is the source from `lag` on plus noise, clipped to the
    int16 range; `edges` puts -32768 and 32767 into both arrays."""
    rng = np.random.default_rng(seed)
    lag = int(rng.integers(0, L)) if lag is None else lag
    src = np.clip(np.round(rng.normal(0, 6000, 2 * L)), -32768, 32767)
    smp = np.clip(src[lag:lag + L] + np.round(rng.normal(0, 1500, L)), -32768, 32767)
    if edges:
        for a in (src, smp):
            a[rng.integers(0, L, 8)] = -32768
            a[rng.integers(0, L, 8)] = 32767
    return src.astype(np.int16), smp.astype(np.int16)


def widen(x):
    return x.astype(np.float64) / 32768.0


def _xcorr(fn, src, smp):
    r, path = Rec(), C.c_int()
    assert fn(src.ctypes.data, smp.ctypes.data, len(smp), PATH_FFT, C.byref(r), C.byref(path)) == 0
    return r.tuple(), path.value


def _generic(fn, src, smp, precise):
    r = Rec()
    assert fn(src.ctypes.data, smp.ctypes.data, len(smp), int(precise), C.byref(r)) == 0
    return r.tuple()


def _check_xcorr(E, src, smp, path):
    """S16 through the int16 kernels == the f64 instantiation on the widened values, field for field."""
    got, p = _xcorr(E.emu16_xcorr_s16, src, smp)
    ref, q = _xcorr(E.emu16_xcorr_f64, widen(src), widen(smp))
    assert p == q == path
    assert got == ref, (got, ref)
    assert got[3] != 12345                      # the kernels cleared the planted peak key
    return got


def test_header_s16_matches_binding():
    import audiosync_cuda as ac
    hdr = open(os.path.join(ROOT, "include", "audiosync_cuda.h")).read()
    m = re.search(r"AUDIOSYNC_CUDA_S16\s*=\s*(\d+)", hdr)
    assert m and int(m.group(1)) == ac.S16 == 2
    assert "S16" in ac.__all__


@pytest.mark.parametrize("L", STATIC_LENGTHS)
def test_static_kernels_s16_equal_f64(emu16, L):
    """K_A's int16 register path (4-byte loads) then K_B / K_C: the f64 instantiation's record."""
    src, smp = pcm_pair(L, seed=L)
    assert _check_xcorr(emu16, src, smp, PATH_STATIC)[0] != 0


@pytest.mark.parametrize("L", SMALL_LENGTHS)
def test_single_cta_kernel_s16_equal_f64(emu16, L):
    src, smp = pcm_pair(L, seed=L + 1)
    _check_xcorr(emu16, src, smp, PATH_SMALL)


@pytest.mark.parametrize("precise", [False, True], ids=["fp32", "fp64"])
@pytest.mark.parametrize("L", GENERIC_LENGTHS)
def test_generic_kernels_s16_equal_f64(emu16, L, precise):
    """Runtime-radix plans, fp32 and fp64 arithmetic: smooth, static rows, power of two, embedded odd."""
    src, smp = pcm_pair(L, seed=L + 2)
    got = _generic(emu16.emu16_generic_s16, src, smp, precise)
    assert got == _generic(emu16.emu16_generic_f64, widen(src), widen(smp), precise)


@pytest.mark.parametrize("L", [144000, 4096, 24000, 100001])
def test_odd_element_offset_takes_two_byte_loads(emu16, L):
    """Bases at an odd element offset (views x[1:]) are only 2-byte aligned: the kernels read them with
    two 2-byte loads per packed point and must give what the aligned copies give, which is F64's."""
    src, smp = pcm_pair(L, seed=L + 3)
    bs = np.empty(2 * L + 1, np.int16); bs[1:] = src
    bm = np.empty(L + 1, np.int16); bm[1:] = smp
    vs, vm = bs[1:], bm[1:]
    assert vs.ctypes.data % 4 == 2 and vm.ctypes.data % 4 == 2
    assert src.ctypes.data % 4 == 0 and smp.ctypes.data % 4 == 0
    aligned = _xcorr(emu16.emu16_xcorr_s16, src, smp)
    for odd_src, odd_smp in ((vs, smp), (src, vm), (vs, vm)):
        assert _xcorr(emu16.emu16_xcorr_s16, odd_src, odd_smp) == aligned
    _check_xcorr(emu16, vs, vm, aligned[1])


@pytest.mark.parametrize("L", [144000, 4096])
def test_full_scale_inputs(emu16, L):
    """Full-scale square waves (every sample -32768 or 32767) and constant full-scale inputs."""
    path = PATH_STATIC if L == 144000 else PATH_SMALL
    rng = np.random.default_rng(L + 4)
    src = np.where(rng.random(2 * L) < 0.5, -32768, 32767).astype(np.int16)
    _check_xcorr(emu16, src, src[17:17 + L].copy(), path)
    _check_xcorr(emu16, np.full(2 * L, -32768, np.int16), np.full(L, 32767, np.int16), path)


@pytest.mark.parametrize("L,phat", [(144000, False), (960000, False), (4096, False), (4096, True),
                                    (6000, False), (6000, True)])
def test_fp_element_loads_equal_pair_loads(emu16, L, phat):
    """fp32 / fp64 inputs at an odd element offset are read one element at a time (vec = 0) by K_A's
    register path and the single-CTA kernel (both weightings): the same peak key, second-peak and seed
    bits as one float2 / double2 load per packed point (vec = 1).  On the host no load can be
    misaligned, so this checks the arithmetic of the element-load branch, not the alignment."""
    path = PATH_STATIC if L >= 144000 else PATH_SMALL         # K_A is the same kernel under PHAT
    src, smp = pcm_pair(L, seed=L + 5)
    for dt, fn in ((np.float32, emu16.emu16_xcorr_vec_f32), (np.float64, emu16.emu16_xcorr_vec_f64)):
        s, m = widen(src).astype(dt), widen(smp).astype(dt)
        got = []
        for vec in (0, 1):
            r, p = Rec(), C.c_int()
            assert fn(s.ctypes.data, m.ctypes.data, L, int(phat), vec, C.byref(r), C.byref(p)) == 0
            assert p.value == path
            got.append(r.tuple())
        assert got[0] == got[1], (dt, got)
        assert got[0][3] != 12345                   # the kernels cleared the planted peak key
