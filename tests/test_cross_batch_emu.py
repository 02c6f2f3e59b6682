"""Cross-batch path of the static plans through the CPU emulation of the kernel bodies -- no GPU.

tests/emu/emu_cross.cu runs a static plan on every (source, sample) combination of two sources and three
samples two ways: per pair (K_A on both signals, the pair row kernel, K_C, with each source replicated)
and cross (each source's spectrum once; per wave of samples the sample-only K_A and the samples' forward
rows in place in plane 1; per source the row kernel from both spectra and K_C).  The contract of
audiosync_cuda_xcorr_cross is that the two agree bit for bit: here the product planes K_C reads and the
packed peak records (key, second_bits, seed_bits), under NONE and PHAT weighting, with the samples split
over two waves.
"""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
STATIC_LENGTHS = (144000, 288000, 480000, 720000, 960000, 1440000)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("emu_cross") / "libasc_emu_cross.so")
    cuda_inc = os.environ.get("CUDA_INC", "/usr/local/cuda/include")
    subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-fPIC", "-shared", "-x", "c++",
                    "-I" + cuda_inc, "-I" + os.path.join(ROOT, "old-audiosync_b200", "csrc"),
                    "-o", out, os.path.join(HERE, "emu", "emu_cross.cu")], check=True)
    E = C.CDLL(out)
    E.emucross_run.argtypes = [C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int,
                               C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    return E


def run(E, L, phat, cross, sources, samples, wave=2):
    S, n = sources.shape[0], samples.shape[0]
    prod = np.zeros((S, n, 2 * L), np.float32)
    key = np.zeros((S, n), np.uint64)
    second_bits = np.zeros((S, n), np.uint32)
    seed_bits = np.zeros((S, n), np.uint32)
    assert E.emucross_run(L, int(phat), int(cross), sources.ctypes.data, S, samples.ctypes.data, n, wave,
                          prod.ctypes.data, key.ctypes.data, second_bits.ctypes.data, seed_bits.ctypes.data) == 0
    return dict(product=prod, key=key, second_bits=second_bits, seed_bits=seed_bits)


def cross_batch(L, seed):
    """Two sources and three samples.  Source 0 is loud and every sample is cut from it (at a positive
    and a negative lag, one inverted); source 1 is quiet noise, so that each of its records is below
    source 0's for the same sample and would come out as source 0's if the record were not cleared."""
    rng = np.random.default_rng(seed)
    loud = rng.standard_normal(2 * L)
    quiet = 1e-3 * rng.standard_normal(2 * L)
    a, b, c = 3 * L // 7, L - 11, L // 5
    samples = np.stack([loud[a:a + L] + 0.25 * rng.standard_normal(L),
                        -loud[b:b + L],
                        loud[c:c + L] + 0.5 * rng.standard_normal(L)])
    return np.ascontiguousarray(np.stack([loud, quiet])), np.ascontiguousarray(samples)


@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("L", STATIC_LENGTHS)
def test_cross_pipeline_is_bit_identical(emu, L, phat):
    sources, samples = cross_batch(L, seed=L + int(phat))
    pair = run(emu, L, phat, False, sources, samples)
    cross = run(emu, L, phat, True, sources, samples)
    for f in ("product", "key", "second_bits", "seed_bits"):
        assert np.array_equal(pair[f].view(np.uint8), cross[f].view(np.uint8)), f
    assert np.isfinite(cross["product"]).all()          # plane 0 and unstaged shared memory (NaN) were never read
    assert (cross["key"] != 12345).all()
    # a record the row kernel did not clear would keep source 0's larger key
    assert (pair["key"][1] < pair["key"][0]).all()
