"""Shared-source reuse path of the static plans through the CPU emulation of the kernel bodies -- no GPU.

tests/emu/emu_shared.cu runs a static plan on pairs that share one source two ways: replicated (K_A on
both signals of every pair, the pair row kernel, K_C) and reuse (K_A on the source alone, the
source-spectrum kernel, the sample-only K_A, the shared-source row kernel, K_C).  The contract of
audiosync_cuda_xcorr_shared_source is that the two agree bit for bit: here the product planes K_C
reads and the packed peak records (key, second_bits, seed_bits), under NONE and PHAT weighting.
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
    out = str(tmp_path_factory.mktemp("emu_shared") / "libasc_emu_shared.so")
    cuda_inc = os.environ.get("CUDA_INC", "/usr/local/cuda/include")
    subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-fPIC", "-shared", "-x", "c++",
                    "-I" + cuda_inc, "-I" + os.path.join(ROOT, "old-audiosync_b200", "csrc"),
                    "-o", out, os.path.join(HERE, "emu", "emu_shared.cu")], check=True)
    E = C.CDLL(out)
    E.emushared_run.argtypes = [C.c_longlong, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    return E


def run(E, L, phat, shared, source, samples):
    n = samples.shape[0]
    prod = np.zeros((n, 2 * L), np.float32)
    key = np.zeros(n, np.uint64)
    second_bits = np.zeros(n, np.uint32)
    seed_bits = np.zeros(n, np.uint32)
    assert E.emushared_run(L, int(phat), int(shared), source.ctypes.data, samples.ctypes.data, n, prod.ctypes.data,
                           key.ctypes.data, second_bits.ctypes.data, seed_bits.ctypes.data) == 0
    return dict(product=prod, key=key, second_bits=second_bits, seed_bits=seed_bits)


def shared_batch(L, seed):
    """One source; samples cut from it at a positive and a negative lag plus noise, and one inverted."""
    rng = np.random.default_rng(seed)
    source = rng.standard_normal(2 * L)
    a, b = 3 * L // 7, L - 11
    samples = np.stack([source[a:a + L] + 0.25 * rng.standard_normal(L),
                        -source[b:b + L]])
    return np.ascontiguousarray(source), np.ascontiguousarray(samples)


@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("L", STATIC_LENGTHS)
def test_reuse_pipeline_is_bit_identical(emu, L, phat):
    source, samples = shared_batch(L, seed=L + int(phat))
    rep = run(emu, L, phat, False, source, samples)
    sh = run(emu, L, phat, True, source, samples)
    for f in ("product", "key", "second_bits", "seed_bits"):
        assert np.array_equal(rep[f].view(np.uint8), sh[f].view(np.uint8)), f
    assert np.isfinite(sh["product"]).all()            # plane 0 (NaN-filled) was never read
    assert (sh["key"] != 12345).all() and sh["key"][0] != sh["key"][1]

