"""Compile a CPU emulator of tests/emu once per test process -- TEST INFRASTRUCTURE.

The emulators include the kernel headers with every static plan (g++ needs about two minutes for
one), so the modules that load the same emulator share one build in a temporary directory.
"""
from __future__ import annotations

import atexit
import functools
import os
import shutil
import subprocess
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))


@functools.lru_cache(maxsize=None)
def build(source: str) -> str:
    """Path of the shared library built from tests/emu/<source> (g++, no GPU)."""
    out_dir = tempfile.mkdtemp(prefix="asc_emu_")
    atexit.register(shutil.rmtree, out_dir, True)
    out = os.path.join(out_dir, "lib" + os.path.splitext(source)[0] + ".so")
    cuda_inc = os.environ.get("CUDA_INC", "/usr/local/cuda/include")
    subprocess.run([os.environ.get("CXX", "g++"), "-std=c++17", "-O2", "-fPIC", "-shared", "-x", "c++",
                    "-I" + cuda_inc, "-I" + os.path.join(ROOT, "old-audiosync_b200", "csrc"),
                    "-o", out, os.path.join(ROOT, "tests", "emu", source)], check=True)
    return out
