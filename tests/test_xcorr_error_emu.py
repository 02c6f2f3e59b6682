"""Every lag of the correlation r through the CPU emulation of the kernel bodies -- runs without a GPU.

tests/emu/emu_lagwin.cu runs the windowed kernels with a one-lag window [k, k]: the record's peak is
the kernel's r[k] (raw_index k).  Each run reads one slot; the runs go to a thread pool (ctypes
releases the GIL).  Every value read is held to tests/golden/xcorr_error.py's bound against the fp64
reference (fp32 arithmetic) or the exact integer reference (fp64 arithmetic).

The sensitivity test corrupts one entry of a table the static plan builds on the host and shows
that the record checks of the existing suite (raw_index exact, peak within 1e-5) still pass while
the per-lag bound fails.
"""
import ctypes as C
import os
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import emu_build  # noqa: E402
import lagwin_oracle as lo  # noqa: E402
import xcorr_error as xe  # noqa: E402

STATIC, SMALL, GEN32, GEN64 = 0, 1, 2, 3
THREADS = max(1, min(16, os.cpu_count() or 1))


class Rec(C.Structure):
    _fields_ = [("raw_index", C.c_longlong), ("peak", C.c_double), ("second", C.c_double),
                ("key", C.c_ulonglong), ("second_bits", C.c_uint), ("seed_bits", C.c_uint)]


@pytest.fixture(scope="module")
def emu():
    E = C.CDLL(emu_build.build("emu_lagwin.cu"))
    E.emulw_run.argtypes = [C.c_int, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_longlong, C.c_int,
                            C.POINTER(Rec)]
    E.emulw_perturb.argtypes = [C.c_int, C.c_longlong, C.c_longlong, C.c_double]
    E.emulw_table_sizes.argtypes = [C.c_longlong, C.POINTER(C.c_longlong)]
    E.emulw_table_sizes.restype = C.c_longlong
    E.emulw_describe.argtypes = [C.c_int, C.c_longlong, C.c_char_p, C.c_int]
    yield E
    E.emulw_perturb(0, 0, 0, 0.0)


def run_one(E, kind, src, smp, window=None):
    r = Rec()
    lo_, hi_ = window if window else (0, 0)
    rc = E.emulw_run(kind, src.ctypes.data, smp.ctypes.data, len(smp), lo_, hi_, 1 if window else 0, C.byref(r))
    assert rc == 0, rc
    return r


def read_slots(E, kind, src, smp, slots):
    """The kernel's r at each raw slot (one windowed run per slot, in parallel)."""
    src = np.ascontiguousarray(src, np.float64)
    smp = np.ascontiguousarray(smp, np.float64)
    L = len(smp)

    def one(k):
        w = k if k < L else k - 2 * L
        r = run_one(E, kind, src, smp, (w, w))
        assert r.raw_index == k, (k, r.raw_index)
        return r.peak

    with ThreadPoolExecutor(THREADS) as ex:
        return np.array(list(ex.map(one, slots)), np.float64)


def plan_of(E, kind, L):
    if kind == STATIC:
        return xe.STATIC_PLANS[L]
    if kind == SMALL:
        return xe.single_cta_plan(L)
    buf = C.create_string_buffer(512)
    assert E.emulw_describe(kind, L, buf, 512) > 0
    return xe.parse_plan(L, buf.value.decode())


def check(E, kind, L, family, n_slots, seed=1):
    exact = kind == GEN64
    p = xe.make_pair(family, L, seed)
    if exact:
        p = xe.quantised(p)
        r = xe.exact_reference(p.src_int, p.smp_int)
    else:
        r = xe.reference(p.src, p.smp)
    sl = xe.slots(plan_of(E, kind, L), n_slots, seed=L)
    # the peak's neighbourhood and its 2L/12 offsets as slots too: rotations are not needed here
    sl = list(dict.fromkeys(sl + xe.structured_lags(xe.xn.max_abs_index(r), L)[::8]))
    got = read_slots(E, kind, p.src, p.smp, sl)
    res = xe.judge(sl, got, r, fp64=exact, yard=None if exact else xe.yardstick(p.src, p.smp))
    assert res["ok"], "%s L=%d %s: %s" % (kind, L, family, res["msg"])
    return res


@pytest.mark.parametrize("family", ["white", "delayed"])
@pytest.mark.parametrize("L", [4096, 6000])
def test_single_cta_every_slot(emu, L, family):
    check(emu, SMALL, L, family, 2 * L)


@pytest.mark.parametrize("family", ["white", "delayed"])
@pytest.mark.parametrize("L", [24000, 48000, 100001])
def test_runtime_radix_fp32(emu, L, family):
    check(emu, GEN32, L, family, 96)


@pytest.mark.parametrize("family", [f for f in xe.FAMILIES])
def test_static_144000(emu, family):
    check(emu, STATIC, 144000, family, 96)


@pytest.mark.parametrize("family", ["white", "delayed"])
def test_static_1440000(emu, family):
    check(emu, STATIC, 1440000, family, 32)


@pytest.mark.parametrize("family", ["s16", "s16_white", "delayed"])
@pytest.mark.parametrize("L", [24000, 100001])
def test_runtime_radix_fp64_exact(emu, L, family):
    check(emu, GEN64, L, family, 64)


# ----------------------------------------------------------------------------- sensitivity
SENS_L = 144000
# one pass twiddle scaled by (1 + EPS): the smallest scale the bound catches on every entry tried (at
# 3e-6 one of them is rounded away in fp32 and another leaves the error within the bound)
EPS = 1e-5
ROW_S0, ROW_TABP = 120, 124        # Plan144k rows 4x8x15: stride of the first pass, build_row_tab row pitch


def perturbations(E):
    """(name, what, i, j, eps) of the corruptions tried at SENS_L (tables of the static plan): column
    pass twiddles of the first and middle passes; the final-pass part exp(-2 pi i k S0 k1 / M) of
    build_row_tab at rows k1 = 1, 2; neighbouring row pass twiddles."""
    n = (C.c_longlong * 3)()
    assert E.emulw_table_sizes(SENS_L, n) == 0
    n_col, n_row, n_tab = int(n[0]), int(n[1]), int(n[2])
    assert n_tab == 300 * ROW_TABP
    return [("col_tw[%d]*(1+eps)" % i, 1, i, 0, EPS) for i in (1, n_col // 3, 120)] + \
           [("row_tab[%d] conjugated" % i, 2, i, 0, 0.0) for i in (ROW_TABP + ROW_S0 + 1, 2 * ROW_TABP + ROW_S0 + 2)] + \
           [("row_tw[%d] <-> row_tw[%d]" % (i, i + 1), 3, i, i + 1, 0.0) for i in (1, n_row // 3)]


def test_perturbed_tables_pass_records_fail_bound(emu):
    p = xe.make_pair("delayed", SENS_L, seed=9)
    r = xe.reference(p.src, p.smp)
    o = lo.record(p.src, p.smp, -SENS_L, SENS_L - 1)
    peak = xe.xn.max_abs_index(r)
    sl = xe.slots(xe.STATIC_PLANS[SENS_L], 48, seed=3)
    sl = list(dict.fromkeys(sl + xe.structured_lags(peak, SENS_L)[::16]))
    assert xe.judge(sl, read_slots(emu, STATIC, p.src, p.smp, sl), r)["ok"]      # unperturbed: passes
    caught = []
    try:
        for name, what, i, j, eps in perturbations(emu):
            emu.emulw_perturb(what, i, j, eps)
            rec = run_one(emu, STATIC, np.ascontiguousarray(p.src), np.ascontiguousarray(p.smp))
            # the suite's record checks still pass ...
            assert rec.raw_index == o["raw_index"], (name, rec.raw_index, o["raw_index"])
            assert abs(rec.peak - o["peak"]) <= 1e-5 * abs(o["peak"]), (name, rec.peak, o["peak"])
            # ... and the per-lag bound fails
            res = xe.judge(sl, read_slots(emu, STATIC, p.src, p.smp, sl), r)
            caught.append((name, res["ok"], res["a"], res["b"]))
    finally:
        emu.emulw_perturb(0, 0, 0, 0.0)
    missed = [c for c in caught if c[1]]
    assert not missed, "perturbations within the bound: %s" % missed
