"""Closed-form probes (tests/golden/probes.py) through the CPU emulation of the kernel bodies.

Every frequency-bin class of each plan (DC, Nyquist, the self-paired bin M/2, row 0 and row M1/2
of the row kernel, the split pairs e <-> M2-1-e ...), every output-position class (0, L, 2L-1,
both outputs of a packed point, column-tile edges, the recurring copy of an embedded plan), the
placement of the second peak and the signed r[0] seed, checked against the exact record
r[j] = N * source[(j + a) mod 2L] of a one-hot sample: raw index exact, peak and second peak
within 2e-6 of N * sum |spike| (the fp32 kernels' floor is ~3e-7 of it).
"""
import ctypes as C
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import probes as pr  # noqa: E402
from test_emu import emu, run_emu, run_generic  # noqa: E402,F401  (module-scoped fixture)

STATIC_LENGTHS = sorted(pr.STATIC_PLANS)
# runtime-radix plans: smooth (24,000), static-rows (48,000), power of two (65,536), embedded (100,001)
GENERIC_LENGTHS = [24000, 48000, 65536, 100001]
SMALL_LENGTHS = [4096, 6000]


def _generic_plan(E, L, precise=False):
    buf = C.create_string_buffer(256)
    assert E.emu_generic_describe(L, int(precise), buf, 256) == 0
    return pr.parse_plan(L, buf.value.decode())


def _fold_lag(E, idx, L):
    lag, xo, yo, n = (C.c_longlong() for _ in range(4))
    E.emu_fold(idx, L, C.byref(lag), C.byref(xo), C.byref(yo), C.byref(n))
    return lag.value


def _run_all(E, probes, runner, tol=pr.TOL_F32):
    """Runs every probe; one assertion listing every mismatch.  Returns the worst relative error."""
    bad, worst = [], 0.0
    for p in probes:
        idx, peak, second = runner(p)
        exp = pr.resolve_tie(p, p.expect(tol=tol), idx, tol)
        msg = pr.check(p, exp, idx, peak, second, tol)
        if not msg and _fold_lag(E, idx, p.L) != exp["lag"]:
            msg = "%s: lag %d != %d" % (p.name, _fold_lag(E, idx, p.L), exp["lag"])
        if msg:
            bad.append(msg)
        else:
            worst = max(worst, pr.error_of(p, exp, peak, second))
    assert not bad, "%d of %d probes:\n  " % (len(bad), len(probes)) + "\n  ".join(bad)
    print("L=%d: %d probes, worst peak/second error %.2e of N * sum|spike|" % (probes[0].L, len(probes), worst))
    return worst


def _static_runner(E, f64=False):
    def run(p):
        src, smp = p.build(np.float64 if f64 else np.float32)
        idx, peak, used = run_emu(E, src, smp, f64=f64)
        assert used == 0, "static plan expected"
        return idx, peak, E.emu_last_second()
    return run


def _generic_runner(E, f64=False, precise=False):
    def run(p):
        src, smp = p.build(np.float64 if f64 else np.float32)
        idx, peak, second, desc = run_generic(E, src, smp, f64=f64, precise=precise)
        return idx, peak, second
    return run


def _small_runner(E):
    def run(p):
        src, smp = p.build(np.float32)
        idx, peak, used = run_emu(E, src, smp)
        assert used == 1, "single-CTA plan expected"
        return idx, peak, E.emu_last_second()
    return run


@pytest.mark.parametrize("L", STATIC_LENGTHS)
def test_static_kernels_bin_probes(emu, L):
    """Family A through K_A / K_B / K_C: every bin class of the plan's M1 x M2 split (the longer
    lengths with one bin per class, 144,000 and 288,000 with several and 16 random bins)."""
    dense = L <= 288000
    pr_ = pr.bin_probes(pr.STATIC_PLANS[L], seed=L, n_random=16 if dense else 2, dense=dense)
    _run_all(emu, pr_, _static_runner(emu))


@pytest.mark.parametrize("L", STATIC_LENGTHS)
def test_static_kernels_position_second_and_seed_probes(emu, L):
    """Families B, C, D through the static kernels: output positions at the edges of the index
    space and of the column tiles, the second peak wherever it sits relative to the peak, and a
    negative r[0] that must neither win nor hide the true peak."""
    plan = pr.STATIC_PLANS[L]
    probes = pr.seed_probes(plan, L + 3)
    if L <= 288000:
        probes = pr.position_probes(plan, L + 1) + pr.second_probes(plan, L + 2) + probes
    else:   # the expensive lengths: the seed family, and one of each placement kind
        probes = pr.position_probes(plan, L + 1)[:8] + pr.second_probes(plan, L + 2)[:6] + \
            [p for p in probes if "0.99" in p.name or "shoulders" in p.name or "tie" in p.name]
    _run_all(emu, probes, _static_runner(emu))


def test_static_kernels_fp64_input(emu):
    """The static kernels instantiated for fp64 input (converted to fp32 on load)."""
    plan = pr.STATIC_PLANS[144000]
    probes = pr.bin_probes(plan, 7, n_random=2, dense=False) + pr.seed_probes(plan, 8)[:6]
    _run_all(emu, probes, _static_runner(emu, f64=True))


@pytest.mark.parametrize("L", GENERIC_LENGTHS)
def test_generic_kernels_all_probe_families(emu, L):
    """The runtime-radix fp32 kernels (fft_generic.cuh): all four families, dense."""
    plan = _generic_plan(emu, L)
    assert plan.embedded == (L == 100001), plan
    _run_all(emu, pr.all_probes(plan, L), _generic_runner(emu))


@pytest.mark.parametrize("L", [24000, 100001])
def test_generic_fp64_instantiation_probes(emu, L):
    """The fp64-arithmetic instantiation (precise mode) on the same probes, fp64 in, within 1e-9."""
    plan = _generic_plan(emu, L, precise=True)
    probes = pr.all_probes(plan, L + 11, dense=False)
    _run_all(emu, probes, _generic_runner(emu, f64=True, precise=True), tol=pr.TOL_F64)


@pytest.mark.parametrize("L", SMALL_LENGTHS)
def test_single_cta_kernel_probes(emu, L):
    """The single-CTA kernel (fft_small.cuh), including a true peak among the seed thread's items."""
    _run_all(emu, pr.all_probes(pr.single_cta_plan(L), L), _small_runner(emu))
