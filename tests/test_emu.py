"""CPU emulation of the CUDA kernel bodies vs the oracle -- runs without a GPU.

tests/emu compiles the same kernel source the GPU runs (ColFwd / RowFused /
ColInv / SmallXcorr in old-audiosync_b200/csrc) against a host executor.  This
checks the product's index maps, digit reversal, twiddle tables, real-FFT
split/merge and argmax keys for every static plan (all six lengths of the
reference's interval schedule, src/audiosync.c:50-57) and for short lengths.
"""
import ctypes as C
import json
import os
import subprocess

import numpy as np
import pytest

from oracle import capi

HERE = os.path.dirname(os.path.abspath(__file__))
SYNTH = json.load(open(os.path.join(HERE, "golden", "synth.json")))


@pytest.fixture(scope="module")
def emu():
    path = os.path.join(HERE, "emu", "libasc_emu.so")
    subprocess.run(["make", "-C", os.path.join(HERE, "emu")], check=True, stdout=subprocess.DEVNULL)
    E = C.CDLL(path)
    sig = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.POINTER(C.c_longlong),
           C.POINTER(C.c_double), C.POINTER(C.c_int)]
    E.emu_xcorr_f32.argtypes = sig
    E.emu_xcorr_f32_ka_registers.argtypes = sig
    E.emu_xcorr_f64.argtypes = sig
    E.emu_fold.argtypes = [C.c_longlong, C.c_longlong] + [C.POINTER(C.c_longlong)] * 4
    E.emu_key_abs.restype = C.c_ulonglong
    E.emu_key_abs.argtypes = [C.c_float, C.c_uint]
    E.emu_key_seed.restype = C.c_ulonglong
    E.emu_key_seed.argtypes = [C.c_float]
    E.emu_key_index.restype = C.c_uint
    E.emu_key_index.argtypes = [C.c_ulonglong]
    E.emu_key_value.restype = C.c_float
    E.emu_key_value.argtypes = [C.c_ulonglong]
    E.emu_path_for.argtypes = [C.c_longlong, C.c_int]
    E.emu_path_for_precise.argtypes = [C.c_longlong, C.c_int]
    gsig = [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int, C.POINTER(C.c_longlong), C.POINTER(C.c_double),
            C.POINTER(C.c_double), C.c_char_p, C.c_size_t]
    E.emu_generic_f32.argtypes = gsig
    E.emu_generic_f64.argtypes = gsig
    E.emu_generic_describe.argtypes = [C.c_longlong, C.c_int, C.c_char_p, C.c_size_t]
    E.emu_last_second.restype = C.c_double
    return E


PATH_AUTO, PATH_FFT = 0, 1


def run_emu(E, src, smp, f64=False, forced=PATH_FFT, ka_registers=False):
    """ka_registers: the static plans' K_A takes fp32 through its register load instead of TMA staging."""
    L = len(smp)
    idx, pk, path = C.c_longlong(), C.c_double(), C.c_int()
    dt = np.float64 if f64 else np.float32
    s = np.ascontiguousarray(src, dt); p = np.ascontiguousarray(smp, dt)
    fn = E.emu_xcorr_f64 if f64 else (E.emu_xcorr_f32_ka_registers if ka_registers else E.emu_xcorr_f32)
    rc = fn(s.ctypes.data, p.ctypes.data, L, forced, C.byref(idx), C.byref(pk), C.byref(path))
    assert rc == 0
    return idx.value, pk.value, path.value


STATIC_LENGTHS = (144000, 288000, 480000, 720000, 960000, 1440000)


def _fft_cases():
    out = []
    for c in SYNTH["cases"]:
        if c["L"] % 2 == 0 and c["tag"] == "pair" and c["pair_id"] in (0, 3):
            out.append(pytest.param(c, False, id="L%d-p%d" % (c["L"], c["pair_id"])))
            # fp32 at a static length: also through K_A's register load (unaligned inputs)
            if c["pair_id"] == 0 and c["L"] in STATIC_LENGTHS:
                out.append(pytest.param(c, True, id="L%d-p%d-ka_registers" % (c["L"], c["pair_id"])))
    return out


@pytest.mark.parametrize("case,ka_registers", _fft_cases())
def test_emulated_kernels_match_golden(emu, case, ka_registers):
    L = case["L"]
    path = emu.emu_path_for(L, PATH_FFT)
    if path == 2:
        pytest.skip("length has no FFT plan (direct path: nothing to emulate)")
    src, smp = capi.synth_pair(case["seed"], case["pair_id"], L)
    idx, peak, used = run_emu(emu, src, smp, f64=(case["pair_id"] == 3), ka_registers=ka_registers)
    assert used == path
    assert case["margin"] > 1e-4                     # unique peak => index must be exact
    assert idx == case["raw_index"]
    assert abs(peak - case["peak"]) <= 1e-4 * abs(case["peak"])
    # second peak (largest |r[i]|, i != argmax) from the same reduction: fp32 transform noise is
    # relative to the PEAK, so the tolerance is 1e-4 of the second peak plus 1e-6 of the peak
    assert abs(emu.emu_last_second() - case["second"]) <= 1e-4 * case["second"] + 1e-6 * abs(case["peak"])
    # the fold compiled into the product gives the reference's lag
    lag, xo, yo, n = (C.c_longlong() for _ in range(4))
    emu.emu_fold(idx, L, C.byref(lag), C.byref(xo), C.byref(yo), C.byref(n))
    assert lag.value == case["lag"]


def test_static_plans_cover_interval_schedule(emu):
    for L in STATIC_LENGTHS:
        assert emu.emu_path_for(L, PATH_AUTO) == 0          # PATH_STATIC_FFT
    for L in (4096, 4320, 5000, 6250, 8192):
        assert emu.emu_path_for(L, PATH_AUTO) == 1          # PATH_SMALL_FFT
    for L in (2, 6, 10, 12, 1000, 2000):
        assert emu.emu_path_for(L, PATH_AUTO) == 2          # short: fp64 direct by default
        assert emu.emu_path_for(L, PATH_FFT) == 1           # ... FFT when asked for
    for L in (1, 5, 7, 14):
        assert emu.emu_path_for(L, PATH_AUTO) == 2          # PATH_DIRECT
        assert emu.emu_path_for(L, PATH_FFT) == 2
    # every other length has an O(N log N) plan: the runtime-radix four-step kernels, at the
    # length itself when it is 2/3/5-smooth, embedded in N' >= 3L otherwise (odd, other primes)
    for L in (4374 * 2 + 1, 4099, 10007, 24000, 65536, 100000, 10 ** 6, 1048576, 1440002, 2 * 3 ** 12, 5 * 10 ** 6):
        assert emu.emu_path_for(L, PATH_AUTO) == 3          # PATH_GENERIC_FFT
    for L in (257, 1001, 2187):                             # short, no single-CTA plan: generic when a transform is asked for
        assert emu.emu_path_for(L, PATH_AUTO) == 2 and emu.emu_path_for(L, PATH_FFT) == 3
    assert emu.emu_path_for(40 * 10 ** 6, PATH_AUTO) == 4   # PATH_NONE: refused, never O(L^2)
    assert emu.emu_path_for(10 ** 6, 2) == 4                # forced direct above 65,536 frames: refused
    # fp64-arithmetic mode: the schedule lengths leave the static fp32 kernels
    for L in (144000, 1440000, 24000, 10007):
        assert emu.emu_path_for_precise(L, PATH_AUTO) == 3
    assert emu.emu_path_for_precise(1000, PATH_AUTO) == 2   # the direct kernel is fp64 already


@pytest.mark.parametrize("L", [2, 4, 6, 8, 10, 12, 16, 18, 20, 30, 36, 48, 50, 100, 250, 486, 1000,
                               1024, 2000, 3600, 4096, 6250, 8192])
def test_small_path_against_oracle(emu, L):
    for pid in (0, 1, 2):
        src, smp = capi.synth_pair(0xABCD, pid, L)
        o = capi.cross_correlation(src, smp)
        idx, peak, used = run_emu(emu, src, smp)
        assert used == 1
        margin = (abs(o["peak"]) - o["second"]) / abs(o["peak"])
        if margin > 1e-4:
            assert idx == o["raw_index"]
            assert abs(peak - o["peak"]) <= 1e-4 * abs(o["peak"])


def test_kat_sine_cases_through_emulator(emu):
    # reference tests/test_cross_correlation.c T7, T8 (L = 1000)
    # T7 (sin(i) vs sin(i)) has peaks at 0, 710 (= 113 * 2pi + 6e-5) and, negated, 355
    # (= 113 * pi + 3e-5) whose magnitudes differ by ~1e-9 relative: only the fp64 direct
    # path, AUTO's choice at L = 1000, can separate them.  The fp32 transform must still
    # land on one of the three.
    p7 = np.sin(np.arange(1000.0))
    idx, _, _ = run_emu(emu, np.sin(np.arange(2000.0)), p7, f64=True)
    assert idx in (0, 355, 710)
    s8 = np.concatenate([np.sin(np.arange(1000.0) + 180), np.zeros(1000)])
    idx, peak, _ = run_emu(emu, s8, p7, f64=True)
    assert idx == 1999 and peak < 0               # lag -1, negative correlation


def test_argmax_key_semantics(emu):
    # reference src/cross_correlation.c:52-67 as a max-reduction over packed keys
    ka, ks, ki, kv = emu.emu_key_abs, emu.emu_key_seed, emu.emu_key_index, emu.emu_key_value
    nan = float("nan")
    assert ks(5.0) > ka(-5.0, 1) and ks(5.0) > ka(5.0, 7)         # ties keep index 0
    assert ka(1.0, 3) > ka(-1.0, 4) and ka(-1.0, 3) > ka(1.0, 4)   # ties keep the earlier index
    assert ka(0.0, 1) > ks(-5.0) and ka(0.0, 1) > ks(-0.5)         # negative seed loses to |0|
    assert ks(0.0) > ka(0.0, 1) and ks(-0.0) > ka(-0.0, 1)         # all-zero -> index 0
    assert ka(nan, 1) < ks(-1e30) and ka(nan, 1) < ka(0.0, 2)      # NaN never wins
    assert ks(nan) > ka(float("inf"), 1)                           # NaN seed is never beaten
    assert ka(2.0, 9) > ka(1.5, 1)
    for v, i in ((3.5, 1), (-2.25, 12345), (1e-30, 2 ** 22), (-7.0, 2879999)):
        k = ka(v, i)
        assert ki(k) == i and kv(k) == np.float32(v)
    assert ki(ks(-4.0)) == 0 and kv(ks(-4.0)) == -4.0


def test_tma_tile_boxes_cover_the_staged_rows(emu):
    # Column tiles are staged as tile_boxes(rows) tensor-map boxes of tile_box_rows(rows) rows
    # (a box holds at most 256), the last one shifted up to end on the last row: every staged row
    # is covered, nothing outside [0, rows) is touched.  rows = M1 - 1 (source, K_C) or M1 / 2.
    for rows in list(range(3, 1300)) + [149, 150, 199, 200, 299, 300, 399, 599]:
        nb, br = emu.emu_tile_boxes(rows), emu.emu_tile_box_rows(rows)
        assert 1 <= br <= 256 and nb * br >= rows and (nb - 1) * br < rows
        covered = set()
        for i in range(nb):
            r0 = emu.emu_tile_box_start(rows, i)
            assert 0 <= r0 and r0 + br <= rows
            covered.update(range(r0, r0 + br))
        assert covered == set(range(rows))


def _hard_144k():
    import sys
    sys.path.insert(0, os.path.join(HERE, "golden"))
    d = json.load(open(os.path.join(HERE, "golden", "hard.json")))
    return [c for c in d["cases"] if c["L"] == 144000]


def _random_lengths(seed, count, lo, hi):
    """Seeded mix of arbitrary integers, 2/3/5-smooth numbers and their +-1 neighbours in [lo, hi]."""
    rng = np.random.default_rng(seed)
    smooth = sorted({2 ** a * 3 ** b * 5 ** c for a in range(22) for b in range(14) for c in range(10)
                     if lo <= 2 ** a * 3 ** b * 5 ** c <= hi})
    out = set()
    while len(out) < count:
        k = len(out) % 4
        if k == 0:
            out.add(int(rng.integers(lo, hi + 1)))
        elif k == 1:
            out.add(int(np.exp(rng.uniform(np.log(lo), np.log(hi)))))
        elif k == 2:
            out.add(smooth[int(rng.integers(len(smooth)))])
        else:
            out.add(min(hi, max(lo, smooth[int(rng.integers(len(smooth)))] + int(rng.choice([-1, 1])))))
    return sorted(out)


def test_generic_planner_on_two_thousand_random_lengths():
    """Property sweep of the planner the runtime-radix kernels rely on (gen_plan.h): for ANY
    sample_len up to 3 million frames a plan exists, M = M1 * M2 is the length itself when it is
    2/3/5-smooth and an embedding 2M >= 3L otherwise (at most ~20 % above the minimum), every radix
    is one the kernels implement, and both the column tile and the four rows fit one SM."""
    import re
    E = C.CDLL(os.path.join(HERE, "emu", "libasc_emu.so"))
    E.emu_generic_describe.argtypes = [C.c_longlong, C.c_int, C.c_char_p, C.c_size_t]
    buf = C.create_string_buffer(256)
    for L in _random_lengths(0xA11, 2000, 64, 3 * 10 ** 6):
        for precise in (0, 1):
            assert E.emu_generic_describe(L, precise, buf, 256) == 0, (L, precise)
            d = buf.value.decode()
            m = re.search(r"M=(\d+) M1=(\d+) M2=(\d+) col=([0-9x]+) row=([0-9x]+) (?:padded|plain) tile=(\d+)", d)
            assert m, d
            M, M1, M2, ct = int(m.group(1)), int(m.group(2)), int(m.group(3)), int(m.group(6))
            col = [int(x) for x in m.group(4).split("x")]; row = [int(x) for x in m.group(5).split("x")]
            assert M1 * M2 == M and int(np.prod(col)) == M1 and int(np.prod(row)) == M2, d
            assert all(r in (2, 3, 4, 5, 6, 8, 9, 10, 12, 15, 16) for r in col + row), d
            n = L
            for q in (2, 3, 5):
                while n % q == 0:
                    n //= q
            if n == 1 and M == L:
                assert "embedded" not in d
            else:                                   # embedded (a smooth length may be too: no split of it fits)
                assert "embedded" in d and 2 * M >= 3 * L and M <= 1.2 * 1.5 * L + 64, (L, d)
            elem = 16 if precise else 8
            assert M1 * ct * elem <= 220 * 1024 and 4 * (M2 + M2 // 8 + 1) * elem <= 220 * 1024, d
            assert len(col) <= 6 and len(row) <= 6, d


@pytest.mark.parametrize("L", _random_lengths(0xB22, 16, 300, 30000))
def test_generic_kernels_random_lengths_vs_oracle(emu, L):
    """The runtime-radix kernel bodies on the CPU at seeded random lengths (arbitrary, smooth,
    smooth +- 1): raw index exact, peak within the fp32 tolerance."""
    from oracle import xcorr_numpy
    src, smp = capi.synth_pair(0xFACE + 1, L % 7, L)
    o = xcorr_numpy.cross_correlation(src, smp)
    assert o["margin"] > 1e-3
    idx, peak, sec, desc = run_generic(emu, src, smp)
    assert idx == o["raw_index"], desc
    assert abs(peak - o["peak"]) <= 1e-5 * abs(o["peak"]), desc
    assert abs(sec - o["second"]) <= 1e-4 * o["second"] + 1e-6 * abs(o["peak"]), desc


@pytest.mark.parametrize("case", _hard_144k(), ids=lambda c: "%s-%.0e" % (c["kind"], c["margin"] or 0))
def test_emulated_kernels_resolve_low_margins_and_edges(emu, case):
    """The fp32 four-step kernel bodies on the hard goldens at L = 144,000: peaks 3e-4 .. 1e-2 apart,
    lags 0 / +-1 / L-1, idx == L, idx == L + 1 and the all-zero sample -- raw index bit-exact."""
    import hard_cases as hc
    src, smp = hc.build(case, np.float32)
    idx, peak, used = run_emu(emu, src, smp)
    assert used == 0 and idx == case["raw_index"]
    assert abs(peak - case["peak"]) <= 1e-4 * abs(case["peak"])
    assert abs(emu.emu_last_second() - case["second"]) <= 1e-4 * case["second"] + 1e-6 * abs(case["peak"])


# ------------------------------------------------------------------ runtime-radix kernels (any length)

def run_generic(E, src, smp, f64=False, precise=False):
    L = len(smp)
    idx, pk, sec = C.c_longlong(), C.c_double(), C.c_double()
    desc = C.create_string_buffer(256)
    dt = np.float64 if f64 else np.float32
    s = np.ascontiguousarray(src, dt); p = np.ascontiguousarray(smp, dt)
    fn = E.emu_generic_f64 if f64 else E.emu_generic_f32
    rc = fn(s.ctypes.data, p.ctypes.data, L, int(precise), C.byref(idx), C.byref(pk), C.byref(sec), desc, 256)
    assert rc == 0
    return idx.value, pk.value, sec.value, desc.value.decode()


GENERIC_LENGTHS = [256, 257, 1001, 2187, 4099, 6561, 8749, 10007, 24000, 39366, 65536, 98415, 100000, 250000]


@pytest.mark.parametrize("L", GENERIC_LENGTHS)
def test_generic_kernels_any_length_vs_oracle(emu, L):
    """fft_generic.cuh bodies on the CPU: 2/3/5-smooth lengths at their own size, everything else
    (odd, prime, 7-smooth ...) embedded in N' >= 3L -- raw index exact, peak and second peak within
    the fp32 tolerance; the fp64 instantiation within 1e-12 of the fp64 oracle."""
    from oracle import xcorr_numpy
    for pid in (0, 1):
        src, smp = capi.synth_pair(0xFACE, pid, L)
        o = xcorr_numpy.cross_correlation(src, smp)
        assert o["margin"] > 1e-3
        idx, peak, sec, desc = run_generic(emu, src, smp)
        assert idx == o["raw_index"], desc
        assert abs(peak - o["peak"]) <= 1e-5 * abs(o["peak"])
        assert abs(sec - o["second"]) <= 1e-4 * o["second"] + 1e-6 * abs(o["peak"])
        idx, peak, sec, desc = run_generic(emu, src, smp, f64=True, precise=True)
        assert idx == o["raw_index"] and "fp64" in desc
        assert abs(peak - o["peak"]) <= 1e-12 * abs(o["peak"])
        assert abs(sec - o["second"]) <= 1e-9 * abs(o["peak"])
    n = L
    for q in (2, 3, 5):
        while n % q == 0:
            n //= q
    assert ("embedded" in desc) == (n != 1)


def test_generic_plan_shapes():
    """The planner: every radix supported, passes minimal, both buffers within one SM's shared memory."""
    import re
    E = C.CDLL(os.path.join(HERE, "emu", "libasc_emu.so"))
    E.emu_generic_describe.argtypes = [C.c_longlong, C.c_int, C.c_char_p, C.c_size_t]
    for L in [256, 4099, 24000, 100000, 250000, 10 ** 6, 1048576, 1440002, 1440000, 3 * 10 ** 6, 5 * 10 ** 6, 7 * 10 ** 6 + 1]:
        for precise in (0, 1):
            buf = C.create_string_buffer(256)
            rc = E.emu_generic_describe(L, precise, buf, 256)
            if rc != 0:
                assert L > 3 * 10 ** 6, (L, precise)       # only very long inputs may lack a plan
                continue
            d = buf.value.decode()
            m = re.search(r"M=(\d+) M1=(\d+) M2=(\d+) col=([0-9x]+) row=([0-9x]+) (?:padded|plain) tile=(\d+)", d)
            M, M1, M2, ct = int(m.group(1)), int(m.group(2)), int(m.group(3)), int(m.group(6))
            col = [int(x) for x in m.group(4).split("x")]; row = [int(x) for x in m.group(5).split("x")]
            assert M1 * M2 == M and np.prod(col) == M1 and np.prod(row) == M2
            assert all(r in (2, 3, 4, 5, 6, 8, 9, 10, 12, 15, 16) for r in col + row)
            assert (M == L) or (2 * M >= 3 * L and M <= 1.2 * 1.5 * L + 64)
            elem = 16 if precise else 8
            assert ct in ((8,) if precise else (8, 16))
            assert M1 * ct * elem <= 220 * 1024 and 4 * (M2 + M2 // 8 + 1) * elem <= 220 * 1024
            assert len(col) <= 6 and len(row) <= 6, d


@pytest.mark.parametrize("case", _hard_144k(), ids=lambda c: "%s-%.0e" % (c["kind"], c["margin"] or 0))
def test_fp64_arithmetic_mode_on_hard_goldens(emu, case):
    """The fp64 instantiation (audiosync_cuda_set_precise) as a second oracle: on the low-margin /
    edge inputs at L = 144,000 it reproduces the compiled reference's raw index, its peak to
    1e-12 and its second peak, and the fp32 runtime-radix kernels agree on the index."""
    import hard_cases as hc
    src, smp = hc.build(case, np.float64)
    idx, peak, sec, _ = run_generic(emu, src, smp, f64=True, precise=True)
    assert idx == case["raw_index"]
    assert abs(peak - case["peak"]) <= 1e-12 * abs(case["peak"]) + 1e-300
    assert abs(sec - case["second"]) <= 1e-9 * abs(case["peak"]) + 1e-300
    idx32, _, _, _ = run_generic(emu, src, smp)
    assert idx32 == case["raw_index"]


def test_fast_division_is_exact(emu):
    """FastDiv (fft_generic.cuh): n / d by multiply-high + shift for every divisor a plan can produce
    (strides and butterflies per row, < 2^20) and every n a kernel forms (< 2^31)."""
    emu.emu_fastdiv_first_error.restype = C.c_longlong
    emu.emu_fastdiv_first_error.argtypes = [C.c_uint, C.c_uint]
    assert emu.emu_fastdiv_first_error(4100, 3000000) == 0
