"""Exact-sum pairs (tests/golden/exact_pairs.py) through every record path on the device.

On these pairs every sum of the Pearson step is exact, so each record is checked against the exact
record at the tightest tolerance the arithmetic allows, and every path that reads the same values must
return the same bits:
  - raw_index, lag, ret and success equal the exact values;
  - |coef - exact| <= 1e-13 (NaN where the exact value is 0/0, windows of n = 0 and 1);
  - ncc within 2 ulp of peak / (2L sqrt(Ex Ey)) with the record's own peak and the exact window
    energies (+-inf for n = 0); under PHAT exactly peak / N;
  - margin equal to (|peak| - second) / |peak| of the record's own fields;
  - peak and second within 2e-6 (fp32 transforms) or 1e-12 (fp64: precise mode, the direct kernel)
    of N * |source| * |sample|.
Dropping, repeating or shifting one window element moves the exact coef by at least 1e-11 on every
pair (the builder checks it), 100 times the coef tolerance.

Legs, each on the same arrays, bit-identical to the first in every field: F32 device (aligned, and
with the bases at element offsets that select every load width), F64 device (aligned and one element
off), S16 device (aligned and at odd offsets), F64 host (narrowing off, lossless narrowing of pageable
pairs, always narrowing), and the session pool (F64 and F32 slots, a sample length below the pool's
maximum).  Also: precise mode, PHAT on the device dtypes and the narrowed host leg (bit-identical to
each other), the drop-in cross_correlation, pearson_coefficient on explicit windows, three wave sizes,
and the refusal of a base that is not aligned to its element.
"""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import exact_pairs as ep  # noqa: E402

STATIC = (144000, 288000, 480000, 720000, 960000, 1440000)
LENGTHS = STATIC + (524288, 524289, 6000, 4096, 1000)
FULL = (144000, 1440000)           # every window of exact_pairs.WINDOW_NS; elsewhere a short list
# plan class of each length: 524,288 is a runtime-radix plan of exactly 32 Pearson chunks, 524,289
# (odd) an embedded one of 33 -- the first length whose last-CTA lanes sum more than one chunk
PLAN = {**{L: "static four-step fp32" for L in STATIC}, 524288: "generic four-step fp32",
        524289: "generic four-step, embedded", 6000: "single-CTA", 4096: "single-CTA", 1000: "direct"}
TOL_F32, TOL_F64 = 2e-6, 1e-12     # peak / second error bounds, relative to N * |source| * |sample|
COEF_TOL = 1e-13
F32_OFFSETS = ((1, 3), (2, 0), (3, 1))     # (source, sample) element offsets of the bases
FIELDS = ("lag", "coef", "peak", "ret", "success", "raw_index", "second", "margin", "ncc")

_PAIRS = {}
_LEG1 = {}
_WORST = {}


@pytest.fixture(scope="module")
def ac():
    import audiosync_cuda
    audiosync_cuda.lib()
    return audiosync_cuda


def pairs_for(L):
    if L not in _PAIRS:
        _PAIRS[L] = ep.build_set(L, full=L in FULL)
    return _PAIRS[L]


def host_arrays(pairs, dtype):
    s = np.stack([p.values(dtype)[0] for p in pairs])
    m = np.stack([p.values(dtype)[1] for p in pairs])
    return s, m


def device_records(ctx, pairs, dtype, off=(0, 0)):
    """xcorr_batch_torch on contiguous views whose bases sit `off` elements into their buffers."""
    import torch
    tdt = {np.float32: torch.float32, np.float64: torch.float64, np.int16: torch.int16}[dtype]
    s, m = host_arrays(pairs, dtype)
    n, L = m.shape
    bs = torch.zeros(s.size + 8, dtype=tdt, device="cuda:0")
    bm = torch.zeros(m.size + 8, dtype=tdt, device="cuda:0")
    vs = bs[off[0]:off[0] + s.size]
    vm = bm[off[1]:off[1] + m.size]
    vs.copy_(torch.from_numpy(s.reshape(-1)))
    vm.copy_(torch.from_numpy(m.reshape(-1)))
    esz = np.dtype(dtype).itemsize
    assert vs.data_ptr() % (2 * esz) == (esz if off[0] % 2 else 0)
    return ctx.xcorr_batch_torch(vs.view(n, 2 * L), vm.view(n, L)).copy()


def same(a, b):
    return a.tobytes() == b.tobytes()


def diff_fields(a, b):
    return [f for f in FIELDS if a[f].tobytes() != b[f].tobytes()]


def check(pairs, recs, bound, phat=False):
    """Descriptions of every record field that misses the exact record; the worst peak / second
    error relative to N * |source| * |sample| (None under PHAT)."""
    bad, worst = [], 0.0
    for p, r in zip(pairs, recs):
        e, L = p.exp, p.L
        N = 2 * L
        errs = []
        for f in ("raw_index", "lag", "ret", "success"):
            if int(r[f]) != e[f]:
                errs.append("%s %d != %d" % (f, int(r[f]), e[f]))
        coef = float(r["coef"])
        if e["coef"] != e["coef"]:
            if coef == coef:
                errs.append("coef %.17g, exact 0/0" % coef)
        elif not abs(coef - e["coef"]) <= COEF_TOL:
            errs.append("coef %.17g vs exact %.17g (%.2g)" % (coef, e["coef"], coef - e["coef"]))
        peak, second = np.float64(r["peak"]), np.float64(r["second"])
        ap = abs(peak)
        margin = (ap - second) / ap if ap > 0 else np.float64(0.0)
        if not same(np.float64(r["margin"]), margin):
            errs.append("margin %.17g != %.17g from its own peak / second" % (float(r["margin"]), margin))
        with np.errstate(divide="ignore"):
            if phat:
                ncc = peak / np.float64(N)
                ok = float(r["ncc"]) == ncc
            else:
                ncc = peak / (np.float64(N) * np.sqrt(np.float64(e["ex"]) * np.float64(e["ey"])))
                ok = (float(r["ncc"]) == ncc if not np.isfinite(ncc)
                      else abs(float(r["ncc"]) - ncc) <= 2 * np.spacing(abs(ncc)))
        if not ok:
            errs.append("ncc %.17g vs %.17g" % (float(r["ncc"]), ncc))
        if phat:
            if not ap <= N * (1 + 1e-6):
                errs.append("|peak| %.9g > N" % ap)
        else:
            err = max(abs(float(peak) - e["peak"]), abs(float(second) - e["second"])) / e["scale"]
            worst = max(worst, err)
            if not err <= bound:
                errs.append("peak / second %.9g / %.9g vs exact %.9g / %.9g (%.2e of the scale)"
                            % (peak, second, e["peak"], e["second"], err))
        if errs:
            bad.append("%s: %s" % (p.name, "; ".join(errs)))
    return bad, (None if phat else worst)


def assert_exact(pairs, recs, bound, what, phat=False):
    bad, worst = check(pairs, recs, bound, phat)
    assert not bad, "%s: %d of %d records:\n  " % (what, len(bad), len(pairs)) + "\n  ".join(bad)
    return worst


def leg1(ac, L):
    """F32 device, aligned bases: the records every other NONE leg must reproduce bit for bit."""
    if L not in _LEG1:
        pairs = pairs_for(L)
        with ac.Context([0]) as c:
            desc = c.describe_plan(L)
            _LEG1[L] = device_records(c, pairs, np.float32)
        bound = TOL_F64 if "direct" in desc else TOL_F32
        _WORST[L] = assert_exact(pairs, _LEG1[L], bound, "F32 device " + desc)
        print("L=%d %s: %d pairs, worst peak/second error %.2e of N*|src|*|smp|" % (L, desc, len(pairs), _WORST[L]))
    return _LEG1[L]


@pytest.mark.parametrize("L", LENGTHS)
def test_device_legs_exact_and_bit_identical(ac, L):
    """Legs 1-4: F32 aligned and at element offsets (1, 3), (2, 0), (3, 1); F64 aligned and one
    element off; S16 aligned and at odd offsets."""
    pairs = pairs_for(L)
    with ac.Context([0]) as c:
        assert PLAN[L] in c.describe_plan(L)
    ref = leg1(ac, L)
    with ac.Context([0]) as c:
        legs = [("F32 +%d/+%d" % o, device_records(c, pairs, np.float32, o)) for o in F32_OFFSETS]
        legs += [("F64 +%d/+%d" % o, device_records(c, pairs, np.float64, o)) for o in ((0, 0), (1, 1))]
        legs += [("S16 +%d/+%d" % o, device_records(c, pairs, np.int16, o)) for o in ((0, 0), (1, 1), (0, 3))]
    for name, recs in legs:
        assert not diff_fields(recs, ref), "%s differs from F32 aligned in %s" % (name, diff_fields(recs, ref))


@pytest.mark.parametrize("L", LENGTHS)
def test_host_pool_and_precise_legs(ac, L):
    """Leg 5: F64 host pairs with narrowing off, lossless (pageable; the pairs are narrowed) and always;
    leg 8: session pools with F64 and F32 slots run at this length below their maximum; all bit-identical
    to leg 1.  Leg 6: precise mode, exact within the fp64 bound."""
    pairs = pairs_for(L)
    ref = leg1(ac, L)
    n = len(pairs)
    s, m = host_arrays(pairs, np.float64)
    with ac.Context([0]) as c:
        got = {}
        c.set_host_narrowing(ac.NARROW_OFF)
        c.host_feed_stats(reset=True)
        got["host narrowing off"] = c.xcorr_batch_records(s.ctypes.data, m.ctypes.data, n, L, ac.F64, ac.HOST)
        assert c.host_feed_stats(reset=True) == (n, 0)
        c.set_host_narrowing(ac.NARROW_LOSSLESS)
        got["host lossless narrowing"] = c.xcorr_batch_records(s.ctypes.data, m.ctypes.data, n, L, ac.F64, ac.HOST)
        assert c.host_feed_stats(reset=True) == (0, n)
        c.set_host_narrowing(ac.NARROW_ALWAYS)
        got["host always narrowing"] = c.xcorr_batch_records(s.ctypes.data, m.ctypes.data, n, L, ac.F64, ac.HOST)
        extra = np.full(101, 3 * ep.SCALE)            # frames past the run's length: never read
        for dt, name in ((ac.F64, "pool F64"), (ac.F32, "pool F32")):
            with ac.SessionPool(c, 0, n, L + 1001, dt) as pool:
                for i in range(n):
                    pool.append(i, np.concatenate([s[i], extra]), np.concatenate([m[i], extra]))
                got[name] = pool.run(0, n, L)
    for name, recs in got.items():
        assert not diff_fields(recs, ref), "%s differs from F32 device in %s" % (name, diff_fields(recs, ref))
    with ac.Context([0]) as c:
        c.set_precise(True)
        desc = c.describe_plan(L)
        assert "fp64" in desc
        pre = c.xcorr_batch_records(s.ctypes.data, m.ctypes.data, n, L, ac.F64, ac.HOST)
    worst = assert_exact(pairs, pre, TOL_F64, "precise " + desc)
    print("L=%d precise %s: worst peak/second error %.2e" % (L, desc, worst))


@pytest.mark.parametrize("L", [L for L in LENGTHS if L != 524289])
def test_phat_legs(ac, L):
    """Leg 7: PHAT on F32, F64 and S16 device pairs and on lossless-narrowed F64 host pairs.  The
    whitened peak sits at the designed raw index; coef, ret and success are those of the exact window;
    ncc is peak / N; the four legs are bit-identical.  (Non-smooth lengths have no PHAT plan.)"""
    pairs = pairs_for(L)
    n = len(pairs)
    with ac.Context([0]) as c:
        c.set_weighting(ac.WEIGHT_PHAT)
        desc = c.describe_plan(L)
        assert desc.endswith(" phat")
        legs = [("F32", device_records(c, pairs, np.float32)), ("F64", device_records(c, pairs, np.float64)),
                ("S16", device_records(c, pairs, np.int16))]
        s, m = host_arrays(pairs, np.float64)
        c.host_feed_stats(reset=True)
        legs.append(("F64 host narrowed", c.xcorr_batch_records(s.ctypes.data, m.ctypes.data, n, L, ac.F64, ac.HOST)))
        assert c.host_feed_stats(reset=True) == (0, n)
    assert_exact(pairs, legs[0][1], None, "PHAT F32 " + desc, phat=True)
    for name, recs in legs[1:]:
        assert not diff_fields(recs, legs[0][1]), "PHAT %s differs from PHAT F32 in %s" % (name, diff_fields(recs, legs[0][1]))


@pytest.mark.parametrize("L", [144000, 524289, 4096, 1000])
def test_dropin_matches_leg1(ac, L):
    """The drop-in cross_correlation (F64 host pairs, one call each): (ret, lag, coef) bit-identical to
    the batch records of leg 1."""
    pairs = pairs_for(L)
    ref = leg1(ac, L)
    idx = range(len(pairs)) if L != 144000 else range(0, len(pairs), 3)
    bad = []
    for i in idx:
        s, m = pairs[i].values(np.float64)
        ret, lag, coef = ac.cross_correlation(s, m)
        want = (int(ref["ret"][i]), int(ref["lag"][i]), np.float64(ref["coef"][i]).tobytes())
        if (ret, lag, np.float64(coef).tobytes()) != want:
            bad.append("%s: %d/%d/%.17g vs %d/%d/%.17g" % (pairs[i].name, ret, lag, coef, want[0], want[1],
                                                          float(ref["coef"][i])))
    assert not bad, "\n  ".join(bad)


def test_pearson_coefficient_explicit_windows(ac):
    """pearson_coefficient on windows of every n of the window list, 1,439,999 and 3 * 16384 + 5."""
    p = pairs_for(1440000)[0]                        # raw 0: source[0, L) is the noisy copy of the sample
    assert p.raw == 0
    s, m = p.values(np.float64)
    bad = []
    for n in list(ep.WINDOW_NS) + [3 * 16384 + 5, p.L - 1]:
        x, y = s[:n].copy(), m[:n].copy()
        exact = float(ep.exact_coef(p.src[:n], p.smp[:n])[0])
        got = ac.pearson_coefficient(x, y)
        if exact != exact:
            ok = got != got
        else:
            ok = abs(got - exact) <= COEF_TOL
        if not ok:
            bad.append("n=%d: %.17g vs exact %.17g" % (n, got, exact))
    assert not bad, "\n  ".join(bad)


def test_wave_sizes_bit_identical(ac):
    """One call of every window shape at 144,000 (32 pairs) under wave sizes 0 (the default), 1 and 7:
    the Pearson step's self-resetting tickets serve waves of every size."""
    pairs = pairs_for(144000)
    assert len(pairs) >= 20
    got = []
    for w in (0, 1, 7):
        with ac.Context([0]) as c:
            c.set_wave_pairs(w)
            got.append(device_records(c, pairs, np.float32))
    assert same(got[0], got[1]) and same(got[0], got[2])
    assert same(got[0], leg1(ac, 144000))


def test_refuses_base_not_aligned_to_its_element(ac):
    """A float base 2 bytes off, a double base 4 bytes off and an int16 base 1 byte off are refused
    with -1 and a message, before anything is launched; the context then still computes."""
    import torch
    L, n = 4096, 2
    with ac.Context([0]) as c:
        d_res = torch.zeros(n * ac.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda:0")
        for tdt, dt, off in ((torch.float32, ac.F32, 2), (torch.float64, ac.F64, 4), (torch.int16, ac.S16, 1)):
            bs = torch.zeros(n * 2 * L + 8, dtype=tdt, device="cuda:0")
            bm = torch.zeros(n * L + 8, dtype=tdt, device="cuda:0")
            for sp, mp in ((bs.data_ptr() + off, bm.data_ptr()), (bs.data_ptr(), bm.data_ptr() + off)):
                with pytest.raises(ac.AudiosyncCudaError, match="aligned"):
                    c.xcorr_batch_device(0, sp, mp, n, L, dt, d_res.data_ptr())
        c.synchronize(0)
        assert same(device_records(c, pairs_for(4096), np.float32), leg1(ac, 4096))
