"""GPU parity: the CUDA path (through the C ABI) against the oracle, the committed
golden vectors of the compiled reference, and size-independent properties.

Tolerances (BASELINE.json north_star): lag index bit-exact and ret / success
identical wherever the oracle's peak is unique (margin > 1e-4 of the peak);
peak correlation value and Pearson coefficient within 1e-4 relative.
"""
import json
import math
import os
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
import sys
sys.path.insert(0, os.path.join(HERE, "golden"))
KAT = json.load(open(os.path.join(HERE, "golden", "kat.json")))
SYNTH = json.load(open(os.path.join(HERE, "golden", "synth.json")))
RTOL = 1e-4
SEED = 0x5EED


@pytest.fixture(scope="module")
def ac():
    import audiosync_cuda
    audiosync_cuda.lib()
    return audiosync_cuda


@pytest.fixture(scope="module")
def capi():
    from oracle import capi
    return capi


@pytest.fixture(scope="module")
def ctx(ac):
    c = ac.Context([0])
    yield c
    c.close()


def close(a, b, rtol=RTOL):
    if a != a or b != b:
        return a != a and b != b
    if a == b:                       # also equal infinities
        return True
    return abs(a - b) <= rtol * max(abs(a), abs(b), 1e-300)


def second_close(got, case):
    """Second peak (largest |r[i]|, i != argmax; SURVEY 8f rank 4) vs the oracle's.  The fp32
    transform's noise is relative to the PEAK: 1e-4 of the second peak + 1e-6 of the peak."""
    return abs(got - case["second"]) <= RTOL * case["second"] + 1e-6 * abs(case["peak"])


def kat_inputs(rec):
    if rec["name"] == "T7":
        return np.sin(np.arange(2000.0)), np.sin(np.arange(1000.0))
    if rec["name"] == "T8":
        src = np.concatenate([np.array([math.sin(i + 180) for i in range(1000)]), np.zeros(1000)])
        return src, np.array([math.sin(i) for i in range(1000)])
    return np.array(rec["source"], float), np.array(rec["sample"], float)


# ------------------------------------------------------------------ reference KATs

@pytest.mark.parametrize("rec", KAT["cross_correlation"], ids=lambda r: r["name"])
def test_kat_cross_correlation_dropin(ac, rec):
    """reference tests/test_cross_correlation.c:13-116 through the unchanged C signature."""
    src, smp = kat_inputs(rec)
    ret, lag, coef = ac.cross_correlation(src, smp)
    exp = rec["expect"]
    assert ret == exp["ret"]
    if "lag" in exp:
        assert lag == exp["lag"]
    if "coef_eq" in exp:
        assert coef == exp["coef_eq"]            # exact 1.0, as the reference asserts
    if "coef_gt" in exp:
        assert coef > exp["coef_gt"]
    if "coef_lt" in exp:
        assert coef < exp["coef_lt"]
    if rec["ref"]["coef"] is None:
        assert coef != coef
    else:
        assert close(coef, rec["ref"]["coef"])


@pytest.mark.parametrize("rec", KAT["pearson"], ids=lambda r: r["name"])
def test_kat_pearson_dropin(ac, rec):
    """reference tests/test_pearson_coefficient.c:13-61 (exact equality)."""
    v = ac.pearson_coefficient(np.array(rec["x"]), np.array(rec["y"]))
    if rec["expect"].get("nan"):
        assert v != v
    else:
        assert v == rec["expect"]["eq"]


# ------------------------------------------------------------------ golden vectors

def _pairs():
    return [c for c in SYNTH["cases"] if c["tag"] == "pair"]


@pytest.mark.parametrize("case", _pairs(), ids=lambda c: "L%d-p%d" % (c["L"], c["pair_id"]))
def test_golden_dropin_f64(ac, capi, case):
    """cross_correlation(double*, ...) vs the compiled reference's recorded outputs."""
    src, smp = capi.synth_pair(case["seed"], case["pair_id"], case["L"])
    ret, lag, coef = ac.cross_correlation(src, smp)
    assert case["margin"] > 1e-4
    assert ret == case["ret"] and lag == case["lag"]
    assert close(coef, case["coef"])
    assert (ret == 0 and coef >= ac.MIN_CONFIDENCE) == case["success"]


def _batch_on_device(ac, ctx, seed, first, n, L, dtype=None):
    import torch
    dtype = ac.F32 if dtype is None else dtype
    tdt = torch.float32 if dtype == ac.F32 else torch.float64
    d_src = torch.empty(n * 2 * L, dtype=tdt, device="cuda:0")
    d_smp = torch.empty(n * L, dtype=tdt, device="cuda:0")
    d_res = torch.zeros(n * ac.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda:0")
    ctx.synth_pairs(0, seed, first, n, L, dtype, d_src.data_ptr(), d_smp.data_ptr())
    ctx.xcorr_batch_device(0, d_src.data_ptr(), d_smp.data_ptr(), n, L, dtype, d_res.data_ptr())
    ctx.synchronize(0)
    return d_res.cpu().numpy().view(ac.RESULT_DTYPE), d_src, d_smp


@pytest.mark.parametrize("L", [144000, 288000, 480000, 720000, 960000, 1440000])
def test_golden_batch_device_f32(ac, ctx, L):
    """Device-resident fp32 batch (the headline configuration) vs golden, all six interval sizes."""
    cases = {c["pair_id"]: c for c in _pairs() if c["L"] == L}
    n = max(cases) + 1
    res, _, _ = _batch_on_device(ac, ctx, SEED, 0, n, L)
    for pid, c in cases.items():
        r = res[pid]
        assert int(r["raw_index"]) == c["raw_index"] and int(r["lag"]) == c["lag"]
        assert int(r["ret"]) == c["ret"] and bool(r["success"]) == c["success"]
        assert close(float(r["coef"]), c["coef"]) and close(float(r["peak"]), c["peak"])
        assert second_close(float(r["second"]), c)


def test_device_generator_is_bit_identical(ac, ctx, capi):
    import torch
    L, n = 6000, 5
    for dtype, npdt in ((ac.F32, np.float32), (ac.F64, np.float64)):
        _, d_src, d_smp = _batch_on_device(ac, ctx, SEED + 7, 3, n, L, dtype)
        hs = d_src.cpu().numpy().reshape(n, 2 * L); hp = d_smp.cpu().numpy().reshape(n, L)
        for i in range(n):
            s, p = capi.synth_pair(SEED + 7, 3 + i, L, npdt)
            assert np.array_equal(hs[i], s) and np.array_equal(hp[i], p)


# ------------------------------------------------------------------ low-margin and edge goldens
HARD = json.load(open(os.path.join(HERE, "golden", "hard.json")))


def _hard_id(c):
    return "%s-L%d-%s" % (c["kind"], c["L"], "m%.0e" % c["margin"] if c["kind"] in ("echo", "periodic")
                          else "-".join("%s%s" % kv for kv in sorted(c["params"].items()) if kv[0] != "seed"))


def _check_hard(c, ret, lag, coef, rec=None):
    assert ret == c["ret"] and lag == c["lag"]                       # bit-exact lag, identical ret
    if c["coef"] is None:
        assert coef != coef
    else:
        assert close(coef, c["coef"])
    assert (ret == 0 and coef >= 0.95) == c["success"]
    if rec is not None:
        assert int(rec["raw_index"]) == c["raw_index"] and bool(rec["success"]) == c["success"]
        assert close(float(rec["peak"]), c["peak"])
        assert abs(float(rec["second"]) - c["second"]) <= RTOL * c["second"] + 1e-6 * abs(c["peak"])
        assert abs(float(rec["margin"]) - c["margin"]) <= 3e-5
        if c["ncc"] is None:
            assert rec["ncc"] != rec["ncc"]
        else:
            assert close(float(rec["ncc"]), c["ncc"])


@pytest.mark.parametrize("case", HARD["cases"], ids=_hard_id)
def test_hard_goldens_dropin_and_batch(ac, ctx, case):
    """Outputs of the compiled reference on inputs an fp32 transform can get wrong (tests/golden/
    hard_cases.py): two lags 3e-4 / 1e-3 / 1e-2 of the peak apart at every interval length, lags
    0, +-1, L-1, the fold boundary idx == L and L + 1 (src/cross_correlation.c:256-276) and the
    all-zero sample, at L = 144,000 and 1,440,000 -- through the unchanged C signature (f64
    host) and through the batched records (fp32, the headline configuration)."""
    import hard_cases as hc
    L = case["L"]
    src, smp = hc.build(case, np.float64)
    ret, lag, coef = ac.cross_correlation(src, smp)
    _check_hard(case, ret, lag, coef)
    s32, m32 = hc.build(case, np.float32)
    assert np.array_equal(s32.astype(np.float64), src)                  # exact in fp32 by construction
    rec = ctx.xcorr_batch_records(s32.ctypes.data, m32.ctypes.data, 1, L, ac.F32, ac.HOST)[0]
    _check_hard(case, int(rec["ret"]), int(rec["lag"]), float(rec["coef"]), rec)


# ------------------------------------------------------------------ any length: runtime-radix plans
GEN_LENGTHS = [4099, 8749, 10007, 24000, 48000, 98415, 100000, 192000, 250000, 1000000, 1048576, 1440002, 2400000]
# rows on a static row kernel (M2 in 480 / 960 / 1200 / 2400: multiples of 480 and every embedded length that can choose one)
STATIC_ROW_LENGTHS = {10007, 48000, 192000, 1440002, 2400000}


@pytest.mark.parametrize("L", GEN_LENGTHS)
def test_generic_plan_any_length_vs_oracle(ac, ctx, capi, L):
    """The reference plans FFTW per call for whatever sample_len arrives (src/cross_correlation.c:34,
    :141-142, :237).  Lengths outside the interval schedule run the runtime-radix four-step
    kernels: 2/3/5-smooth ones at their own size, odd / prime-factor ones embedded in N' >= 3L.
    Device-resident fp32 batch and the f64 drop-in call against the NumPy (pocketfft) oracle."""
    from oracle import xcorr_numpy
    desc = ctx.describe_plan(L)
    assert "generic four-step" in desc and "fp32" in desc, desc
    assert ("static-rows" in desc) == (L in STATIC_ROW_LENGTHS), desc
    n = 3 if L < 2000000 else 2
    res, d_src, d_smp = _batch_on_device(ac, ctx, SEED + 50, 0, n, L)
    for i in range(n):
        src, smp = capi.synth_pair(SEED + 50, i, L)
        o = xcorr_numpy.cross_correlation(src, smp)
        r = res[i]
        assert o["margin"] > 1e-4
        assert int(r["raw_index"]) == o["raw_index"] and int(r["lag"]) == o["lag"] == capi.synth_true_lag(SEED + 50, i, L)
        assert int(r["ret"]) == o["ret"] and bool(r["success"]) == (o["ret"] == 0 and o["coef"] >= 0.95)
        assert close(float(r["coef"]), o["coef"]) and close(float(r["peak"]), o["peak"])
        assert abs(float(r["second"]) - o["second"]) <= RTOL * o["second"] + 1e-6 * abs(o["peak"])
        assert abs(float(r["margin"]) - o["margin"]) <= 1e-4 and close(float(r["ncc"]), o["ncc"])
        if i == 0:
            ret, lag, coef = ac.cross_correlation(src, smp)          # unchanged C signature, f64 host
            assert (ret, lag) == (o["ret"], o["lag"]) and close(coef, o["coef"])


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


def test_any_length_random_sweep(ac, ctx, capi):
    """Sixty seeded random sample_len values between 4,096 and 2.5 million frames -- arbitrary integers,
    2/3/5-smooth numbers, smooth +- 1 -- through whatever plan the library picks: the injected lag of
    every pair, and on the first pair of each length raw index / peak / coefficient against the NumPy
    (pocketfft) oracle.  The reference plans FFTW per call for any length
    (src/cross_correlation.c:34, :141-142, :237)."""
    from oracle import xcorr_numpy
    kinds = set()
    for L in _random_lengths(0xC33, 60, 4096, 2500000):
        n = 3 if L < 500000 else 2
        res, d_src, d_smp = _batch_on_device(ac, ctx, SEED + 90, 0, n, L)
        desc = ctx.describe_plan(L)
        kinds.add(desc.split()[0] + (" embedded" if "embedded" in desc else ""))
        for i in range(n):
            assert int(res["ret"][i]) == 0 and int(res["lag"][i]) == capi.synth_true_lag(SEED + 90, i, L), (L, i, desc)
        src, smp = capi.synth_pair(SEED + 90, 0, L)
        o = xcorr_numpy.cross_correlation(src, smp)
        r = res[0]
        assert o["margin"] > 1e-4
        assert int(r["raw_index"]) == o["raw_index"] and int(r["lag"]) == o["lag"], (L, desc)
        assert close(float(r["coef"]), o["coef"]) and close(float(r["peak"]), o["peak"]), (L, desc)
        assert abs(float(r["margin"]) - o["margin"]) <= 1e-4, (L, desc)
        del d_src, d_smp
    assert any("embedded" in k for k in kinds) and len(kinds) >= 2, kinds


def test_generic_plans_of_different_sizes_in_one_context(ac, ctx, capi):
    """A large plan, a small one, the large one again, all on the same kernels of one context: the
    shared-memory limit of a kernel must not shrink with the last plan built."""
    for L in (1000000, 4099, 1000000, 24000, 250000, 1000000):
        res, _, _ = _batch_on_device(ac, ctx, SEED + 70, 0, 2, L)
        for i in range(2):
            assert int(res["lag"][i]) == capi.synth_true_lag(SEED + 70, i, L) and int(res["ret"][i]) == 0


def test_generic_plan_edges_off_schedule(ac, ctx, capi):
    """idx == L, idx == L + 1, all-zero sample and a NaN input on an embedded (odd) length."""
    import hard_cases as hc
    L = 100001
    for case in (dict(kind="impulse", L=L, params=dict(i_src=L, i_smp=0)),
                 dict(kind="impulse", L=L, params=dict(i_src=0, i_smp=L - 1)),
                 dict(kind="zero_sample", L=L, params=dict(seed=3)),
                 dict(kind="lag", L=L, params=dict(seed=4, lag=L - 1)),
                 dict(kind="lag", L=L, params=dict(seed=5, lag=-1))):
        src, smp = hc.build(case, np.float32)
        o = capi.cross_correlation(src.astype(np.float64), smp.astype(np.float64))
        rec = ctx.xcorr_batch_records(src.ctypes.data, smp.ctypes.data, 1, L, ac.F32, ac.HOST)[0]
        assert (int(rec["ret"]), int(rec["lag"]), int(rec["raw_index"])) == (o["ret"], o["lag"], o["raw_index"]), case
        assert close(float(rec["coef"]), o["coef"]) and close(float(rec["peak"]), o["peak"])
    src, smp = capi.synth_pair(SEED, 0, L, np.float32)
    src = src.copy(); src[L // 3] = np.nan
    rec = ctx.xcorr_batch_records(src.ctypes.data, smp.ctypes.data, 1, L, ac.F32, ac.HOST)[0]
    assert int(rec["ret"]) == -1 and int(rec["lag"]) == 0 and rec["coef"] != rec["coef"]
    with pytest.raises(ac.AudiosyncCudaError):                      # no plan fits: refused, never O(L^2)
        ctx.describe_plan(40 * 10 ** 6)


# ------------------------------------------------------------------ fp64-arithmetic validation mode

@pytest.mark.parametrize("L", [144000, 288000, 480000, 720000, 960000, 1440000])
def test_precise_mode_is_a_second_oracle_at_schedule_lengths(ac, capi, L):
    """audiosync_cuda_set_precise: the transforms in fp64 arithmetic (reference :187-239 computes in
    double complex).  Against the compiled reference's goldens: raw index exact, peak within 1e-12,
    coefficient within 1e-10, on the white-noise pairs AND the low-margin / edge pairs; and the
    fp32 product path agrees with it on every index."""
    import hard_cases as hc
    with ac.Context([0]) as cp, ac.Context([0]) as cf:
        cp.set_precise(True)
        assert "fp64" in cp.describe_plan(L) and "static" in cf.describe_plan(L)
        cases = [(c, capi.synth_pair(c["seed"], c["pair_id"], L)) for c in _pairs() if c["L"] == L]
        cases += [(c, hc.build(c, np.float64)) for c in HARD["cases"] if c["L"] == L]
        for c, (src, smp) in cases:
            rp = cp.xcorr_batch_records(src.ctypes.data, smp.ctypes.data, 1, L, ac.F64, ac.HOST)[0]
            rf = cf.xcorr_batch_records(src.ctypes.data, smp.ctypes.data, 1, L, ac.F64, ac.HOST)[0]
            assert int(rp["raw_index"]) == c["raw_index"] == int(rf["raw_index"])
            assert int(rp["lag"]) == c["lag"] and int(rp["ret"]) == c["ret"]
            assert abs(float(rp["peak"]) - c["peak"]) <= 1e-12 * abs(c["peak"])
            assert abs(float(rp["second"]) - c["second"]) <= 1e-9 * abs(c["peak"])
            if c["coef"] is None:
                assert rp["coef"] != rp["coef"]
            else:
                assert abs(float(rp["coef"]) - c["coef"]) <= 1e-10 * abs(c["coef"])
            # the fp32 kernels against the fp64 ones: peak 1e-5, margin 3e-5
            assert abs(float(rf["peak"]) - float(rp["peak"])) <= 1e-5 * abs(float(rp["peak"]))
            assert abs(float(rf["margin"]) - float(rp["margin"])) <= 3e-5


# ------------------------------------------------------------------ oracle, many shapes

@pytest.mark.parametrize("L", [1, 2, 3, 5, 6, 7, 8, 9, 10, 11, 12, 50, 63, 64, 250, 255, 256, 257, 1000, 1001, 2187])
def test_short_and_odd_lengths_vs_oracle(ac, capi, L):
    """Arbitrary sample_len > 0 (primes, odd, tiny) -- the universal direct path."""
    for pid in range(4):
        src, smp = capi.synth_pair(SEED + 1, pid, L)
        o = capi.cross_correlation(src, smp)
        ret, lag, coef = ac.cross_correlation(src, smp)
        margin = (abs(o["peak"]) - o["second"]) / abs(o["peak"]) if o["peak"] != 0 else 0.0
        assert ret == o["ret"]
        if margin > 1e-4:
            assert lag == o["lag"]
            assert close(coef, o["coef"])


@pytest.mark.parametrize("L", [64, 250, 1000, 1024, 3600, 4096, 6000, 8192])
def test_small_fft_path_vs_direct_and_oracle(ac, capi, L):
    """Single-CTA FFT kernel (forced) and the direct kernel agree with the oracle."""
    n = 6
    srcs = np.empty((n, 2 * L), np.float32); smps = np.empty((n, L), np.float32)
    for i in range(n):
        srcs[i], smps[i] = capi.synth_pair(SEED + 2, i, L, np.float32)
    outs = {}
    for path in (ac.PATH_FFT, ac.PATH_DIRECT):
        with ac.Context([0]) as c:
            c.set_path(path)
            desc = c.describe_plan(L)
            assert desc.startswith("fft" if path == ac.PATH_FFT else "direct"), desc
            outs[path] = c.xcorr_batch(srcs, smps)
    for i in range(n):
        o = capi.cross_correlation(srcs[i].astype(np.float64), smps[i].astype(np.float64))
        for path in outs:
            r = outs[path]
            assert r["lags"][i] == o["lag"] and r["rets"][i] == o["ret"]
            assert close(r["coefs"][i], o["coef"]) and close(r["peaks"][i], o["peak"])


def test_all_zero_sample_and_constant_inputs(ac):
    L = 1000
    src = np.arange(2 * L, dtype=np.float64)
    ret, lag, coef = ac.cross_correlation(src, np.zeros(L))
    assert ret == -1 and lag == 0 and coef != coef         # T2 at a larger size
    ret, lag, coef = ac.cross_correlation(np.ones(2 * L), np.ones(L))
    assert ret == -1 and coef != coef                      # zero variance -> NaN gate


def test_fold_boundary_idx_equals_L(ac, capi):
    """idx == L => empty Pearson window => NaN => -1 with lag = -L written (cross_correlation.c:256-276)."""
    for L in (8, 1000, 4096):
        src = np.zeros(2 * L); smp = np.zeros(L)
        smp[0] = 1.0; src[L] = 1.0
        o = capi.cross_correlation(src, smp)
        ret, lag, coef = ac.cross_correlation(src, smp)
        assert (ret, lag) == (o["ret"], o["lag"]) == (-1, -L) and coef != coef


def test_argmax_ties_and_sign_semantics(ac, capi):
    """max_abs_index (cross_correlation.c:52-67): first index wins ties; r[0] enters signed."""
    L = 9   # odd -> direct fp64 path, exact arithmetic on these integers
    smp = np.zeros(L); smp[0] = 1.0
    src = np.zeros(2 * L); src[3] = 2.0; src[11] = -2.0            # |r[3]| == |r[11]|
    o = capi.cross_correlation(src, smp)
    ret, lag, coef = ac.cross_correlation(src, smp)
    assert o["raw_index"] == 3 and (ret, lag) == (o["ret"], o["lag"])
    src = np.zeros(2 * L); src[0] = -5.0; src[4] = 1.0              # r[0] < 0 never wins
    o = capi.cross_correlation(src, smp)
    ret, lag, coef = ac.cross_correlation(src, smp)
    assert o["raw_index"] == 4 and (ret, lag) == (o["ret"], o["lag"])
    src = np.zeros(2 * L); src[0] = 5.0; src[4] = -5.0              # r[0] >= |r[i]| keeps index 0
    o = capi.cross_correlation(src, smp)
    ret, lag, coef = ac.cross_correlation(src, smp)
    assert o["raw_index"] == 0 and (ret, lag) == (o["ret"], o["lag"])


# ------------------------------------------------------------------ interval schedule (config 2)

@pytest.mark.parametrize("pid", [0, 6])
def test_interval_schedule_vs_golden(ac, capi, pid):
    """src/audiosync.c:226-259 on one full-length pair: per-interval (ret, lag, coef, success)."""
    cases = [c for c in SYNTH["cases"] if c["tag"] == "interval-prefix" and c["pair_id"] == pid]
    src, smp = capi.synth_pair(cases[0]["seed"], pid, 1440000)
    out = ac.interval_loop(src, smp)
    first_ok = next(i for i, c in enumerate(cases) if c["success"])
    assert out["n"] == first_ok + 1 and out["final_ret"] == 0
    for i in range(out["n"]):
        c = cases[i]
        assert out["rets"][i] == c["ret"] and bool(out["succ"][i]) == c["success"]
        if c["margin"] > 1e-4:
            assert out["lags"][i] == c["lag"]
            assert abs(out["coefs"][i] - c["coef"]) <= max(RTOL * abs(c["coef"]), 1e-6)
    assert out["final_lag"] == ac.frames_to_ms(cases[first_ok]["lag"])
    # every interval individually, also past the first success
    for c in cases:
        ret, lag, coef = ac.cross_correlation(src[:2 * c["L"]], smp[:c["L"]])
        assert ret == c["ret"] and (ret == 0 and coef >= 0.95) == c["success"]
        if c["margin"] > 1e-4:
            assert lag == c["lag"]


@pytest.mark.parametrize("L,where", [(10, "source"), (1000, "sample"), (6000, "source"), (144000, "sample"),
                                     (144000, "source")])
def test_nan_input_behaves_like_the_reference(ac, capi, L, where):
    """A NaN anywhere in the inputs makes every r[i] NaN.  Reference :52-67: the seed r[0] = NaN
    is never beaten (`fabs(x) > NaN` is false), so idx = 0, lag = 0; the Pearson sums are NaN and
    the NaN gate (:276) returns -1 with both outputs written.  All three GPU paths must agree."""
    src, smp = capi.synth_pair(SEED + 21, 0, L)
    src = src.copy(); smp = smp.copy()
    (src if where == "source" else smp)[L // 3] = np.nan
    o = capi.cross_correlation(src, smp)
    assert (o["ret"], o["lag"]) == (-1, 0) and o["coef"] != o["coef"]
    ret, lag, coef = ac.cross_correlation(src, smp)
    assert (ret, lag) == (-1, 0) and coef != coef
    with ac.Context([0]) as c:
        for npdt, dt in ((np.float32, ac.F32), (np.float64, ac.F64)):
            s1 = np.ascontiguousarray(src, npdt); p1 = np.ascontiguousarray(smp, npdt)
            rec = c.xcorr_batch_records(s1.ctypes.data, p1.ctypes.data, 1, L, dt, ac.HOST)
            assert int(rec["ret"][0]) == -1 and int(rec["lag"][0]) == 0 and int(rec["raw_index"][0]) == 0
            assert rec["coef"][0] != rec["coef"][0] and int(rec["success"][0]) == 0
            assert float(rec["second"][0]) == 0.0                     # NaNs never count (oracle: second = 0)


# ------------------------------------------------------------------ interval-schedule residency

def _schedule_case(capi, pid):
    cases = sorted((c for c in SYNTH["cases"] if c["tag"] == "interval-prefix" and c["pair_id"] == pid),
                   key=lambda c: c["L"])
    src, smp = capi.synth_pair(cases[0]["seed"], pid, 1440000)
    assert [c["L"] for c in cases] == [3 * 48000, 6 * 48000, 10 * 48000, 15 * 48000, 20 * 48000, 30 * 48000]
    return src, smp, cases


@pytest.mark.parametrize("pid", [0, 6])
def test_residency_uploads_only_new_frames_and_matches(ac, capi, pid):
    """SURVEY 8f rank 1: with the source in an fftw_alloc_real buffer (reference
    src/audiosync.c:189) the six growing calls of the interval loop (:226-259) upload every
    frame exactly once -- 3 * 1,440,000 doubles in total instead of 3 * sum(L) -- and return
    exactly what the non-resident calls return."""
    src, smp, cases = _schedule_case(capi, pid)
    Ls = ac.INTERV_SAMPLE
    with ac.RealBuffer(2 * Ls[-1]) as sb, ac.RealBuffer(Ls[-1]) as mb:
        sb.array[:] = src; mb.array[:] = smp
        out = {}
        for resident in (False, True):
            ac.set_residency(resident)
            c0, b0, h0 = ac.dropin_stats()
            res = [ac.cross_correlation_ptr(sb.ptr, mb.ptr, L) for L in Ls]
            c1, b1, h1 = ac.dropin_stats()
            out[resident] = (res, c1 - c0, b1 - b0, h1 - h0)
        ac.set_residency(False)
    assert out[False][0] == out[True][0]                       # identical (ret, lag, coef), bit for bit
    assert out[False][1:] == (6, 8 * 3 * sum(Ls), 0)
    assert out[True][1:] == (6, 8 * 3 * Ls[-1], 5)            # first call opens the session, five reuse it
    for (ret, lag, coef), c in zip(out[True][0], cases):
        assert ret == c["ret"] and (ret == 0 and coef >= 0.95) == c["success"]
        if c["margin"] > 1e-4:
            assert lag == c["lag"] and close(coef, c["coef"])


def test_residency_guards(ac, capi):
    """A session is reused only for the same buffers, a strictly larger sample_len, an unchanged
    allocator generation and matching prefix fingerprints; everything else re-uploads."""
    L1, L2 = 144000, 288000
    src, smp = capi.synth_pair(SEED, 1, L2)
    src_b, smp_b = capi.synth_pair(SEED, 2, L2)
    ac.set_residency(True)
    with ac.RealBuffer(2 * L2) as sb, ac.RealBuffer(L2) as mb:
        def hits():
            return ac.dropin_stats()[2]
        sb.array[:] = src; mb.array[:] = smp
        ref1 = ac.cross_correlation(src[:2 * L1], smp[:L1]); ref2 = ac.cross_correlation(src, smp)
        h = hits()
        assert ac.cross_correlation_ptr(sb.ptr, mb.ptr, L1) == ref1 and hits() == h
        assert ac.cross_correlation_ptr(sb.ptr, mb.ptr, L2) == ref2 and hits() == h + 1
        # same length again / shorter length: no reuse (a new run of the loop starts over)
        assert ac.cross_correlation_ptr(sb.ptr, mb.ptr, L2) == ref2 and hits() == h + 1
        assert ac.cross_correlation_ptr(sb.ptr, mb.ptr, L1) == ref1 and hits() == h + 1
        # the buffers are refilled with another recording between two growing calls
        sb.array[:] = src_b; mb.array[:] = smp_b
        assert ac.cross_correlation_ptr(sb.ptr, mb.ptr, L2) == ac.cross_correlation(src_b, smp_b)
        assert hits() == h + 1
        # a free anywhere in between bumps the allocator generation
        assert ac.cross_correlation_ptr(sb.ptr, mb.ptr, L1) == ac.cross_correlation(src_b[:2 * L1], smp_b[:L1])
        ac.RealBuffer(16).free()
        assert ac.cross_correlation_ptr(sb.ptr, mb.ptr, L2) == ac.cross_correlation(src_b, smp_b)
        assert hits() == h + 1
    # a source that is not a library allocation is never cached
    h = ac.dropin_stats()[2]
    a = np.ascontiguousarray(src); b = np.ascontiguousarray(smp)
    ac.cross_correlation_ptr(a.ctypes.data, b.ctypes.data, L1)
    ac.cross_correlation_ptr(a.ctypes.data, b.ctypes.data, L2)
    assert ac.dropin_stats()[2] == h
    ac.set_residency(False)


def test_default_reads_the_host_buffers_on_every_call(ac, capi):
    """Reference semantics (src/cross_correlation.c reads its arguments afresh on every call):
    residency is opt-in, so with the default setting an in-place edit of ONE already-submitted
    sample between two growing calls on the same library-allocated buffers is seen.  The edit
    plants an impulse pair that dominates the correlation at a known lag."""
    L1, L2 = 144000, 288000
    src, smp = capi.synth_pair(SEED, 4, L2)
    with ac.RealBuffer(2 * L2) as sb, ac.RealBuffer(L2) as mb:
        sb.array[:] = src; mb.array[:] = smp
        h0 = ac.dropin_stats()[2]
        first = ac.cross_correlation_ptr(sb.ptr, mb.ptr, L1)
        assert first == ac.cross_correlation(src[:2 * L1], smp[:L1])
        # one sample of each prefix rewritten in place: a huge coincident impulse at lag 777
        sb.array[1000 + 777] = 1.0e6; mb.array[1000] = 1.0e6
        edited_src = np.array(sb.array); edited_smp = np.array(mb.array)
        second = ac.cross_correlation_ptr(sb.ptr, mb.ptr, L2)
        o = capi.cross_correlation(edited_src, edited_smp)
        assert o["lag"] == 777
        assert second[:2] == (o["ret"], o["lag"]) and close(second[2], o["coef"])
        assert ac.dropin_stats()[2] == h0                      # no resident session was used


# ------------------------------------------------------------------ second peak / torch surface

@pytest.mark.parametrize("L", [10, 12, 250, 1000, 3600, 6000, 144000])
def test_second_peak_all_paths_vs_oracle(ac, capi, L):
    """direct (fp64), single-CTA FFT and four-step paths all report the oracle's `second`."""
    n = 4
    srcs = np.empty((n, 2 * L), np.float64); smps = np.empty((n, L), np.float64)
    for i in range(n):
        srcs[i], smps[i] = capi.synth_pair(SEED + 11, i, L)
    with ac.Context([0]) as c:
        for path in ((ac.PATH_AUTO, ac.PATH_DIRECT) if L < 144000 else (ac.PATH_AUTO,)):
            c.set_path(path)
            rec = c.xcorr_batch_records(srcs.ctypes.data, smps.ctypes.data, n, L, ac.F64, ac.HOST)
            for i in range(n):
                o = capi.cross_correlation(srcs[i], smps[i])
                assert int(rec["raw_index"][i]) == o["raw_index"] and int(rec["lag"][i]) == o["lag"]
                assert close(float(rec["peak"][i]), o["peak"])
                assert abs(float(rec["second"][i]) - o["second"]) <= RTOL * o["second"] + 1e-6 * abs(o["peak"])
                # peak quality (SURVEY 8f rank 4): margin and normalised correlation vs the NumPy restatement
                assert abs(float(rec["margin"][i]) - o["margin"]) <= 1e-4
                assert close(float(rec["ncc"][i]), o["ncc"])


@pytest.mark.parametrize("dtype_name", ["f32", "f64"])
def test_peak_quality_both_lag_signs_and_degenerate_windows(ac, ctx, capi, dtype_name):
    """margin / ncc of the result records (oracle/xcorr_numpy.py: peak_quality).  Positive lags: ncc
    is the cosine similarity of the aligned windows; negative lags use the shorter window of
    cross_correlation.c:256-263; an empty window (idx == L) gives peak / 0 = inf, an all-zero one 0 / 0 = NaN."""
    from oracle import xcorr_numpy
    npdt = np.float32 if dtype_name == "f32" else np.float64
    dt = ac.F32 if dtype_name == "f32" else ac.F64
    L, n = 144000, 8
    srcs = np.empty((n, 2 * L), npdt); smps = np.empty((n, L), npdt)
    for i in range(n):
        srcs[i], smps[i] = capi.synth_pair(SEED + 17, i, L, npdt)
    rec = ctx.xcorr_batch_records(srcs.ctypes.data, smps.ctypes.data, n, L, dt, ac.HOST)
    signs = set()
    for i in range(n):
        o = xcorr_numpy.cross_correlation(srcs[i].astype(np.float64), smps[i].astype(np.float64))
        assert int(rec["raw_index"][i]) == o["raw_index"]
        signs.add(o["lag"] >= 0)
        assert abs(float(rec["margin"][i]) - o["margin"]) <= 1e-4 and 0.9 < o["margin"] <= 1.0
        assert close(float(rec["ncc"][i]), o["ncc"])
        if o["lag"] >= 0:
            assert -1.0 <= float(rec["ncc"][i]) <= 1.0
    assert signs == {True, False}
    # empty window (idx == L) and all-zero sample: NaN, like the coefficient
    src = np.zeros((1, 2 * L), npdt); smp = np.zeros((1, L), npdt); smp[0, 0] = 1.0; src[0, L] = 1.0
    r = ctx.xcorr_batch_records(src.ctypes.data, smp.ctypes.data, 1, L, dt, ac.HOST)
    assert int(r["raw_index"][0]) == L and np.isinf(r["ncc"][0]) and float(r["margin"][0]) > 0.9999   # peak / 0
    smp[:] = 0
    r = ctx.xcorr_batch_records(src.ctypes.data, smp.ctypes.data, 1, L, dt, ac.HOST)
    assert float(r["peak"][0]) == 0.0 and float(r["margin"][0]) == 0.0 and r["ncc"][0] != r["ncc"][0]


def test_second_peak_of_a_tie_equals_the_peak(ac):
    """Two equal maxima: the first index wins (reference :52-67) and the second peak equals the
    peak, i.e. margin 0 -- exactly the case the parity precondition excludes."""
    L = 8
    src = np.zeros(2 * L); smp = np.zeros(L)
    src[3] = 1.0; src[9] = 1.0; smp[0] = 1.0           # r[3] == r[9]
    with ac.Context([0]) as c:
        rec = c.xcorr_batch_records(src.ctypes.data, smp.ctypes.data, 1, L, ac.F64, ac.HOST)
    assert int(rec["raw_index"][0]) == 3 and float(rec["second"][0]) == abs(float(rec["peak"][0])) > 0


def test_torch_zero_copy_batch(ac, ctx, capi):
    """SURVEY 8f rank 3: CUDA tensors in, records out, on torch's current stream, no copies."""
    import torch
    L, n = 144000, 6
    gold = {c["pair_id"]: c for c in _pairs() if c["L"] == L}
    for tdt, dt in ((torch.float32, ac.F32), (torch.float64, ac.F64)):
        src = torch.empty(n, 2 * L, dtype=tdt, device="cuda:0"); smp = torch.empty(n, L, dtype=tdt, device="cuda:0")
        ctx.synth_pairs(0, SEED, 0, n, L, dt, src.data_ptr(), smp.data_ptr())
        ctx.synchronize(0)
        rec = ctx.xcorr_batch_torch(src, smp)                       # default stream
        st = torch.cuda.Stream("cuda:0")
        with torch.cuda.stream(st):
            out = ctx.xcorr_batch_torch(src, smp, sync=False)        # side stream, stream-ordered
            host = out.cpu()
        st.synchronize()
        rec2 = host.numpy().view(ac.RESULT_DTYPE)
        for name in ac.RESULT_DTYPE.names:
            assert np.array_equal(rec[name], rec2[name], equal_nan=True), name
        for pid, c in gold.items():
            if pid < n:
                assert int(rec["lag"][pid]) == c["lag"] and int(rec["ret"][pid]) == c["ret"]
                assert close(float(rec["coef"][pid]), c["coef"]) and second_close(float(rec["second"][pid]), c)
    with pytest.raises(ValueError):
        ctx.xcorr_batch_torch(src[:, ::2], smp[:, ::2])              # non-contiguous: refused, not copied
    with pytest.raises(TypeError):
        ctx.xcorr_batch_torch(src.half(), smp.half())


# ------------------------------------------------------------------ session pool

def test_session_pool_matches_dropin_over_the_schedule(ac, capi):
    """SURVEY 8f rank 1, second half: five concurrent sessions whose audio arrives in pieces;
    at every interval of the schedule (src/audiosync.c:50-70) ONE batched call evaluates all of
    them from their device-resident buffers.  F64 slots must return exactly what
    cross_correlation() returns on the same prefixes; each frame crosses PCIe once."""
    Ls = ac.INTERV_SAMPLE[:4]                      # 144,000 .. 720,000: all four kernel plans
    n, Lmax = 5, Ls[-1]
    data = [capi.synth_pair(SEED + 31, pid, Lmax) for pid in range(n)]
    with ac.Context([0]) as c, ac.SessionPool(c, 0, n + 1, Lmax, ac.F64) as pool:
        prev = 0
        for L in Ls:
            for slot, (src, smp) in enumerate(data):
                # ragged arrival: the source in two pieces, the sample in one
                mid = 2 * prev + (2 * L - 2 * prev) // 3
                pool.append(slot + 1, src[2 * prev:mid], None)
                pool.append(slot + 1, src[mid:2 * L], smp[prev:L])
                assert pool.fill(slot + 1) == (2 * L, L)
            rec = pool.run(1, n, L)
            for slot, (src, smp) in enumerate(data):
                ret, lag, coef = ac.cross_correlation(src[:2 * L], smp[:L])
                assert (int(rec["ret"][slot]), int(rec["lag"][slot])) == (ret, lag)
                assert float(rec["coef"][slot]) == coef                  # same kernels, same doubles
                o = capi.cross_correlation(src[:2 * L], smp[:L])
                assert lag == o["lag"] and close(coef, o["coef"]) and close(float(rec["peak"][slot]), o["peak"])
            prev = L
        # an interval the slots have not reached yet, an empty slot, an overflow
        with pytest.raises(ac.AudiosyncCudaError):
            pool.run(0, 2, Ls[0])                                         # slot 0 is empty
        with pytest.raises(ac.AudiosyncCudaError):
            pool.append(1, np.zeros(8), None)                             # slot 1 is full
        pool.reset(1)
        assert pool.fill(1) == (0, 0)


def test_session_pool_async_append_is_ordered(ac, capi):
    """Stream-ordered appends (pinned source buffers, no host synchronisation between them) followed
    directly by run(): the batch call orders itself behind every pending copy / conversion, for F64
    and F32 slots, and returns what the synchronous path returns."""
    L, n = 288000, 4
    data = [capi.synth_pair(SEED + 33, pid, L) for pid in range(n)]
    for dt in (ac.F64, ac.F32):
        with ac.Context([0]) as c, ac.SessionPool(c, 0, n, L, dt) as pa, ac.SessionPool(c, 0, n, L, dt) as ps, \
                ac.RealBuffer(2 * L) as sb, ac.RealBuffer(L) as mb:
            for slot, (src, smp) in enumerate(data):
                ps.append(slot, src, smp)                                   # synchronous reference
            ref = ps.run(0, n, L)
            for slot, (src, smp) in enumerate(data):
                pa.flush()                                                  # the pinned buffers are about to be rewritten
                sb.array[:] = src; mb.array[:] = smp
                half = L // 2
                pa.append_ptr(slot, sb.ptr, 2 * half, mb.ptr, half)         # two pieces, ragged, back to back
                pa.append_ptr(slot, sb.ptr + 16 * half, 2 * (L - half), mb.ptr + 8 * half, L - half)
            rec = pa.run(0, n, L)                                           # no flush: run orders itself
            for name in ("lag", "ret", "raw_index", "coef", "peak"):
                assert np.array_equal(rec[name], ref[name], equal_nan=True), name
            for slot in range(n):
                assert int(rec["lag"][slot]) == capi.synth_true_lag(SEED + 33, slot, L)


def test_session_pool_fp32_slots(ac, capi):
    """F32 slots convert the f64le frames on arrival: same lag, coefficient within tolerance."""
    L, n = 144000, 3
    data = [capi.synth_pair(SEED + 32, pid, L) for pid in range(n)]
    with ac.Context([0]) as c, ac.SessionPool(c, 0, n, L, ac.F32) as pool:
        for slot, (src, smp) in enumerate(data):
            pool.append(slot, src, smp)
        rec = pool.run(0, n, L)
    for slot, (src, smp) in enumerate(data):
        o = capi.cross_correlation(src, smp)
        assert int(rec["lag"][slot]) == o["lag"] == capi.synth_true_lag(SEED + 32, slot, L)
        assert int(rec["ret"][slot]) == o["ret"] and close(float(rec["coef"][slot]), o["coef"])


# ------------------------------------------------------------------ host batch API

@pytest.mark.parametrize("npdt", [np.float32, np.float64])
def test_host_batch_api(ac, ctx, capi, npdt):
    L, n = 144000, 7
    srcs = np.empty((n, 2 * L), npdt); smps = np.empty((n, L), npdt)
    for i in range(n):
        srcs[i], smps[i] = capi.synth_pair(SEED, i, L, npdt)
    r = ctx.xcorr_batch(srcs, smps)
    gold = {c["pair_id"]: c for c in _pairs() if c["L"] == L}
    for i in range(n):
        assert r["lags"][i] == capi.synth_true_lag(SEED, i, L)
        if i in gold:
            assert r["rets"][i] == gold[i]["ret"] and close(r["coefs"][i], gold[i]["coef"])
            assert close(r["peaks"][i], gold[i]["peak"])


def _narrow_case(capi, L, n, seed):
    s64 = np.empty((n, 2 * L), np.float64); p64 = np.empty((n, L), np.float64)
    for i in range(n):
        s64[i], p64[i] = capi.synth_pair(seed, i, L)            # fp32-exact values
    return s64, p64


def _records_equal(ac, a, b):
    for name in ac.RESULT_DTYPE.names:
        assert np.array_equal(a[name], b[name], equal_nan=True), name


@pytest.mark.parametrize("L,n", [(480000, 24), (6000, 300), (1000, 40), (100000, 9)])
def test_lossless_host_narrowing_is_bit_identical(ac, capi, L, n):
    """Default mode of the F64 HOST batch call: pairs whose doubles are exact images of floats cross
    PCIe as fp32 (narrowed by the copy threads) while others go up as doubles, and EVERY field of
    every record equals the un-narrowed call's -- static plans, runtime-radix plans, the single-CTA
    and the time-domain kernels; pinned (fed both ways at once) and pageable (all narrowed) inputs."""
    s64, p64 = _narrow_case(capi, L, n, SEED + 80)
    with ac.Context([0]) as c:
        c.set_host_narrowing(ac.NARROW_OFF)
        ref = c.xcorr_batch_records(s64.ctypes.data, p64.ctypes.data, n, L, ac.F64, ac.HOST)
        c.set_host_narrowing(ac.NARROW_LOSSLESS)
        c.host_feed_stats(reset=True)
        got = c.xcorr_batch_records(s64.ctypes.data, p64.ctypes.data, n, L, ac.F64, ac.HOST)      # pageable
        assert c.host_feed_stats(reset=True) == (0, n)                                             # every pair narrowed
        with ac.RealBuffer(n * 2 * L) as sb, ac.RealBuffer(n * L) as mb:                           # pinned
            sb.array[:] = s64.reshape(-1); mb.array[:] = p64.reshape(-1)
            got_pinned = c.xcorr_batch_records(sb.ptr, mb.ptr, n, L, ac.F64, ac.HOST)
        as_doubles, narrowed = c.host_feed_stats(reset=True)
        assert as_doubles + narrowed == n
        units = -(-n // max(1, (32 << 20) // (3 * L * 8)))             # the chunk is fed in units of ~32 MB of doubles
        if ac.copy_threads() >= 8 and units >= 2:
            assert narrowed > 0                                                                    # fed both ways
        else:
            assert narrowed == 0                                                                   # one unit / too few threads: copy engine only
    _records_equal(ac, got, ref)
    _records_equal(ac, got_pinned, ref)
    for i in range(0, n, max(1, n // 5)):
        assert int(ref["lag"][i]) == capi.synth_true_lag(SEED + 80, i, L)


@pytest.mark.parametrize("where", ["first", "middle", "last_pair_sample", "nan"])
def test_lossless_host_narrowing_gives_up_on_inexact_values(ac, capi, where):
    """One double that is not the image of a float -- anywhere in the batch -- and the records still
    equal the un-narrowed call's bit for bit (that chunk and all later ones go up as doubles)."""
    L, n = 144000, 130                     # several upload chunks, pinned and pageable
    s64, p64 = _narrow_case(capi, L, n, SEED + 81)
    if where == "first":
        s64[0, 5] += 2.0 ** -40
    elif where == "middle":
        s64[n // 2, L] = np.pi / 8
    elif where == "last_pair_sample":
        p64[n - 1, L - 1] += 2.0 ** -33
    else:
        p64[n // 3, 17] = np.nan
    with ac.Context([0]) as c:
        c.set_host_narrowing(ac.NARROW_OFF)
        ref = c.xcorr_batch_records(s64.ctypes.data, p64.ctypes.data, n, L, ac.F64, ac.HOST)
        c.set_host_narrowing(ac.NARROW_LOSSLESS)
        got = c.xcorr_batch_records(s64.ctypes.data, p64.ctypes.data, n, L, ac.F64, ac.HOST)
        with ac.RealBuffer(n * 2 * L) as sb, ac.RealBuffer(n * L) as mb:
            sb.array[:] = s64.reshape(-1); mb.array[:] = p64.reshape(-1)
            got_pinned = c.xcorr_batch_records(sb.ptr, mb.ptr, n, L, ac.F64, ac.HOST)
            again = c.xcorr_batch_records(sb.ptr, mb.ptr, n, L, ac.F64, ac.HOST)
    _records_equal(ac, got, ref)
    _records_equal(ac, got_pinned, ref)
    _records_equal(ac, again, ref)
    if where == "nan":
        assert int(ref["ret"][n // 3]) == -1


def test_host_narrowing_always_equals_the_fp32_batch(ac, capi):
    """NARROW_ALWAYS: an f64 HOST batch converted to fp32 while it is staged returns, bit for bit,
    what the fp32 batch of the rounded values returns (pinned and pageable sources, more than one
    ring buffer per pair), and stays within tolerance of the f64 path."""
    L, n = 480000, 5
    s64, p64 = _narrow_case(capi, L, n, SEED + 80)
    s64 *= 1.0 + 2.0 ** -30                                 # no longer exact in fp32
    p64 *= 1.0 - 2.0 ** -31
    s32, p32 = s64.astype(np.float32), p64.astype(np.float32)
    with ac.Context([0]) as c:
        ref32 = c.xcorr_batch_records(s32.ctypes.data, p32.ctypes.data, n, L, ac.F32, ac.HOST)
        ref64 = c.xcorr_batch_records(s64.ctypes.data, p64.ctypes.data, n, L, ac.F64, ac.HOST)    # lossless: gives up
        c.set_host_narrowing(ac.NARROW_ALWAYS)
        got = c.xcorr_batch_records(s64.ctypes.data, p64.ctypes.data, n, L, ac.F64, ac.HOST)      # pageable
        with ac.RealBuffer(n * 2 * L) as sb, ac.RealBuffer(n * L) as mb:                           # pinned
            sb.array[:] = s64.reshape(-1); mb.array[:] = p64.reshape(-1)
            got_pinned = c.xcorr_batch_records(sb.ptr, mb.ptr, n, L, ac.F64, ac.HOST)
        c.set_precise(True)                                                                        # precise mode ignores it
        assert "fp64" in c.describe_plan(L)
    _records_equal(ac, got, ref32)
    _records_equal(ac, got_pinned, ref32)
    for i in range(n):
        assert int(got["lag"][i]) == int(ref64["lag"][i]) == capi.synth_true_lag(SEED + 80, i, L)
        assert close(float(got["coef"][i]), float(ref64["coef"][i]), 1e-6)


def test_host_batch_multi_chunk_and_wave_sizes(ac, capi):
    """More pairs than one upload chunk / one kernel wave; every wave size gives the same answer."""
    L, n = 6000, 300
    srcs = np.empty((n, 2 * L), np.float32); smps = np.empty((n, L), np.float32)
    for i in range(n):
        srcs[i], smps[i] = capi.synth_pair(SEED + 3, i, L, np.float32)
    base = None
    for wave in (0, 1, 7, 64):
        with ac.Context([0]) as c:
            c.set_wave_pairs(wave)
            r = c.xcorr_batch(srcs, smps)
        for i in range(n):
            assert r["lags"][i] == capi.synth_true_lag(SEED + 3, i, L)
        if base is None:
            base = r
        else:
            for k in base:
                assert np.array_equal(base[k], r[k], equal_nan=True)   # deterministic


def test_multi_device_dispatcher_matches_single_device(ac, capi):
    """SURVEY 8e: the in-library dispatcher shards contiguous pair blocks over every visible
    GPU (one host thread + stream per device, host gather); results must be identical to the
    single-device run, in pair order.  Needs >= 2 GPUs (the 1-GPU box skips it)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    L, n = 144000, 11                                   # odd count: uneven blocks
    srcs = np.empty((n, 2 * L), np.float32); smps = np.empty((n, L), np.float32)
    for i in range(n):
        srcs[i], smps[i] = capi.synth_pair(SEED + 5, i, L, np.float32)
    with ac.Context([0]) as c:
        one = c.xcorr_batch(srcs, smps)
    with ac.Context(None) as c:
        assert c.device_count() == torch.cuda.device_count()
        many = c.xcorr_batch(srcs, smps)
    for k in one:
        assert np.array_equal(one[k], many[k], equal_nan=True), k
    assert [int(x) for x in many["lags"]] == [capi.synth_true_lag(SEED + 5, i, L) for i in range(n)]


# ------------------------------------------------------------------ full-size properties

def test_full_size_batch_recovers_injected_lags(ac, ctx, capi):
    """L = 1,440,000 (BASELINE configs 3-5): a batch generated on the device; the recovered
    lag must equal the injected one and success must follow the generator's noise level."""
    L, n, first = 1440000, 48, 100
    res, _, _ = _batch_on_device(ac, ctx, SEED, first, n, L)
    for i in range(n):
        pid = first + i
        assert int(res["lag"][i]) == capi.synth_true_lag(SEED, pid, L)
        assert int(res["ret"][i]) == 0
        assert bool(res["success"][i]) == (pid % 4 != 3)
        c = float(res["coef"][i])
        assert (0.994 < c < 0.996) if pid % 4 != 3 else (0.79 < c < 0.81)


def test_full_size_shift_property(ac, ctx):
    """L = 1,440,000, independent of the oracle: r[j] = N * sum_n source[(n + j) mod N] * sample[n], so
    rotating the source by d rotates r by d -- the raw index must move by exactly d (mod 2L), the
    peak and the second peak must stay (to fp32 rounding), for shifts that cross the fold boundary
    idx = L in both directions."""
    import torch
    L, n = 1440000, 6
    res0, d_src, d_smp = _batch_on_device(ac, ctx, SEED + 60, 0, n, L)
    src = d_src.view(n, 2 * L)
    shifts = [1, -1, 12345, L, L + 7, -(L // 3)]
    rolled = torch.stack([torch.roll(src[i], shifts[i]) for i in range(n)]).contiguous()
    rec = ctx.xcorr_batch_torch(rolled, d_smp.view(n, L))
    for i in range(n):
        want = (int(res0["raw_index"][i]) + shifts[i]) % (2 * L)
        assert int(rec["raw_index"][i]) == want
        assert int(rec["lag"][i]) == (want if want < L else want - 2 * L)
        assert close(float(rec["peak"][i]), float(res0["peak"][i]), 1e-5)
        assert abs(float(rec["second"][i]) - float(res0["second"][i])) <= 1e-5 * abs(float(res0["peak"][i]))


def test_scaling_and_negation_properties(ac, ctx, capi):
    """r is bilinear: scaling the sample by a power of two scales the peak exactly and leaves
    lag and coefficient unchanged; negating it flips the peak sign and the coefficient."""
    L = 480000
    src, smp = capi.synth_pair(SEED, 5, L, np.float32)
    srcs = np.stack([src, src, src]); smps = np.stack([smp, smp * np.float32(4.0), -smp])
    r = ctx.xcorr_batch(srcs, smps)
    assert r["lags"][0] == r["lags"][1] == r["lags"][2]
    assert r["peaks"][1] == 4.0 * r["peaks"][0] and r["peaks"][2] == -r["peaks"][0]
    assert close(r["coefs"][1], r["coefs"][0], 1e-12) and close(r["coefs"][2], -r["coefs"][0], 1e-12)


def test_identical_windows_give_exactly_one(ac, capi):
    """coef == 1.0 exactly when the windows are identical (reference T1 at real sizes)."""
    for L in (1000, 144000):
        src, _ = capi.synth_pair(SEED, 2, L)
        for lag in (0, 17):
            smp = src[lag:lag + L].copy()
            ret, got, coef = ac.cross_correlation(src, smp)
            assert ret == 0 and got == lag and coef == 1.0


# ------------------------------------------------------------------ allocator + threads

def test_pinned_allocator_roundtrip(ac, capi):
    import ctypes
    L = 144000
    lib = ac.lib()
    p = lib.fftw_alloc_real(2 * L)
    assert p
    buf = np.ctypeslib.as_array((ctypes.c_double * (2 * L)).from_address(p))
    src, smp = capi.synth_pair(SEED, 0, L)
    buf[:] = src
    ret, lag, coef = ac.cross_correlation(buf, smp)
    assert ret == 0 and lag == capi.synth_true_lag(SEED, 0, L)
    del buf
    lib.fftw_free(p)


def test_concurrent_callers(ac, capi):
    """Eight threads, three calls each, more callers than slots: every answer equals the
    single-threaded one (each caller leases its own stream / mirrors / scratch)."""
    L = 144000
    pairs = [capi.synth_pair(SEED, i, L) for i in range(4)]
    single = [ac.cross_correlation(*p) for p in pairs]
    out = [[None] * 3 for _ in range(8)]

    def work(t):
        for k in range(3):
            out[t][k] = ac.cross_correlation(*pairs[(t + k) % 4])

    ac.dropin_max_inflight(reset=True)
    th = [threading.Thread(target=work, args=(t,)) for t in range(8)]
    [t.start() for t in th]
    [t.join() for t in th]
    assert ac.dropin_max_inflight() >= 2            # callers overlapped on the GPU, no global lock
    for t in range(8):
        for k in range(3):
            i = (t + k) % 4
            assert out[t][k] == single[i]
            assert out[t][k][0] == 0 and out[t][k][1] == capi.synth_true_lag(SEED, i, L)


def test_streams_may_be_mixed_on_one_context(ac, ctx, capi):
    """Stream-ordered device calls on DIFFERENT streams share the context's scratch: each call is
    ordered behind the previous user of it, so back-to-back calls on two side streams (and the
    library's own stream) without any host synchronisation all return the single-stream answers."""
    import torch
    L, n = 144000, 6
    src = torch.empty(3, n * 2 * L, dtype=torch.float32, device="cuda:0")
    smp = torch.empty(3, n * L, dtype=torch.float32, device="cuda:0")
    res = torch.zeros(3, n * ac.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda:0")
    for k in range(3):
        ctx.synth_pairs(0, SEED + 40 + k, 0, n, L, ac.F32, src[k].data_ptr(), smp[k].data_ptr())
    ctx.synchronize(0)
    streams = [torch.cuda.Stream("cuda:0"), torch.cuda.Stream("cuda:0")]
    for rep in range(4):
        for k in range(3):
            st = streams[k].cuda_stream if k < 2 else 0
            ctx.xcorr_batch_device(0, src[k].data_ptr(), smp[k].data_ptr(), n, L, ac.F32, res[k].data_ptr(), st)
    torch.cuda.synchronize()
    ctx.synchronize(0)
    for k in range(3):
        r = res[k].cpu().numpy().view(ac.RESULT_DTYPE)
        for i in range(n):
            assert int(r["lag"][i]) == capi.synth_true_lag(SEED + 40 + k, i, L) and int(r["ret"][i]) == 0


def test_profile_and_launch_accounting(ac, capi):
    L, n = 144000, 16
    with ac.Context([0]) as c:
        c.profile_enable(True)
        before = c.launch_count()
        res, _, _ = _batch_on_device(ac, c, SEED, 0, n, L)
        prof = c.profile_read()
        assert c.launch_count() > before
    for k in ("col_fwd", "row_fused", "col_inv_argmax", "pearson"):
        assert prof[k][0] >= 1 and prof[k][1] > 0.0, (k, prof)


# ------------------------------------------------------------------ staging / launch variants
_VARIANT_SNIPPET = r"""
import sys, json
sys.path.insert(0, {root!r}); sys.path.insert(0, {pkg!r})
import numpy as np, torch
import audiosync_cuda as ac
L, n, off = {L}, 5, {off}
with ac.Context([0]) as c:
    d_src = torch.empty(n * 2 * L + off, dtype=torch.float32, device="cuda:0")
    d_smp = torch.empty(n * L, dtype=torch.float32, device="cuda:0")
    d_res = torch.zeros(n * ac.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda:0")
    src = d_src.data_ptr() + 4 * off
    c.synth_pairs(0, {seed}, 0, n, L, ac.F32, src, d_smp.data_ptr())
    c.xcorr_batch_device(0, src, d_smp.data_ptr(), n, L, ac.F32, d_res.data_ptr())
    c.synchronize(0)
    r = d_res.cpu().numpy().view(ac.RESULT_DTYPE)
print(json.dumps({{k: [float(x).hex() for x in r[k]] for k in ("raw_index", "lag", "peak", "coef", "second", "ret")}}))
"""


@pytest.mark.parametrize("L", [144000, 1440000])
def test_staging_and_launch_variants_are_bit_identical(L):
    """The TMA-staged column tiles with programmatic dependent launch (default), the first column
    pass loading through registers (source base 8 bytes off a 16-byte boundary) and plain
    stream-ordered launches run the same arithmetic: every field of the result records must agree
    bit for bit.  The offset is two floats, not one: the register path loads float2."""
    import subprocess
    import sys
    root = os.path.dirname(HERE)
    outs = []
    for extra, off in (({}, 0), ({}, 2), ({"AUDIOSYNC_CUDA_NO_PDL": "1"}, 0)):
        code = _VARIANT_SNIPPET.format(root=root, pkg=os.path.join(root, "old-audiosync_b200"), L=L, seed=SEED, off=off)
        env = dict(os.environ, **extra)
        p = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stderr[-2000:]
        outs.append(json.loads(p.stdout.strip().splitlines()[-1]))
    assert outs[0] == outs[1] == outs[2]
    assert all(float.fromhex(x) == 0.0 for x in outs[0]["ret"])


def test_full_size_peak_and_coefficient_from_first_principles(ac, ctx):
    """L = 1,440,000, independent of the oracle: at the lag the kernels report, the peak must be
    the circular correlation sum itself (reference src/cross_correlation.c:232-239: c2r of the
    product is N * sum_n source[(n + idx) mod N] * sample_pad[n]) and the coefficient the
    Pearson coefficient of the reference's windows (:256-271, :74-116), both evaluated here in
    fp64 with torch on the device from the same inputs."""
    import torch
    L, n, first = 1440000, 12, 40
    res, d_src, d_smp = _batch_on_device(ac, ctx, SEED, first, n, L)
    signs = set()
    for i in range(n):
        src = d_src[i * 2 * L:(i + 1) * 2 * L].double()
        smp = d_smp[i * L:(i + 1) * L].double()
        idx, lag = int(res["raw_index"][i]), int(res["lag"][i])
        assert lag == (idx if idx < L else idx - 2 * L)
        signs.add(lag >= 0)
        # peak: N * sum_n source[(n + idx) mod N] * sample[n], n < L
        rolled = torch.roll(src, -idx)[:L]
        peak = 2.0 * L * float(torch.dot(rolled, smp))
        assert abs(float(res["peak"][i]) - peak) <= RTOL * abs(peak)
        # coefficient over the reference's windows
        if lag >= 0:
            x, y = src[lag:lag + L], smp
        else:
            x, y = src[:L + lag], smp[-lag:]
        dx, dy = x - x.mean(), y - y.mean()
        coef = float(torch.dot(dx, dy) / torch.sqrt(torch.dot(dx, dx) * torch.dot(dy, dy)))
        assert abs(float(res["coef"][i]) - coef) <= 1e-6 * abs(coef)
        # nothing else in r reaches the peak: spot-check a few hundred other lags
        g = torch.Generator(device="cpu").manual_seed(i)
        for j in torch.randint(0, 2 * L, (8,), generator=g).tolist():
            if j != idx:
                other = 2.0 * L * float(torch.dot(torch.roll(src, -j)[:L], smp))
                assert abs(other) <= float(res["second"][i]) * (1 + 1e-3) + 1e-6 * abs(peak)
    assert signs == {True, False}      # both lag signs were exercised
