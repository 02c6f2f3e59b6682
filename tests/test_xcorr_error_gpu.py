"""Every lag of the correlation r against an fp64 (or exact) reference, on every kind of plan.

No call writes r out; two properties of the public API read it at any lag:
  - a one-lag window [k, k] reports r[k] of the product kernels as the record's peak (raw_index k);
  - rotating the source by d (x'[m] = x[(m + d) mod 2L]) moves the lags: r'[k] = r[(k + d) mod 2L].
So one call with window k and B rotations of one source against the same sample reads B chosen lags
through output slot k.  Slots cover the fold edges, the first and last positions of rows, columns
and column tiles of the plan's layout and seeded random positions; the lags cover +-64 around the
peak, the peak's offsets by multiples of 2L/12 and seeded random lags (every lag for L <= 24,000).
Each lag read is held to tests/golden/xcorr_error.py's bound.  With XCORR_ERROR_REPORT set to a
file path, every case appends its measured ratios there as one JSON line.
"""
import functools
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import xcorr_error as xe  # noqa: E402

pytestmark = pytest.mark.gpu

AUTO, DIRECT = 0, 2
SLOTS, PER_SLOT = 512, 64            # lags read per case above 24,000 frames: SLOTS x PER_SLOT
EVERY_MAX_L = 24000                  # at and below: every lag of the base pair
STATIC_LS = (144000, 288000, 480000, 720000, 960000, 1440000)
FULL_LS = (144000, 1440000)          # every input family; white and delayed elsewhere


@pytest.fixture(scope="module")
def ac():
    import audiosync_cuda
    return audiosync_cuda


def ctx_for(ac, path=AUTO, precise=False, phat=False):
    c = ac.Context([0])
    c.set_path(path)
    c.set_precise(precise)
    c.set_weighting(ac.WEIGHT_PHAT if phat else ac.WEIGHT_NONE)
    c.set_wave_pairs(1024)
    return c


def plan_of(desc: str, L: int):
    if "generic four-step" in desc:
        return xe.parse_plan(L, desc)
    if L in xe.STATIC_PLANS and "static" in desc:
        return xe.STATIC_PLANS[L]
    return xe.single_cta_plan(L)


def _device_rows(t, odd):
    """t [B, n] as a contiguous tensor whose data starts at an odd element offset when `odd`."""
    import torch
    if not odd:
        return t.contiguous()
    buf = torch.empty(t.numel() + 1, dtype=t.dtype, device=t.device)
    buf[1:].copy_(t.reshape(-1))
    return buf[1:].view(t.shape)


def read_lags(c, src, smp, assignment, odd=False):
    """(lags, values): for each slot k, one call with window [k, k] over rotations of src (1-D
    device tensor [2L]) that put each assigned lag on slot k."""
    import torch
    N = src.shape[0]
    L = N // 2
    ar = torch.arange(N, device=src.device)
    lags, vals = [], []
    for k, want in assignment.items():
        want = np.asarray(want, np.int64)
        d = torch.as_tensor((want - k) % N, device=src.device)
        rot = _device_rows(src[(ar[None, :] + d[:, None]) % N], odd)
        smps = _device_rows(smp[None, :].expand(len(want), L), odd)
        w = k if k < L else k - N
        c.set_lag_window(w, w)
        rec = c.xcorr_batch_torch(rot, smps)
        assert (rec["raw_index"] == k).all(), (k, rec["raw_index"][:4])
        lags.append(want)
        vals.append(rec["peak"].astype(np.float64))
    c.set_lag_window()
    return np.concatenate(lags), np.concatenate(vals)


@functools.lru_cache(maxsize=2)
def base_case(family, L, seed, phat, exact):
    """(pair, reference r, float32 yardstick or None) of one base pair."""
    pair = xe.make_pair(family, L, seed)
    if exact and not phat:
        r = xe.exact_reference(pair.src_int, pair.smp_int)
    else:
        r = xe.reference(pair.src, pair.smp, phat)
    return pair, r, (None if exact else xe.yardstick(pair.src, pair.smp, phat))


def report(case, res):
    path = os.environ.get("XCORR_ERROR_REPORT")
    if path:
        with open(path, "a") as f:
            f.write(json.dumps(dict(case=case, **{k: v for k, v in res.items() if k != "msg"})) + "\n")


def run_case(ac, case, family, L, seed, path=AUTO, precise=False, phat=False, dtype="f32", exact=False, odd=False,
             slots=SLOTS, per_slot=PER_SLOT, every_slot=False):
    import torch
    N = 2 * L
    pair, r, yard = base_case(family, L, seed, phat, exact)
    tdt = torch.float32 if dtype == "f32" else torch.float64
    if dtype == "f32":
        assert xe.fp32_exact(pair)
    src = torch.tensor(pair.src, dtype=tdt, device="cuda:0")
    smp = torch.tensor(pair.smp, dtype=tdt, device="cuda:0")
    with ctx_for(ac, path, precise, phat) as c:
        plan = plan_of(c.describe_plan(L), L)
        # the one-lag readout is the product kernels' r: window [p, p] at the unwindowed call's raw
        # index p returns that call's peak bit for bit
        base = c.xcorr_batch_torch(src[None], smp[None])[0]
        p = int(base["raw_index"])
        c.set_lag_window(p if p < L else p - N, p if p < L else p - N)
        one = c.xcorr_batch_torch(src[None], smp[None])[0]
        assert int(one["raw_index"]) == p and one["peak"].tobytes() == base["peak"].tobytes(), (case, base, one)
        c.set_lag_window()
        peak = xe.xn.max_abs_index(r)
        if every_slot:
            sl = list(range(N))
            asg = xe.assign_lags(sl, per_slot, L, peak, seed=L, every=True)
        elif L <= EVERY_MAX_L:
            sl = xe.slots(plan, slots, seed=L)
            asg = xe.assign_lags(sl, max(per_slot, -(-N // len(sl)) + 1), L, peak, seed=L, every=True)
        else:
            sl = xe.slots(plan, slots, seed=L)
            asg = xe.assign_lags(sl, per_slot, L, peak, seed=L)
        lags, vals = read_lags(c, src, smp, asg, odd)
    if L <= EVERY_MAX_L:
        assert np.unique(lags).size == N
    res = xe.judge(lags, vals, r, fp64=exact or precise, yard=yard, phat=phat)
    report(case, res)
    assert res["ok"], "%s: %s" % (case, res["msg"])
    return res


# ----------------------------------------------------------------------------- static plans
STATIC_CASES = []
for _L in STATIC_LS:
    for _dt in ("f32", "f64"):
        for _fam in (xe.FAMILIES if _L in FULL_LS else ("white", "delayed")):
            if _fam == "f64" and _dt == "f32":
                continue
            STATIC_CASES.append((_L, _dt, _fam))


@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("L,dtype,family", STATIC_CASES, ids=["%d-%s-%s" % c for c in STATIC_CASES])
def test_static_plans(ac, L, dtype, family, phat):
    run_case(ac, "static-%d-%s-%s-%s" % (L, dtype, family, "phat" if phat else "none"),
             family, L, 1, phat=phat, dtype=dtype)


def test_static_odd_offset_view(ac):
    """An F32 view at an odd element offset: K_A loads through registers instead of TMA."""
    L = 144000
    run_case(ac, "static-144000-f32-odd-delayed", "delayed", L, 2, odd=True)


# ----------------------------------------------------------------------------- single-CTA kernel
@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("family", ["white", "delayed"])
@pytest.mark.parametrize("L", [4096, 6000])
def test_single_cta_every_slot(ac, L, family, phat):
    run_case(ac, "single_cta-%d-%s-%s" % (L, family, "phat" if phat else "none"), family, L, 3,
             phat=phat, per_slot=2, every_slot=True)


# ----------------------------------------------------------------------------- runtime-radix fp32
def small_threads_length(ac):
    """A short smooth length whose runtime-radix plan runs 64-thread CTAs."""
    with ctx_for(ac, path=1) as c:
        for L in (2048, 3000, 4000, 4800, 6400, 7200, 8000, 9600, 12000):
            d = c.describe_plan(L)
            if "generic four-step" in d and "threads=64/64" in d:
                return L
    pytest.fail("no short runtime-radix plan on 64-thread CTAs")


RADIX_LS = [24000, "small", 48000, 192000, 100001, 1440002, 1000000]


@pytest.mark.parametrize("family", ["white", "delayed"])
@pytest.mark.parametrize("L", RADIX_LS, ids=[str(x) for x in RADIX_LS])
def test_runtime_radix_fp32(ac, L, family):
    path = AUTO
    if L == "small":
        L, path = small_threads_length(ac), 1
    with ctx_for(ac, path) as c:
        desc = c.describe_plan(L)
    assert "generic four-step" in desc and desc.endswith("fp32"), desc
    phats = [False] + ([True] if "embedded" not in desc else [])
    for phat in phats:
        run_case(ac, "radix-%d-%s-%s" % (L, family, "phat" if phat else "none"), family, L, 4,
                 path=path, phat=phat)


# ----------------------------------------------------------------------------- fp64 paths, exact
@pytest.mark.parametrize("family", ["s16", "s16_white"])
@pytest.mark.parametrize("L", [144000, 1440000, 24000])
def test_precise_exact(ac, L, family):
    run_case(ac, "precise-%d-%s" % (L, family), family, L, 5, precise=True, dtype="f64",
             exact=True)


def test_precise_phat(ac):
    """fp64 PHAT against numpy's fp64 r_w (no exact form): the bound covers both errors."""
    run_case(ac, "precise-24000-delayed-phat", "delayed", 24000, 6, precise=True, phat=True,
             dtype="f64")


@pytest.mark.parametrize("family", ["s16", "s16_white"])
def test_direct_exact(ac, family):
    run_case(ac, "direct-4096-%s" % family, family, 4096, 7, path=DIRECT, dtype="f64", exact=True)
