"""Closed-form probes (tests/golden/probes.py) through the CUDA kernels on the device.

Per length, a batch of at least 128 probes -- every frequency-bin class, output-position class,
second-peak placement and signed-seed case -- runs device-resident through xcorr_batch_device in
waves of 48 pairs, so the probes sit at different places in the launch order of the column
kernels (the running second peak of a pair is shared between its CTAs).  Every field of every
record is compared with the exact record of r[j] = N * source[(j + a) mod 2L]: raw index, lag
and ret exact, peak and second peak within 2e-6 of N * sum |spike|, coef, margin and ncc within
what those bounds imply.  A subset also runs through the F64 drop-in cross_correlation and
through precise (fp64-arithmetic) mode.
"""
import os
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import probes as pr  # noqa: E402
from test_gpu_parity import GEN_LENGTHS  # noqa: E402

from oracle.xcorr_numpy import MIN_CONFIDENCE  # noqa: E402

STATIC_LENGTHS = sorted(pr.STATIC_PLANS)
BATCH_MIN = 128
WAVE = 48


@pytest.fixture(scope="module")
def ac():
    import audiosync_cuda
    audiosync_cuda.lib()
    return audiosync_cuda


@pytest.fixture(scope="module")
def ctx(ac):
    c = ac.Context([0])
    c.set_wave_pairs(WAVE)
    yield c
    c.close()


def _plan(ctx, L):
    return pr.STATIC_PLANS[L] if L in pr.STATIC_PLANS else pr.parse_plan(L, ctx.describe_plan(L))


def _batch(plan, seed):
    """>= BATCH_MIN probes: all families (bins dense up to 300,000 frames, one per class above),
    filled up with more second-peak placements (cheap: spikes only)."""
    dense = plan.L <= 300000
    probes = pr.all_probes(plan, seed, dense=dense)
    k = 1
    while len(probes) < BATCH_MIN:
        probes += pr.second_probes(plan, seed + 100 + k)
        k += 1
    return probes


def _near(got, want, bound):
    """|got - want| <= bound; a non-finite expectation (an empty or zero-energy window) exactly."""
    if not np.isfinite(want):
        return got == want or (got != got and want != want)
    return abs(got - want) <= bound


def _check_record(p, exp, rec, tol):
    """'' or a description of every field of the record that misses the closed form."""
    idx = int(rec["raw_index"])
    exp = pr.resolve_tie(p, exp, idx, tol)
    msg = pr.check(p, exp, idx, float(rec["peak"]), float(rec["second"]), tol)
    errs = [msg] if msg else []
    if (int(rec["lag"]), int(rec["ret"])) != (exp["lag"], exp["ret"]):
        errs.append("lag/ret %d/%d != %d/%d" % (int(rec["lag"]), int(rec["ret"]), exp["lag"], exp["ret"]))
    # success = ret == 0 and coef >= MIN_CONFIDENCE (src/audiosync.c:254); either way within the
    # coef bound of the threshold
    succ = exp["ret"] == 0 and exp["coef"] >= MIN_CONFIDENCE
    if int(rec["success"]) != int(succ) and not abs(exp["coef"] - MIN_CONFIDENCE) <= 1e-6:
        errs.append("success %d != %d" % (int(rec["success"]), int(succ)))
    if not _near(float(rec["coef"]), exp["coef"], 1e-6):
        errs.append("coef %.12g vs %.12g" % (float(rec["coef"]), exp["coef"]))
    rel = tol * p.scale() / abs(exp["peak"])          # the peak / second bound relative to |peak|
    if not _near(float(rec["margin"]), exp["margin"], 3 * rel):
        errs.append("margin %.9g vs %.9g" % (float(rec["margin"]), exp["margin"]))
    if not _near(float(rec["ncc"]), exp["ncc"], 2 * rel * abs(exp["ncc"]) + 1e-12):
        errs.append("ncc %.9g vs %.9g" % (float(rec["ncc"]), exp["ncc"]))
    return "" if not errs else "%s a=%d: %s" % (p.name, p.a, "; ".join(errs))


@pytest.mark.parametrize("L", STATIC_LENGTHS + GEN_LENGTHS)
def test_probe_batch_on_device_matches_closed_form(ac, ctx, L):
    import torch
    plan = _plan(ctx, L)
    probes = _batch(plan, seed=L)
    n = len(probes)
    src = torch.empty((n, 2 * L), dtype=torch.float32)
    smp = torch.empty((n, L), dtype=torch.float32)
    exps = []
    for i, p in enumerate(probes):
        s, m = p.build(np.float32)
        src[i] = torch.from_numpy(s); smp[i] = torch.from_numpy(m)
        exps.append(p.expect(arrays=(s, m)))
    d_src, d_smp = src.cuda(), smp.cuda()
    d_res = torch.zeros(n * ac.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda:0")
    ctx.xcorr_batch_device(0, d_src.data_ptr(), d_smp.data_ptr(), n, L, ac.F32, d_res.data_ptr())
    ctx.synchronize(0)
    recs = d_res.cpu().numpy().view(ac.RESULT_DTYPE)
    bad = [m for m in (_check_record(p, e, r, pr.TOL_F32) for p, e, r in zip(probes, exps, recs)) if m]
    worst = max(pr.error_of(p, pr.resolve_tie(p, e, int(r["raw_index"]), pr.TOL_F32), float(r["peak"]), float(r["second"]))
                for p, e, r in zip(probes, exps, recs))
    print("L=%d %s: %d probes, worst peak/second error %.2e of N * sum|spike|" % (L, ctx.describe_plan(L)[:40], n, worst))
    assert not bad, "%d of %d probes (%s):\n  " % (len(bad), n, ctx.describe_plan(L)) + "\n  ".join(bad)


def _subset(plan, seed):
    """A few of each family: one bin per class is too many for the per-call paths; take the
    classes most likely to break (M/2, Nyquist, row 0), the position edges and the seed cases."""
    bins = [p for p in pr.bin_probes(plan, seed, n_random=1, dense=False)
            if any(t in p.name for t in ("M/2(", "nyquist", "row0", "stripe", "rand"))]
    pos = [p for p in pr.position_probes(plan, seed + 1) if any(t in p.name for t in ("B:0(", "B:L(", "B:2L-1", "recur"))]
    seeds = [p for p in pr.seed_probes(plan, seed + 3) if "0.99" in p.name or "shoulders" in p.name or "tie" in p.name]
    return bins + pos + pr.second_probes(plan, seed + 2)[:3] + seeds


@pytest.mark.parametrize("L", [144000, 1440000, 24000, 100001])
def test_probe_subset_dropin_f64_and_precise_mode(ac, L):
    """The F64 drop-in cross_correlation (ret, lag, coef) and precise mode (whole records, fp64
    arithmetic: peak and second within 1e-9 of N * sum |spike|) on a subset of the probes."""
    bad = []
    with ac.Context([0]) as cp:
        cp.set_precise(True)
        assert "fp64" in cp.describe_plan(L)
        plan = pr.parse_plan(L, cp.describe_plan(L))      # precise mode: runtime-radix plans only
        for p in _subset(plan, L + 7):
            s, m = p.build(np.float64)
            exp = p.expect(arrays=(s, m))            # the drop-in runs the fp32 kernels
            ret, lag, coef = ac.cross_correlation(s, m)
            cands = [exp] + [p.expect(i, (s, m)) for i in exp["tied"] if i != exp["raw_index"]]
            if not any((ret, lag) == (c["ret"], c["lag"]) and
                       _near(coef, c["coef"], 1e-6) for c in cands):
                bad.append("drop-in %s: ret/lag/coef %d/%d/%.12g, expected %d/%d/%.12g"
                           % (p.name, ret, lag, coef, exp["ret"], exp["lag"], exp["coef"]))
            rec = cp.xcorr_batch_records(s.ctypes.data, m.ctypes.data, 1, L, ac.F64, ac.HOST)[0]
            msg = _check_record(p, p.expect(arrays=(s, m), tol=pr.TOL_F64), rec, pr.TOL_F64)
            if msg:
                bad.append("precise " + msg)
    assert not bad, "\n  ".join(bad)
