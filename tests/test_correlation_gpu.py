"""Correlation export (audiosync_cuda_xcorr_correlation) on the GPU.

The records must be the non-exporting calls' byte for byte on every plan kind, dtype, weighting and
lag window, in both memspaces and with a shared source.  The exported values must be the kernel's own:
the reference argmax rule over them reproduces raw_index, peak and second bit for bit (near-ties,
negative-r[0] probes, an all-NaN pair), they pass tests/golden/xcorr_error.py's per-lag bound, and at
a lag k they equal the peak of a one-lag window [k, k].  Sub-ranges are slices of the full export;
rows land in place across waves, chunks, devices, offsets and streams; host narrowing keeps them; the
refusals write nothing.
"""
import json
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import hard_cases  # noqa: E402
import lagwin_oracle as lo  # noqa: E402
import probes as pr  # noqa: E402
import xcorr_error as xe  # noqa: E402

pytestmark = pytest.mark.gpu

AUTO, DIRECT = 0, 2
PATHS = [("static", 144000, AUTO, False), ("single_cta", 4096, AUTO, False),
         ("radix_smooth", 24000, AUTO, False), ("radix_static_rows", 48000, AUTO, False),
         ("radix_embedded", 100001, AUTO, False), ("direct", 4096, DIRECT, False),
         ("precise", 24000, AUTO, True)]
PHAT_PATHS = {"static", "single_cta", "radix_smooth", "radix_static_rows", "precise"}
EXACT_PATHS = {"direct", "precise"}
DTYPES = ("f32", "f64", "s16")


@pytest.fixture(scope="module")
def ac():
    import audiosync_cuda
    return audiosync_cuda


def ctx_for(ac, path=AUTO, precise=False, phat=False, window=None, devices=(0,), wave=16):
    c = ac.Context(list(devices) if devices is not None else None)
    c.set_path(path)
    c.set_precise(precise)
    c.set_weighting(ac.WEIGHT_PHAT if phat else ac.WEIGHT_NONE)
    c.set_wave_pairs(wave)
    if window is not None:
        c.set_lag_window(*window)
    return c


def pairs(L, n, seed):
    """n delayed noise pairs (fp32 on cuda:0)."""
    import torch
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    src = torch.randn(n, 2 * L, device="cuda:0", generator=g)
    lag = torch.randint(0, L, (n, 1), device="cuda:0", generator=g)
    smp = torch.gather(src, 1, lag + torch.arange(L, device="cuda:0")[None, :])
    smp = smp + 0.3 * torch.randn(n, L, device="cuda:0", generator=g)
    return src.contiguous(), smp.contiguous(), lag.view(-1).tolist()


def as_dtype(src, smp, dt):
    import torch
    if dt == "f32":
        return src, smp
    if dt == "f64":
        return src.double(), smp.double()
    q = lambda t: (t * 6000).clamp(-32768, 32767).round().to(torch.int16).contiguous()   # noqa: E731
    return q(src), q(smp)


def same(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


def plain_call(c, s, m, memspace, shared):
    """Records of the non-exporting call."""
    if memspace == "device":
        return c.xcorr_shared_source_torch(s[0], m) if shared else c.xcorr_batch_torch(s, m)
    hs, hm = s.cpu().numpy(), m.cpu().numpy()
    if shared:
        return c.xcorr_shared_source(hs[0], hm)
    return c.xcorr_batch_records(hs.ctypes.data, hm.ctypes.data, hm.shape[0], hm.shape[1],
                                 {np.float32: 0, np.float64: 1, np.int16: 2}[hs.dtype.type], 0)


def export_call(c, s, m, memspace, shared, lo_=None, hi_=None):
    """(records, corr as a NumPy [n, W] array) of the exporting call."""
    if memspace == "device":
        rec, corr = c.xcorr_correlation_torch(s[0] if shared else s, m, lo_, hi_, shared_source=shared)
        return rec, corr.cpu().numpy()
    hs, hm = s.cpu().numpy(), m.cpu().numpy()
    return c.xcorr_correlation(hs[0] if shared else hs, hm, lo_, hi_, shared_source=shared)


def raw_order(corr, L):
    lags = np.arange(-L, L)
    r = np.empty(corr.shape[:-1] + (2 * L,))
    r[..., np.where(lags >= 0, lags, lags + 2 * L)] = corr
    return r


def self_consistent(rec, corr, L, window):
    """The reference argmax rule over the exported values reproduces each record exactly."""
    raw = lo.allowed_raw(*(lo.effective(*window, L) if window else (-L, L - 1)), L)
    r = raw_order(corr, L)
    for i in range(len(rec)):
        idx, second = lo.windowed_argmax(r[i], raw)
        assert idx == int(rec["raw_index"][i]), (i, idx, int(rec["raw_index"][i]))
        assert same(r[i][idx], rec["peak"][i]) or (np.isnan(r[i][idx]) and np.isnan(rec["peak"][i])), \
            (i, r[i][idx], rec["peak"][i])
        assert same(np.float64(second), rec["second"][i]), (i, second, rec["second"][i])
        if window is None or lo.effective(*window, L) == (-L, L - 1):
            lag = int(rec["lag"][i])
            assert same(corr[i][lag + L], rec["peak"][i]) or np.isnan(rec["peak"][i])


# ----------------------------------------------------------------------------- 1 + 2: records, self-consistency
@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("name,L,path,precise", PATHS, ids=[p[0] for p in PATHS])
def test_records_identical_and_self_consistent(ac, name, L, path, precise, phat):
    if phat and name not in PHAT_PATHS:
        pytest.skip("PHAT needs a transform at N = 2L")
    src, smp, lags = pairs(L, 3, seed=L + 7)
    src[1:] = src[0]                     # one source for all: the shared-source call reads the same pairs
    for window in (None, (lags[0] - 500, lags[0] + 700)):
        with ctx_for(ac, path, precise, phat, window=window) as c:
            for dt in DTYPES:
                s, m = as_dtype(src, smp, dt)
                for memspace in ("device", "host"):
                    for shared in (False, True):
                        want = plain_call(c, s, m, memspace, shared)
                        rec, corr = export_call(c, s, m, memspace, shared)
                        assert same(rec, want), (dt, memspace, shared, window)
                        assert corr.shape == (3, 2 * L)
                        self_consistent(rec, corr, L, window)


def plan_of(c, kind_name, L):
    if kind_name == "static":
        return pr.STATIC_PLANS[L]
    if kind_name in ("single_cta", "direct"):
        return pr.single_cta_plan(L)
    return pr.parse_plan(L, c.describe_plan(L))


@pytest.mark.parametrize("name,L,path,precise", PATHS, ids=[p[0] for p in PATHS])
def test_self_consistent_on_hard_inputs(ac, name, L, path, precise):
    """Near-ties of tests/golden/hard.json (at their own lengths, on the plan kind where they fit),
    the negative-r[0] probes of family D, and an all-NaN pair."""
    import torch
    with ctx_for(ac, path, precise) as c:
        batch = []
        for probe in pr.seed_probes(plan_of(c, name, L), seed=11):
            batch.append(probe.build(np.float32))
        s = np.stack([b[0] for b in batch]); m = np.stack([b[1] for b in batch])
        nan_s = np.full((1, 2 * L), np.nan, np.float32); nan_m = np.full((1, L), np.nan, np.float32)
        s = np.concatenate([s, nan_s]); m = np.concatenate([m, nan_m])
        ts, tm = torch.from_numpy(s).cuda(), torch.from_numpy(m).cuda()
        rec, corr = export_call(c, ts, tm, "device", False)
        assert same(rec, plain_call(c, ts, tm, "device", False))
        self_consistent(rec, corr, L, None)
        assert np.isnan(rec["peak"][-1])
    cases = [cs for cs in json.load(open(os.path.join(HERE, "golden", "hard.json")))["cases"] if cs["L"] == L]
    if name == "static":
        cases = cases[:6]
    for cs in cases:
        hs, hm = hard_cases.build(cs, np.float64)
        with ctx_for(ac, path, precise) as c:
            rec, corr = c.xcorr_correlation(hs[None, :], hm[None, :])
            self_consistent(rec, corr, L, None)


# ----------------------------------------------------------------------------- 3: accuracy
@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("name,L,path,precise", PATHS, ids=[p[0] for p in PATHS])
def test_accuracy_and_one_lag_windows(ac, name, L, path, precise, phat):
    if phat and name not in PHAT_PATHS:
        pytest.skip("PHAT needs a transform at N = 2L")
    exact = name in EXACT_PATHS
    for family in (("s16", "s16_white") if exact else ("delayed", "white", "brown")):
        p = xe.make_pair(family, L, seed=5)
        if exact and not phat:
            r = xe.exact_reference(p.src_int, p.smp_int)
        else:
            r = xe.reference(p.src, p.smp, phat=phat)
        with ctx_for(ac, path, precise, phat) as c:
            rec, corr = c.xcorr_correlation(p.src[None, :], p.smp[None, :])
            got = raw_order(corr, L)[0]
            res = xe.judge(np.arange(2 * L), got, r, fp64=exact or precise,
                           yard=None if exact or precise else xe.yardstick(p.src, p.smp, phat=phat), phat=phat)
            assert res["ok"], "%s %s: %s" % (name, family, res["msg"])
            for k in (0, 1, L - 1, -L, -1, min(int(rec["lag"][0]) + 3, L - 1), 12345 % L):
                c.set_lag_window(k, k)
                one = c.xcorr_batch_records(p.src.ctypes.data, p.smp.ctypes.data, 1, L, ac.F64, ac.HOST)
                assert same(one["peak"][0], corr[0][k + L]), (k, one["peak"][0], corr[0][k + L])


# ----------------------------------------------------------------------------- 4: ranges
@pytest.mark.parametrize("name,L,path,precise", PATHS, ids=[p[0] for p in PATHS])
def test_sub_ranges_are_slices(ac, name, L, path, precise):
    src, smp, lags = pairs(L, 3, seed=L + 3)
    with ctx_for(ac, path, precise, window=(lags[0] - 100, lags[0] + 100)) as c:
        full = export_call(c, src, smp, "device", False)[1]
        for lo_, hi_ in ((-L, -L + 40), (L - 41, L - 1), (-70, 90), (33, 33), (-L, L - 1),
                         (-L // 2 - 50, -L // 2 + 50), (5, 3000)):
            rec, corr = export_call(c, src, smp, "device", False, lo_, hi_)
            assert corr.shape == (3, hi_ - lo_ + 1)
            assert same(corr, full[:, lo_ + L: hi_ + L + 1]), (lo_, hi_)


# ----------------------------------------------------------------------------- 5: layout
def test_rows_land_in_place(ac):
    import torch
    L = 24000
    src, smp, _ = pairs(L, 40, seed=99)
    with ctx_for(ac, wave=16) as c:
        rec_all, full = export_call(c, src, smp, "device", False)
        # each pair alone gives its row: several waves put every row in place
        for i in (0, 15, 16, 17, 39):
            rec_i, row = export_call(c, src[i:i + 1], smp[i:i + 1], "device", False)
            assert same(row[0], full[i]) and same(rec_i, rec_all[i:i + 1]), i
        # odd-offset device inputs (views at element offset 1)
        big_s = torch.zeros(40 * 2 * L + 1, device="cuda:0"); big_m = torch.zeros(40 * L + 1, device="cuda:0")
        big_s[1:] = src.view(-1); big_m[1:] = smp.view(-1)
        d_res = torch.zeros(40 * 64, dtype=torch.uint8, device="cuda:0")
        d_corr = torch.full((40 * 2 * L,), 7.0, dtype=torch.float64, device="cuda:0")
        c.xcorr_correlation_device(0, big_s[1:].data_ptr(), big_m[1:].data_ptr(), 40, L, ac.F32, -L, L - 1,
                                   d_res.data_ptr(), d_corr.data_ptr())
        c.synchronize(0)
        assert same(d_corr.cpu().numpy().reshape(40, 2 * L), full)
        # a non-default torch stream
        st = torch.cuda.Stream()
        with torch.cuda.stream(st):
            rec_s, corr_s = c.xcorr_correlation_torch(src, smp)
        st.synchronize()
        assert same(corr_s.cpu().numpy(), full) and same(rec_s, rec_all)
        # host calls: pageable and pinned corr, at least three chunks (rows of 23 MB at 1.44M)
        hs, hm = src.cpu().numpy(), smp.cpu().numpy()
        rec_h, corr_h = c.xcorr_correlation(hs, hm)
        assert same(corr_h, full) and same(rec_h, rec_all)
        pinned = torch.empty((40, 2 * L), dtype=torch.float64).pin_memory()
        res = np.zeros(40, ac.RESULT_DTYPE)
        assert ac.lib().audiosync_cuda_xcorr_correlation(c.handle, hs.ctypes.data, hm.ctypes.data, 40, L, ac.F32, ac.HOST,
                                                          0, -L, L - 1, res.ctypes.data, pinned.data_ptr()) == 0
        assert same(pinned.numpy(), full) and same(res, rec_all)
    # F64 host pairs at 1.44M frames with the full range: 23 + 11.5 MB of input and 23 MB of staged
    # export per pair, three pairs per chunk, three chunks
    Lb, n = 1440000, 9
    p2 = [xe.make_pair("delayed", Lb, i) for i in range(2)]
    s9 = np.stack([p2[i % 2].src for i in range(n)]); m9 = np.stack([p2[i % 2].smp for i in range(n)])
    with ctx_for(ac, wave=0) as c:
        rec, corr = c.xcorr_correlation(s9, m9)
        want = c.xcorr_batch_records(s9.ctypes.data, m9.ctypes.data, n, Lb, ac.F64, ac.HOST)
        assert same(rec, want)
        rec_d, corr_d = export_call(c, torch.from_numpy(s9[:2]).cuda(), torch.from_numpy(m9[:2]).cuda(), "device", False)
        for i in range(n):
            assert same(corr[i], corr_d[i % 2]), i
    # every device of the machine
    if torch.cuda.device_count() > 1:
        with ctx_for(ac, devices=None) as c:
            rec_g, corr_g = c.xcorr_correlation(hs, hm)
        assert same(corr_g, full) and same(rec_g, rec_all)


# ----------------------------------------------------------------------------- 6: host narrowing
def test_lossless_narrowing_keeps_the_export(ac):
    L = 48000
    src, smp, _ = pairs(L, 6, seed=5)
    hs, hm = src.double().cpu().numpy(), smp.double().cpu().numpy()      # fp32-exact doubles
    with ctx_for(ac) as c:
        c.set_host_narrowing(ac.NARROW_LOSSLESS)
        c.host_feed_stats(reset=True)
        rec_on, corr_on = c.xcorr_correlation(hs, hm, -3000, 3000)
        c.set_host_narrowing(ac.NARROW_OFF)
        rec_off, corr_off = c.xcorr_correlation(hs, hm, -3000, 3000)
    assert same(rec_on, rec_off) and same(corr_on, corr_off)


# ----------------------------------------------------------------------------- 7: refusals
def test_refusals_write_nothing(ac):
    import torch
    L = 4096
    src, smp, _ = pairs(L, 2, seed=1)
    hs, hm = src.cpu().numpy(), smp.cpu().numpy()
    lib = ac.lib()

    def host(lo_, hi_, corr=True, ctx=None):
        res = np.zeros(2, ac.RESULT_DTYPE).view(np.uint8)
        res[:] = 0xA5
        cbuf = np.full(2 * max(hi_ - lo_ + 1, 1), 3.25)
        rc = lib.audiosync_cuda_xcorr_correlation(ctx.handle, hs.ctypes.data, hm.ctypes.data, 2, L, ac.F32, ac.HOST, 0,
                                                  lo_, hi_, res.ctypes.data, cbuf.ctypes.data if corr else None)
        return rc, bool((res == 0xA5).all()), bool((cbuf == 3.25).all())

    with ctx_for(ac) as c:
        for lo_, hi_ in ((5, 4), (-L - 1, 0), (0, L), (-L - 5, L + 5)):
            assert host(lo_, hi_, ctx=c) == (-1, True, True), (lo_, hi_)
            assert "range" in ac.last_error()
        assert host(0, 3, corr=False, ctx=c)[:2] == (-1, True)
        c.set_lag_window(10 * L, 11 * L)                 # empty lag window: the batch call's refusal
        assert host(0, 3, ctx=c) == (-1, True, True)
    with ctx_for(ac, phat=True, path=DIRECT) as c:       # PHAT on the direct path is refused
        assert host(0, 3, ctx=c) == (-1, True, True)
    with ctx_for(ac) as c:
        d_res = torch.full((2 * 64,), 0xA5, dtype=torch.uint8, device="cuda:0")
        d_corr = torch.full((2 * 8 + 1,), 3.25, dtype=torch.float64, device="cuda:0")
        odd = d_corr.data_ptr() + 4                      # not 8-byte aligned
        assert lib.audiosync_cuda_xcorr_correlation_device(c.handle, 0, src.data_ptr(), smp.data_ptr(), 2, L, ac.F32, 0,
                                                           0, 7, d_res.data_ptr(), odd, None) == -1
        assert lib.audiosync_cuda_xcorr_correlation_device(c.handle, 0, src.data_ptr() + 2, smp.data_ptr(), 2, L, ac.F32, 0,
                                                           0, 7, d_res.data_ptr(), d_corr.data_ptr(), None) == -1
        c.synchronize(0)
        assert bool((d_res == 0xA5).all()) and bool((d_corr == 3.25).all())
        n0 = c.launch_count()
        assert lib.audiosync_cuda_xcorr_correlation(c.handle, hs.ctypes.data, hm.ctypes.data, 0, L, ac.F32, ac.HOST, 0,
                                                    0, 7, None, None) == 0
        assert c.launch_count() == n0
