"""PHAT weighting (audiosync_cuda_set_weighting) on the GPU.

Every path against the fp64 NumPy restatement (tests/golden/phat_oracle.py) in batches of 128 pairs
over four waves, then bit-identity of the records across dtypes, memspaces, host narrowing, streams,
devices, the session pool and power-of-two input scaling, and the setting's toggling and refusals.
"""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import phat_oracle as po  # noqa: E402

pytestmark = pytest.mark.gpu

N_PAIRS, WAVE = 128, 32
ORACLE_PAIRS_LONG = 8          # pairs checked against the NumPy oracle above 65,536 frames (all below)
ORACLE_LENGTHS = (144000, 288000, 480000, 720000, 960000, 1440000,
                  24000, 48000, 192000, 1000000, 1048576, 1000, 4096, 6000)


@pytest.fixture(scope="module")
def ac():
    import audiosync_cuda
    return audiosync_cuda


def ctx_for(ac, weighting=1, precise=False, devices=(0,)):
    c = ac.Context(list(devices) if devices is not None else None)
    c.set_weighting(weighting)
    c.set_precise(precise)
    c.set_wave_pairs(WAVE)
    return c


def device_pairs(L, n, seed, dtype=None):
    """n delayed white-noise pairs on cuda:0 (sample = source[lag:lag + L] + 0.3 noise), fp32."""
    import torch
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    src = torch.randn(n, 2 * L, device="cuda:0", generator=g)
    lags = torch.randint(0, L, (n, 1), device="cuda:0", generator=g)
    idx = lags + torch.arange(L, device="cuda:0")[None, :]
    smp = torch.gather(src, 1, idx) + 0.3 * torch.randn(n, L, device="cuda:0", generator=g)
    return src.contiguous(), smp.contiguous()


def same(a, b):
    return a.tobytes() == b.tobytes()


@pytest.mark.parametrize("L", ORACLE_LENGTHS)
def test_every_path_against_oracle(ac, L):
    """fp32 and precise mode, 128 pairs in waves of 32: precise within 1e-9 relative of the oracle,
    and the fp32 raw_index equal to the precise one on every pair."""
    import torch
    src, smp = device_pairs(L, N_PAIRS, seed=L)
    with ctx_for(ac) as c32, ctx_for(ac, precise=True) as c64:
        assert c32.describe_plan(L).endswith(" phat") and c64.describe_plan(L).endswith(" phat")
        r32 = c32.xcorr_batch_torch(src, smp)
        r64 = c64.xcorr_batch_torch(src, smp)
    torch.cuda.synchronize()
    assert np.array_equal(r32["raw_index"], r64["raw_index"])
    assert np.array_equal(r32["lag"], r64["lag"])
    N = 2 * L
    assert np.all(np.abs(r32["peak"] - r64["peak"]) <= 1e-6 * N)
    hs, hm = src.cpu().numpy().astype(np.float64), smp.cpu().numpy().astype(np.float64)
    for i in range(N_PAIRS if L <= 65536 else ORACLE_PAIRS_LONG):
        o = po.phat_record(hs[i], hm[i])
        g = r64[i]
        assert int(g["raw_index"]) == o["raw_index"] and int(g["lag"]) == o["lag"], (i, g, o)
        for f in ("peak", "second", "ncc"):
            assert abs(float(g[f]) - o[f]) <= 1e-9 * max(abs(o[f]), 1e-300) + 1e-12 * (N if f != "ncc" else 1), (i, f, g[f], o[f])
        assert abs(float(g["coef"]) - o["coef"]) <= 1e-5 * abs(o["coef"])      # fp32 inputs: the fp32 Pearson path
        assert abs(float(g["ncc"]) - float(g["peak"]) / N) == 0.0


@pytest.mark.parametrize("L", [144000, 4096, 24000])
def test_all_zero_sample_matches_none_but_ncc(ac, L):
    import torch
    src, _ = device_pairs(L, 2, seed=3)
    smp = torch.zeros(2, L, device="cuda:0")
    with ctx_for(ac) as cp, ctx_for(ac, weighting=0) as cn:
        rp = cp.xcorr_batch_torch(src, smp)
        rn = cn.xcorr_batch_torch(src, smp)
    for f in rp.dtype.names:
        if f != "ncc":
            assert np.array_equal(rp[f], rn[f], equal_nan=True), f
    assert np.all(rp["ncc"] == 0.0)


@pytest.mark.parametrize("L,precise", [(144000, False), (4096, False), (24000, False), (24000, True)])
def test_s16_equals_f64(ac, L, precise):
    import torch
    g = torch.Generator(device="cuda:0").manual_seed(L)
    s = (torch.randn(4, 2 * L, device="cuda:0", generator=g) * 6000).clamp(-32768, 32767).round().to(torch.int16)
    lag = L // 3
    m = (s[:, lag:lag + L].float() + torch.randn(4, L, device="cuda:0", generator=g) * 1500).clamp(-32768, 32767).round().to(torch.int16).contiguous()
    with ctx_for(ac, precise=precise) as c:
        a = c.xcorr_batch_torch(s, m)
        b = c.xcorr_batch_torch(s.double() / 32768.0, m.double() / 32768.0)
    assert same(a, b)


def test_host_memspaces_narrowing_and_pool(ac):
    """HOST pageable and pinned against DEVICE (F32); LOSSLESS host narrowing against NARROW_OFF and the
    session pool against the batch call (F64 of fp32-exact values)."""
    import torch
    L, n = 144000, 6
    src, smp = device_pairs(L, n, seed=11)
    with ctx_for(ac) as c:
        dev = c.xcorr_batch_torch(src, smp)
        hs, hm = src.cpu().numpy(), smp.cpu().numpy()
        page = c.xcorr_batch_records(hs.ctypes.data, hm.ctypes.data, n, L, ac.F32, ac.HOST)
        ps, pm = torch.from_numpy(hs).pin_memory(), torch.from_numpy(hm).pin_memory()
        pinned = c.xcorr_batch_records(ps.data_ptr(), pm.data_ptr(), n, L, ac.F32, ac.HOST)
        assert same(dev, page) and same(dev, pinned)
        ds, dm = hs.astype(np.float64), hm.astype(np.float64)
        c.host_feed_stats(reset=True)
        narrowed = c.xcorr_batch_records(ds.ctypes.data, dm.ctypes.data, n, L, ac.F64, ac.HOST)
        assert c.host_feed_stats(reset=True)[1] > 0
        c.set_host_narrowing(ac.NARROW_OFF)
        plain = c.xcorr_batch_records(ds.ctypes.data, dm.ctypes.data, n, L, ac.F64, ac.HOST)
        assert same(narrowed, plain)
        with ac.SessionPool(c, 0, n, L, ac.F64) as pool:
            for i in range(n):
                pool.append(i, ds[i], dm[i])
            assert same(pool.run(0, n, L), plain)


def test_non_default_stream(ac):
    import torch
    L = 48000
    src, smp = device_pairs(L, 8, seed=12)
    with ctx_for(ac) as c:
        ref = c.xcorr_batch_torch(src, smp)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            got = c.xcorr_batch_torch(src, smp)
    assert same(ref, got)


def test_multi_device_split(ac):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("one GPU")
    L, n = 144000, 5
    src, smp = device_pairs(L, n, seed=13)
    hs, hm = src.cpu().numpy(), smp.cpu().numpy()
    with ctx_for(ac) as one, ctx_for(ac, devices=None) as many:
        assert many.device_count() >= 2
        assert same(one.xcorr_batch_records(hs.ctypes.data, hm.ctypes.data, n, L, ac.F32, ac.HOST),
                    many.xcorr_batch_records(hs.ctypes.data, hm.ctypes.data, n, L, ac.F32, ac.HOST))


@pytest.mark.parametrize("L", [144000, 4096, 48000])
def test_power_of_two_scaling_is_invariant(ac, L):
    src, smp = device_pairs(L, 4, seed=14)
    with ctx_for(ac) as c:
        a = c.xcorr_batch_torch(src, smp)
        b = c.xcorr_batch_torch((src * 0.125).contiguous(), (smp * 32.0).contiguous())
    assert same(a, b)


def test_toggle_matches_fresh_contexts(ac):
    L = 144000
    src, smp = device_pairs(L, 4, seed=15)
    with ctx_for(ac, weighting=0) as fn, ctx_for(ac, weighting=1) as fp, ctx_for(ac, weighting=0) as t:
        none, phat = fn.xcorr_batch_torch(src, smp), fp.xcorr_batch_torch(src, smp)
        assert not same(none, phat)
        assert same(t.xcorr_batch_torch(src, smp), none)
        assert not t.describe_plan(L).endswith("phat")
        t.set_weighting(ac.WEIGHT_PHAT)
        assert same(t.xcorr_batch_torch(src, smp), phat)
        assert t.describe_plan(L).endswith(" phat")
        t.set_weighting(ac.WEIGHT_NONE)
        assert same(t.xcorr_batch_torch(src, smp), none)


def test_refusals(ac):
    import torch
    with ctx_for(ac) as c:
        with pytest.raises(ac.AudiosyncCudaError):
            c.set_weighting(7)
        for L in (100001, 1440002):
            src, smp = torch.zeros(1, 2 * L, device="cuda:0"), torch.zeros(1, L, device="cuda:0")
            out = torch.full((64,), 0xAB, dtype=torch.uint8, device="cuda:0")
            with pytest.raises(ac.AudiosyncCudaError, match="2/3/5-smooth"):
                c.xcorr_batch_device(0, src.data_ptr(), smp.data_ptr(), 1, L, ac.F32, out.data_ptr())
            torch.cuda.synchronize()
            assert bool((out == 0xAB).all())                        # no output written
            with pytest.raises(ac.AudiosyncCudaError):
                c.describe_plan(L)
        c.set_path(ac.PATH_DIRECT)
        L = 4096
        src, smp = device_pairs(L, 1, seed=16)
        with pytest.raises(ac.AudiosyncCudaError, match="PATH_DIRECT"):
            c.xcorr_batch_torch(src, smp)
