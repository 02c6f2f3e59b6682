"""Lag window (audiosync_cuda_set_lag_window) on the GPU.

A window that holds every lag is the unwindowed call, byte for byte, on every path, dtype and
weighting.  Restricted windows are checked against the fp64 restatement in
tests/golden/lagwin_oracle.py, including windows that exclude the global peak.  The window also has
to hold across the other surfaces (HOST memspace, the session pool, streams, several devices), and
the setting's refusals and scope are checked.
"""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import lagwin_oracle as lo  # noqa: E402

pytestmark = pytest.mark.gpu

INT64_MIN, INT64_MAX = lo.INT64_MIN, lo.INT64_MAX
AUTO, DIRECT = 0, 2

# (name, L, forced path, precise): every kind of plan the batch calls run
PATHS = [("static", 144000, AUTO, False), ("single_cta", 4096, AUTO, False),
         ("radix_smooth", 24000, AUTO, False), ("radix_static_rows", 48000, AUTO, False),
         ("radix_embedded", 100001, AUTO, False), ("direct", 4096, DIRECT, False),
         ("precise", 24000, AUTO, True)]
PHAT_PATHS = {"static", "single_cta", "radix_smooth", "radix_static_rows", "precise"}
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


def pairs(L, n, seed, lags=None):
    """n delayed noise pairs (fp32 on cuda:0): sample = source[lag : lag + L] + 0.3 noise, lag in [0, L)."""
    import torch
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    src = torch.randn(n, 2 * L, device="cuda:0", generator=g)
    lag = torch.randint(0, L, (n, 1), device="cuda:0", generator=g) if lags is None else \
        torch.tensor(lags, device="cuda:0").view(n, 1)
    smp = torch.gather(src, 1, lag + torch.arange(L, device="cuda:0")[None, :])
    smp = smp + 0.3 * torch.randn(n, L, device="cuda:0", generator=g)
    return src.contiguous(), smp.contiguous(), lag.view(-1).tolist()


def as_dtype(src, smp, dt):
    """The same pairs as F32, F64 or S16 (S16 at 2^-15 scale: F64 of the widened values is its twin)."""
    import torch
    if dt == "f32":
        return src, smp
    if dt == "f64":
        return src.double(), smp.double()
    q = lambda t: (t * 6000).clamp(-32768, 32767).round().to(torch.int16).contiguous()   # noqa: E731
    return q(src), q(smp)


def same(a, b):
    return a.tobytes() == b.tobytes()


@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("name,L,path,precise", PATHS, ids=[p[0] for p in PATHS])
def test_full_windows_are_the_unwindowed_call(ac, name, L, path, precise, phat):
    if phat and name not in PHAT_PATHS:
        pytest.skip("PHAT needs a transform at N = 2L")
    src, smp, _ = pairs(L, 4, seed=L + 1)
    with ctx_for(ac, path, precise, phat) as ref:
        for dt in DTYPES:
            s, m = as_dtype(src, smp, dt)
            want = ref.xcorr_batch_torch(s, m)
            for w in ((INT64_MIN, INT64_MAX), (-L, L - 1), (-10 * L, 10 * L)):
                with ctx_for(ac, path, precise, phat, window=w) as c:
                    assert " lags=" not in c.describe_plan(L)
                    assert same(c.xcorr_batch_torch(s, m), want), (dt, w)


def check_against_oracle(got, src, smp, window, phat, exact):
    """got: records of the pairs; exact: fp64 arithmetic (fp32 otherwise: a near-tie within the
    rounding of the transform may resolve to the other index, which must then carry the same |r|)."""
    for i in range(len(got)):
        o = lo.record(src[i], smp[i], *window, phat=phat)
        g = got[i]
        scale = max(o["rmax"], 1e-300)
        tol = 1e-9 if exact else 1e-5
        if int(g["raw_index"]) != o["raw_index"]:
            assert not exact, (i, window, int(g["raw_index"]), o["raw_index"])
            alt = lo.record(src[i], smp[i], int(g["lag"]), int(g["lag"]), phat=phat)
            assert abs(abs(alt["peak"]) - abs(o["peak"])) <= tol * scale, (i, window, g, o)
            continue
        assert int(g["lag"]) == o["lag"]
        assert abs(float(g["peak"]) - o["peak"]) <= tol * scale, (i, window, float(g["peak"]), o["peak"])
        assert abs(float(g["second"]) - o["second"]) <= tol * scale, (i, window, float(g["second"]), o["second"])
        assert abs(float(g["coef"]) - o["coef"]) <= 1e-4, (i, float(g["coef"]), o["coef"])
        assert int(g["ret"]) == o["ret"]


@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("name,L,path,precise", PATHS, ids=[p[0] for p in PATHS])
def test_restricted_windows_against_oracle(ac, name, L, path, precise, phat):
    """Around the true lag, excluding it (the in-window maximum is reported), and around 0; F32 and
    F64 against the oracle, S16 equal to F64 of the widened values bit for bit."""
    if phat and name not in PHAT_PATHS:
        pytest.skip("PHAT needs a transform at N = 2L")
    n = 3
    lags = [L // 3, L // 2 + 7, 5]
    src, smp, _ = pairs(L, n, seed=L + 2, lags=lags)
    w = max(16, min(48000, L // 8))
    windows = [(lags[0] - w, lags[0] + w),               # holds the true lag of pair 0
               (lags[0] + 3, lags[0] + 3 + w),           # excludes it: the in-window maximum
               (-w, w),                                  # around lag 0: r[0] is the signed seed
               (-L, -L + w)]                             # only negative lags
    exact = precise or name == "direct"
    for window in windows:
        with ctx_for(ac, path, precise, phat, window=window) as c:
            assert c.describe_plan(L).endswith(" lags=[%d,%d]" % lo.effective(*window, L))
            for dt in ("f32", "f64"):
                s, m = as_dtype(src, smp, dt)
                got = c.xcorr_batch_torch(s, m)
                check_against_oracle(got, s.double().cpu().numpy(), m.double().cpu().numpy(), window, phat, exact)
            s16, m16 = as_dtype(src, smp, "s16")
            assert same(c.xcorr_batch_torch(s16, m16), c.xcorr_batch_torch(s16.double() / 32768.0, m16.double() / 32768.0))


@pytest.mark.parametrize("L", [144000, 4096, 24000])
def test_probe_peak_outside_window(ac, L):
    """Closed form: sample one-hot at 0, so r[j] = N source[j].  The largest |r| sits outside the
    window, a larger value just outside it never reaches `second`, and a huge |r[0]| outside it is
    neither the peak nor the second."""
    import torch
    N = 2 * L
    src = torch.zeros(1, N, dtype=torch.float64, device="cuda:0")
    smp = torch.zeros(1, L, dtype=torch.float64, device="cuda:0")
    smp[0, 0] = 1.0
    a, b = L // 4, L // 4 + 40                       # window [a, b]
    src[0, 0] = -50.0                                # r[0]: outside the window, huge
    src[0, a - 1] = 40.0                             # just outside: larger than anything inside
    src[0, a + 5] = 3.0                              # in-window peak
    src[0, a + 9] = -2.0                             # in-window second
    src[0, b + 1] = 30.0
    with ctx_for(ac, window=(a, b)) as c:
        r = c.xcorr_batch_torch(src, smp)[0]
    assert int(r["raw_index"]) == a + 5 and int(r["lag"]) == a + 5
    assert abs(float(r["peak"]) / N - 3.0) <= 1e-5
    assert abs(float(r["second"]) / N - 2.0) <= 1e-5


@pytest.mark.parametrize("L", [144000, 4096, 24000])
def test_probe_one_lag_windows(ac, L):
    """lo = hi = -L: empty Pearson window (ret -1, NaN coef); lo = hi = L - 1 and lo = hi = 0."""
    src, smp, _ = pairs(L, 2, seed=L + 3)
    for lag in (-L, L - 1, 0):
        with ctx_for(ac, window=(lag, lag)) as c:
            got = c.xcorr_batch_torch(src, smp)
        for g in got:
            assert int(g["lag"]) == lag
            assert int(g["raw_index"]) == (lag if lag >= 0 else lag + 2 * L)
            assert float(g["second"]) == 0.0
            if lag == -L:
                assert int(g["ret"]) == -1 and np.isnan(float(g["coef"]))


def test_all_nan_window_resolves_to_lowest_index(ac):
    """Every allowed value NaN: raw_index is the lowest allowed index and the peak is NaN."""
    import torch
    L = 24000
    src, smp, _ = pairs(L, 1, seed=4)
    src[0, 100] = float("nan")                       # poisons every r[j]
    for window, raw in (((5, 50), 5), ((-50, -5), 2 * L - 50), ((-50, 50), 0)):
        with ctx_for(ac, window=window) as c:
            g = c.xcorr_batch_torch(src, smp)[0]
        assert int(g["raw_index"]) == raw, (window, int(g["raw_index"]))
        assert np.isnan(float(g["peak"]))


def test_host_memspace_pool_stream_and_devices(ac):
    """HOST memspace (more pairs than a wave), the session pool, a non-default stream and the
    multi-device split all give the DEVICE call's records under the same window."""
    import torch
    L, n = 144000, 6
    src, smp, lags = pairs(L, n, seed=21)
    window = (lags[0] + 3, lags[0] + 48000)
    with ctx_for(ac, window=window, wave=2) as c:
        dev = c.xcorr_batch_torch(src, smp)
        hs, hm = src.cpu().numpy(), smp.cpu().numpy()
        assert same(c.xcorr_batch_records(hs.ctypes.data, hm.ctypes.data, n, L, ac.F32, ac.HOST), dev)
        ds, dm = hs.astype(np.float64), hm.astype(np.float64)
        f64 = c.xcorr_batch_records(ds.ctypes.data, dm.ctypes.data, n, L, ac.F64, ac.HOST)
        with ac.SessionPool(c, 0, n, L, ac.F64) as pool:
            for i in range(n):
                pool.append(i, ds[i], dm[i])
            assert same(pool.run(0, n, L), f64)
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            assert same(c.xcorr_batch_torch(src, smp), dev)
    check_against_oracle(dev, hs.astype(np.float64), hm.astype(np.float64), window, False, False)
    if torch.cuda.device_count() >= 2:
        with ctx_for(ac, window=window, devices=None) as many:
            assert same(many.xcorr_batch_records(hs.ctypes.data, hm.ctypes.data, n, L, ac.F32, ac.HOST), dev)


def test_setting_refusals_reset_and_scope(ac):
    import torch
    L = 144000
    src, smp, lags = pairs(L, 2, seed=22)
    with ctx_for(ac) as plain, ctx_for(ac) as c, ctx_for(ac) as other:
        want = plain.xcorr_batch_torch(src, smp)
        with pytest.raises(ac.AudiosyncCudaError):
            c.set_lag_window(5, 4)
        assert same(c.xcorr_batch_torch(src, smp), want)             # refused: setting unchanged
        c.set_lag_window(L, None)                                    # effective window empty at L
        out = torch.full((2 * 64,), 0xAB, dtype=torch.uint8, device="cuda:0")
        with pytest.raises(ac.AudiosyncCudaError, match="lag window"):
            c.xcorr_batch_device(0, src.data_ptr(), smp.data_ptr(), 2, L, ac.F32, out.data_ptr())
        assert "lag window" in ac.last_error()
        torch.cuda.synchronize()
        assert bool((out == 0xAB).all())
        hs, hm = src.cpu().numpy(), smp.cpu().numpy()
        with pytest.raises(ac.AudiosyncCudaError, match="lag window"):
            c.xcorr_batch_records(hs.ctypes.data, hm.ctypes.data, 2, L, ac.F32, ac.HOST)
        c.set_lag_window(lags[0] + 3, lags[0] + 4000)
        assert c.describe_plan(L).endswith(" lags=[%d,%d]" % (lags[0] + 3, lags[0] + 4000))
        assert not same(c.xcorr_batch_torch(src, smp), want)
        assert same(other.xcorr_batch_torch(src, smp), want)           # no leak to another context
        assert " lags=" not in other.describe_plan(L)
        c.set_lag_window()                                           # back to the default
        assert same(c.xcorr_batch_torch(src, smp), want)
        assert " lags=" not in c.describe_plan(L)
        # the drop-in never uses a context's window
        c.set_lag_window(lags[0] + 3, lags[0] + 4000)
        _, lag, _ = ac.cross_correlation(hs[0].astype(np.float64), hm[0].astype(np.float64))
        assert lag == lags[0]
