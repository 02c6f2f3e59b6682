"""Runner-up records (audiosync_cuda_xcorr_runner_up) on the GPU.

The records must be the batch / shared-source calls' byte for byte.  The runner-up must be what the
rule of include/audiosync_cuda.h gives over a full-range correlation export of the same inputs (the
export holds exactly the values the search compared, so raw_index, peak and second agree bit for bit),
and its coefficient fields must be the batch record's at a one-lag window [q, q] on the runner-up lag
q.  Covered: the six static lengths, runtime-radix smooth and embedded lengths, the single-CTA kernel,
PATH_DIRECT and precise mode; F32 / F64 / S16; NONE and PHAT; with and without a lag window; one
source per pair and a shared source.  Then the planted second copy of an echo pair, the motivating
pink-noise pair whose `second` is only the other side of its peak, D = 1 against `second`, and the
edge cases.
"""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
import hard_cases  # noqa: E402
import lagwin_oracle as lo  # noqa: E402

pytestmark = pytest.mark.gpu

AUTO, DIRECT = 0, 2
F32, F64, S16 = 0, 1, 2
HOST, DEVICE = 0, 1
INT64_MIN, INT64_MAX = lo.INT64_MIN, lo.INT64_MAX
# (name, L, path, precise, n pairs)
PLANS = [("static", L, AUTO, False, 2) for L in (144000, 288000, 480000, 720000, 960000, 1440000)] + \
        [("single_cta", 4096, AUTO, False, 3), ("radix_smooth", 24000, AUTO, False, 3),
         ("radix_static_rows", 48000, AUTO, False, 3), ("radix_embedded", 100001, AUTO, False, 3),
         ("direct", 3000, DIRECT, False, 3), ("precise", 24000, AUTO, True, 3)]
IDS = ["%s-%d" % (p[0], p[1]) for p in PLANS]
PHAT_PLANS = {"static", "single_cta", "radix_smooth", "radix_static_rows", "precise"}


@pytest.fixture(scope="module")
def ac():
    import audiosync_cuda
    return audiosync_cuda


def ctx_for(ac, path=AUTO, precise=False, phat=False, window=None, wave=16, devices=(0,)):
    c = ac.Context(list(devices) if devices is not None else None)
    c.set_path(path)
    c.set_precise(precise)
    c.set_weighting(ac.WEIGHT_PHAT if phat else ac.WEIGHT_NONE)
    c.set_wave_pairs(wave)
    if window is not None:
        c.set_lag_window(*window)
    return c


def echo_pairs(L, n, seed, shared=False):
    """n pairs whose sample occurs twice in the source (second copy at 3/4 amplitude), float64."""
    rng = np.random.default_rng(seed)
    src, smp = [], []
    for i in range(n):
        d1 = int(rng.integers(-L // 2, L // 2))
        d2 = d1 + int(rng.integers(L // 8, L // 4)) * (1 if d1 < 0 else -1)
        s, m = hard_cases._finish(*hard_cases.echo_pair_int(seed + (0 if shared else i), L, d1, d2, 3072), np.float64)
        src.append(s)
        smp.append(m)
    src, smp = np.stack(src), np.stack(smp)
    if shared:
        src[1:] = src[0]
    return src, smp


def as_dtype(src, smp, dt):
    if dt == F32:
        return src.astype(np.float32), smp.astype(np.float32)
    if dt == F64:
        return src, smp
    q = lambda a: np.clip(np.round(a * 20000), -32768, 32767).astype(np.int16)   # noqa: E731
    return q(src), q(smp)


def same(a, b):
    return np.asarray(a).tobytes() == np.asarray(b).tobytes()


def raw_order(corr, L):
    lags = np.arange(-L, L)
    r = np.empty(corr.shape[:-1] + (2 * L,))
    r[..., np.where(lags >= 0, lags, lags + 2 * L)] = corr
    return r


def runner_up_raw(p, lo_, hi_, D, L):
    """The runner-up set A(p) as ascending raw indices (empty array when empty)."""
    lags = np.arange(lo_, hi_ + 1, dtype=np.int64)
    lags = lags[np.abs(lags - p) >= D]
    return np.sort(np.where(lags >= 0, lags, lags + 2 * L))


def plain(c, s, m, shared):
    if shared:
        return c.xcorr_shared_source(s[0], m)
    dt = {np.float32: F32, np.float64: F64, np.int16: S16}[s.dtype.type]
    return c.xcorr_batch_records(s.ctypes.data, m.ctypes.data, m.shape[0], m.shape[1], dt, HOST)


def check_against_export(c, s, m, shared, D, window, rec, ru):
    """2: the rule over a full export gives raw_index, peak and second bit for bit; 3: a one-lag window
    at the runner-up lag gives its coefficient fields byte for byte."""
    n, L = m.shape
    erec, corr = c.xcorr_correlation(s[0] if shared else s, m, shared_source=shared)
    assert same(erec, rec)
    r = raw_order(corr, L)
    eff = lo.effective(*(window if window else (INT64_MIN, INT64_MAX)), L)
    for i in range(n):
        raw = runner_up_raw(int(rec["lag"][i]), eff[0], eff[1], D, L)
        if raw.size == 0:
            assert int(ru["raw_index"][i]) == -1 and int(ru["ret"][i]) == -1
            continue
        idx, second = lo.windowed_argmax(r[i], raw)
        assert idx == int(ru["raw_index"][i]), (i, idx, int(ru["raw_index"][i]))
        assert same(r[i][idx], ru["peak"][i]) or (np.isnan(r[i][idx]) and np.isnan(ru["peak"][i]))
        assert same(np.float64(second), ru["second"][i]), (i, second, ru["second"][i])
    for i in range(n):
        if int(ru["raw_index"][i]) < 0:
            continue
        q = int(ru["lag"][i])
        c.set_lag_window(q, q)
        one = plain(c, s[i:i + 1] if not shared else s, m[i:i + 1], shared)[0]
        for f in ("coef", "ret", "success", "ncc", "peak", "lag", "raw_index"):
            assert same(one[f], ru[f][i]), (i, f, one[f], ru[f][i])
    c.set_lag_window(*(window if window else (INT64_MIN, INT64_MAX)))


@pytest.mark.parametrize("name,L,path,precise,n", PLANS, ids=IDS)
def test_records_search_and_coefficient(ac, name, L, path, precise, n):
    src, smp = echo_pairs(L, n, seed=L + 3)
    D = max(2, L // 64)
    for phat in (False, True):
        if phat and name not in PHAT_PLANS:
            continue
        for window in (None, (-L // 2, L // 3)):
            with ctx_for(ac, path, precise, phat, window) as c:
                for dt in ((F32, F64, S16) if L <= 144000 else (F32,)):
                    s, m = as_dtype(src, smp, dt)
                    rec, ru = c.xcorr_runner_up(s, m, D)
                    assert same(rec, plain(c, s, m, False)), (dt, phat, window)
                    check_against_export(c, s, m, False, D, window, rec, ru)


@pytest.mark.parametrize("name,L,path,precise,n", [p for p in PLANS if p[1] <= 144000],
                         ids=[i for p, i in zip(PLANS, IDS) if p[1] <= 144000])
def test_shared_source_and_device(ac, name, L, path, precise, n):
    import torch
    src, smp = echo_pairs(L, n, seed=L + 5, shared=True)
    D = max(2, L // 50)
    with ctx_for(ac, path, precise, window=(-L + 7, L - 9)) as c:
        s, m = as_dtype(src, smp, F32)
        rec, ru = c.xcorr_runner_up(s[0], m, D, shared_source=True)
        assert same(rec, plain(c, s, m, True))
        check_against_export(c, s, m, True, D, (-L + 7, L - 9), rec, ru)
        # the device forms give the host call's records
        ts, tm = torch.from_numpy(s).cuda(), torch.from_numpy(m).cuda()
        drec, dru = c.xcorr_runner_up_torch(ts[0], tm, D, shared_source=True)
        assert same(drec, rec) and same(dru, ru)
        drec, dru = c.xcorr_runner_up_torch(ts, tm, D)
        hrec, hru = c.xcorr_runner_up(s, m, D)
        assert same(drec, hrec) and same(dru, hru)
        # device-memspace host-facing call
        out = np.zeros(n, ac.RESULT_DTYPE), np.zeros(n, ac.RESULT_DTYPE)
        rc = ac.lib().audiosync_cuda_xcorr_runner_up(c.handle, ts.data_ptr(), tm.data_ptr(), n, L, F32, DEVICE, 0, D,
                                                     out[0].ctypes.data, out[1].ctypes.data)
        assert rc == 0 and same(out[0], hrec) and same(out[1], hru)


@pytest.mark.parametrize("L", [144000, 48000, 4096])
def test_planted_second_copy(ac, L):
    """The sample occurs twice, the copies apart in the source; the runner-up is the weaker copy's lag
    with a coefficient above 0.95."""
    d1, d2 = L // 2, -(L // 2)
    s, m = hard_cases._finish(*hard_cases.echo_pair_int(11, L, d1, d2, 3900), np.float64)
    with ctx_for(ac) as c:
        rec, ru = c.xcorr_runner_up(s[None].astype(np.float32), m[None].astype(np.float32), 48)
    assert int(rec["lag"][0]) == d1
    assert int(ru["lag"][0]) == d2 and ru["coef"][0] > 0.95 and ru["success"][0] == 1
    assert abs(ru["peak"][0]) < abs(rec["peak"][0])


def pink(n, rng):
    """Pink (1/f) noise: white noise shaped by 1/sqrt(f) in the frequency domain."""
    w = np.fft.rfft(rng.standard_normal(n))
    f = np.arange(w.size, dtype=np.float64)
    f[0] = 1.0
    return np.fft.irfft(w / np.sqrt(f), n)


def test_pink_noise_second_is_the_same_peak(ac):
    """The motivating case: `second` is the other side of the peak, the runner-up is not."""
    L, true_lag = 144000, 30000
    rng = np.random.default_rng(1)
    src = pink(2 * L, rng)
    smp = src[true_lag:true_lag + L].copy()
    s, m = src[None].astype(np.float32), smp[None].astype(np.float32)
    with ctx_for(ac) as c:
        rec, ru = c.xcorr_runner_up(s, m, 48)
        _, corr = c.xcorr_correlation(s, m)
    pk = abs(rec["peak"][0])
    assert int(rec["lag"][0]) == true_lag
    assert rec["second"][0] / pk > 0.8
    near = np.abs(corr[0][true_lag + L - 3:true_lag + L + 4])
    assert np.any(near == rec["second"][0])                  # a neighbouring lag holds `second`
    assert abs(int(ru["lag"][0]) - true_lag) >= 48
    assert abs(ru["peak"][0]) / pk < 0.8 * rec["second"][0] / pk


@pytest.mark.parametrize("name,L,path,precise,n", [p for p in PLANS if p[1] <= 144000],
                         ids=[i for p, i in zip(PLANS, IDS) if p[1] <= 144000])
def test_d1_is_second(ac, name, L, path, precise, n):
    """D = 1: |runner-up peak| is the record's second, unless lag 0 is allowed with a negative r[0]."""
    src, smp = echo_pairs(L, n, seed=L + 9)
    with ctx_for(ac, path, precise) as c:
        s, m = as_dtype(src, smp, F32)
        rec, ru = c.xcorr_runner_up(s, m, 1)
        _, corr = c.xcorr_correlation(s, m)
    for i in range(n):
        r0 = corr[i][L]
        if rec["lag"][i] != 0 and r0 < 0 and -r0 >= rec["second"][i]:
            continue
        assert same(np.float64(abs(ru["peak"][i])), rec["second"][i]), (i, ru["peak"][i], rec["second"][i])


def test_edge_cases(ac):
    L = 48000
    src, smp = echo_pairs(L, 3, seed=21)
    s, m = as_dtype(src, smp, F32)
    with ctx_for(ac) as c:
        base = plain(c, s, m, False)
        # D larger than any distance in the window: an empty set for every pair, return value 0
        c.set_lag_window(-10, 10)
        rec, ru = c.xcorr_runner_up(s, m, 100)
        assert same(rec, plain(c, s, m, False))
        for f, v in (("raw_index", -1), ("lag", 0), ("ret", -1), ("success", 0)):
            assert np.all(ru[f] == v), f
        assert np.all(ru["peak"] == 0) and np.all(ru["second"] == 0) and np.all(ru["margin"] == 0)
        assert np.all(np.isnan(ru["coef"])) and np.all(np.isnan(ru["ncc"]))
        c.set_lag_window(INT64_MIN, INT64_MAX)
        # refusals write nothing
        def marked():
            a = np.zeros(3, ac.RESULT_DTYPE)
            a["lag"] = 7
            return a
        for D in (0, -5):
            a, b = marked(), marked()
            rc = ac.lib().audiosync_cuda_xcorr_runner_up(c.handle, s.ctypes.data, m.ctypes.data, 3, L, F32, HOST, 0, D,
                                                         a.ctypes.data, b.ctypes.data)
            assert rc == -1 and np.all(a["lag"] == 7) and np.all(b["lag"] == 7)
        a = marked()
        assert ac.lib().audiosync_cuda_xcorr_runner_up(c.handle, s.ctypes.data, m.ctypes.data, 3, L, F32, HOST, 0, 5,
                                                       a.ctypes.data, None) == -1
        assert ac.lib().audiosync_cuda_xcorr_runner_up(c.handle, s.ctypes.data, m.ctypes.data, 3, L, 9, HOST, 0, 5,
                                                       a.ctypes.data, a.ctypes.data) == -1
        c.set_lag_window(L + 5, L + 9)                        # empty effective window: the batch call refuses
        b = marked()
        assert ac.lib().audiosync_cuda_xcorr_runner_up(c.handle, s.ctypes.data, m.ctypes.data, 3, L, F32, HOST, 0, 5,
                                                       a.ctypes.data, b.ctypes.data) == -1
        assert np.all(a["lag"] == 7) and np.all(b["lag"] == 7)
        c.set_lag_window(INT64_MIN, INT64_MAX)
        # n_pairs == 0
        assert ac.lib().audiosync_cuda_xcorr_runner_up(c.handle, s.ctypes.data, m.ctypes.data, 0, L, F32, HOST, 0, 5,
                                                       None, None) == 0
        rec, ru = c.xcorr_runner_up(s, m, 200)
        assert same(rec, base)


def test_narrowing_and_devices(ac):
    """LOSSLESS host narrowing equals NARROW_OFF; a HOST call over two devices equals the one-device call."""
    L = 144000
    src, smp = echo_pairs(L, 5, seed=33)
    s, m = as_dtype(src, smp, F64)                            # exact fp32 images: LOSSLESS narrows them
    with ctx_for(ac, wave=2) as c:
        c.set_host_narrowing(ac.NARROW_OFF)
        want = c.xcorr_runner_up(s, m, 300)
        c.set_host_narrowing(ac.NARROW_LOSSLESS)
        got = c.xcorr_runner_up(s, m, 300)
    assert same(got[0], want[0]) and same(got[1], want[1])
    import torch
    if torch.cuda.device_count() < 2:
        return
    with ctx_for(ac, wave=2, devices=(0, 1)) as c2:
        got = c2.xcorr_runner_up(s, m, 300)
    assert same(got[0], want[0]) and same(got[1], want[1])
