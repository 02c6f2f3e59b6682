"""One source against many samples (audiosync_cuda_xcorr_shared_source) on the GPU.

Every record must be, byte for byte, what the batch call returns for the same pairs with the source
replicated into sources[n][2L]: on every kind of plan (the static lengths through the reuse path,
every other plan by reading the one source), in every dtype and memspace, under PHAT and a lag
window, for a source at an odd element offset, over several waves and several devices.  The profile
API shows the source-spectrum kernel once per call and device on the static lengths, never elsewhere.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

AUTO, DIRECT = 0, 2
STATIC_LENGTHS = (144000, 288000, 480000, 720000, 960000, 1440000)
# (name, L, forced path, precise): every kind of plan the batch calls run
PATHS = [("static", 144000, AUTO, False), ("single_cta", 4096, AUTO, False),
         ("radix_smooth", 24000, AUTO, False), ("radix_static_rows", 48000, AUTO, False),
         ("radix_embedded", 100001, AUTO, False), ("direct", 4096, DIRECT, False),
         ("precise", 24000, AUTO, True)]
PHAT_PATHS = {"static", "single_cta", "radix_smooth", "radix_static_rows", "precise"}


@pytest.fixture(scope="module")
def ac():
    import audiosync_cuda
    return audiosync_cuda


def ctx_for(ac, path=AUTO, precise=False, phat=False, window=None, devices=(0,), wave=0):
    c = ac.Context(list(devices) if devices is not None else None)
    c.set_path(path)
    c.set_precise(precise)
    c.set_weighting(ac.WEIGHT_PHAT if phat else ac.WEIGHT_NONE)
    c.set_wave_pairs(wave)
    if window is not None:
        c.set_lag_window(*window)
    c.profile_enable(True)
    return c


def batch(L, seed, extra=1):
    """fp32 on cuda:0: one source [2L] and samples cut from it at a positive and a negative lag plus
    noise, a polarity-inverted cut, an all-zero sample and `extra` noise samples."""
    import torch
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    src = torch.randn(2 * L, device="cuda:0", generator=g)
    noise = lambda: 0.3 * torch.randn(L, device="cuda:0", generator=g)   # noqa: E731
    a, b = L // 3, L // 5
    rows = [src[a:a + L] + noise(),                                           # lag +a
            torch.cat([torch.randn(b, device="cuda:0", generator=g), src[:L - b]]) + noise(),   # lag -b
            -src[L // 2:L // 2 + L],                                          # inverted
            torch.zeros(L, device="cuda:0")]
    rows += [torch.randn(L, device="cuda:0", generator=g) for _ in range(extra)]
    return src.contiguous(), torch.stack(rows).contiguous()


def as_dtype(t, dt):
    import torch
    if dt == "f32":
        return t
    if dt == "f64":
        return t.double()
    return (t * 6000).clamp(-32768, 32767).round().to(torch.int16).contiguous()


def dtype_code(ac, t):
    import torch
    return {torch.float32: ac.F32, torch.float64: ac.F64, torch.int16: ac.S16}[t.dtype]


def replicated(ac, c, src, smp, memspace):
    """The batch call on the source replicated per pair (the contract's reference)."""
    n, L = smp.shape
    sources = src[:2 * L].expand(n, 2 * L).contiguous()
    if memspace == "host":
        s, m = sources.cpu().numpy(), smp.cpu().numpy()
        return c.xcorr_batch_records(s.ctypes.data, m.ctypes.data, n, L, dtype_code(ac, smp), ac.HOST)
    return c.xcorr_batch_torch(sources, smp)


def shared(ac, c, src, smp, memspace):
    if memspace == "host":
        return c.xcorr_shared_source(src.cpu().numpy(), smp.cpu().numpy())
    return c.xcorr_shared_source_torch(src, smp)


def spectra(c):
    return c.profile_read()["src_spectrum"][0]


def check_records(rec):
    """The planted samples resolve as expected (peak cut lags; all-zero sample: NaN coefficient)."""
    assert int(rec["ret"][3]) == -1 and np.isnan(rec["coef"][3])
    assert int(rec["ret"][0]) == 0


def same(a, b):
    return a.tobytes() == b.tobytes()


@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("L", STATIC_LENGTHS)
def test_static_lengths_reuse_the_source_spectrum(ac, L, phat):
    src, smp = batch(L, seed=L)
    with ctx_for(ac, phat=phat) as c:
        ref = replicated(ac, c, src, smp, "device")
        c.profile_reset()
        got = shared(ac, c, src, smp, "device")
        assert spectra(c) == 1
    assert same(ref, got)
    check_records(got)
    if not phat:
        assert (int(got["lag"][0]), int(got["lag"][1])) == (L // 3, -(L // 5))


@pytest.mark.parametrize("memspace", ["device", "host"])
@pytest.mark.parametrize("dt", ["f32", "f64", "s16"])
@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
@pytest.mark.parametrize("name,L,path,precise", PATHS, ids=[p[0] for p in PATHS])
def test_every_plan_dtype_and_memspace(ac, name, L, path, precise, phat, dt, memspace):
    if phat and name not in PHAT_PATHS:
        pytest.skip("PHAT is refused on this path")
    src, smp = batch(L, seed=L + 7)
    src, smp = as_dtype(src, dt), as_dtype(smp, dt)
    with ctx_for(ac, path, precise, phat) as c:
        ref = replicated(ac, c, src, smp, memspace)
        c.profile_reset()
        got = shared(ac, c, src, smp, memspace)
        assert spectra(c) == (1 if name == "static" else 0)
    assert same(ref, got)
    check_records(got)


@pytest.mark.parametrize("name,L,path,precise", [p for p in PATHS if p[0] in ("static", "radix_smooth", "single_cta")],
                         ids=["static", "single_cta", "radix_smooth"])
def test_lag_window_excluding_the_peak(ac, name, L, path, precise):
    src, smp = batch(L, seed=3)
    with ctx_for(ac, path, precise, window=(-L // 10, L // 10)) as c:      # excludes lags +L/3 and -L/5
        ref = replicated(ac, c, src, smp, "device")
        got = shared(ac, c, src, smp, "device")
    assert same(ref, got)
    assert abs(int(got["lag"][0])) <= L // 10 and abs(int(got["lag"][1])) <= L // 10


@pytest.mark.parametrize("dt", ["f32", "f64", "s16"])
@pytest.mark.parametrize("L", [144000, 24000, 4096])
def test_source_at_an_odd_element_offset(ac, L, dt):
    import torch
    src, smp = batch(L, seed=11)
    src, smp = as_dtype(src, dt), as_dtype(smp, dt)
    buf = torch.zeros(2 * L + 1, dtype=src.dtype, device="cuda:0")
    buf[1:] = src
    view = buf[1:]                                     # element aligned, not aligned to two elements
    host_buf = buf.cpu().numpy()
    host_view = host_buf[1:]
    assert host_view.ctypes.data % (2 * host_view.itemsize) != 0
    with ctx_for(ac) as c:
        ref = replicated(ac, c, src, smp, "device")
        assert same(ref, shared(ac, c, view, smp, "device"))
        assert same(ref, c.xcorr_shared_source(host_view, smp.cpu().numpy()))


@pytest.mark.parametrize("L", [144000, 24000])
def test_more_pairs_than_one_wave(ac, L):
    src, smp = batch(L, seed=5, extra=4)               # 8 pairs, waves of 3
    with ctx_for(ac, wave=3) as c:
        ref = replicated(ac, c, src, smp, "device")
        c.profile_reset()
        got = shared(ac, c, src, smp, "device")
        assert spectra(c) == (1 if L == 144000 else 0)     # once per call, not per wave
        host = shared(ac, c, src, smp, "host")
    assert same(ref, got) and same(ref, host)


def test_host_call_of_several_chunks_transforms_the_source_once(ac):
    """A host-fed call is uploaded in chunks of about 192 MB of samples (33 F32 samples at 1,440,000
    frames): the later chunks reuse the first one's source spectrum."""
    L = 1440000
    src, smp = batch(L, seed=29, extra=76)             # 80 samples: three chunks
    with ctx_for(ac) as c:
        ref = replicated(ac, c, src, smp, "host")
        c.profile_reset()
        got = shared(ac, c, src, smp, "host")
        assert spectra(c) == 1
    assert same(ref, got)
    check_records(got)


def test_all_devices_of_the_context(ac):
    import torch
    L = 144000
    src, smp = batch(L, seed=9, extra=2 * torch.cuda.device_count())
    with ctx_for(ac, devices=None) as c:
        G = c.device_count()
        ref = replicated(ac, c, src, smp, "host")
        c.profile_reset()
        got = shared(ac, c, src, smp, "host")
        assert spectra(c) == G                          # the source is transformed once per device
    assert same(ref, got)


def test_f64_host_is_the_unnarrowed_call(ac):
    L = 144000
    src, smp = batch(L, seed=13)
    src, smp = src.double(), smp.double()
    with ctx_for(ac) as c:
        got = shared(ac, c, src, smp, "host")
        c.set_host_narrowing(ac.NARROW_OFF)
        off = replicated(ac, c, src, smp, "host")
        c.set_host_narrowing(ac.NARROW_ALWAYS)
        assert same(off, shared(ac, c, src, smp, "host"))     # narrowing does not apply
    assert same(off, got)


def test_torch_form_on_a_side_stream(ac):
    import torch
    L = 144000
    src, smp = batch(L, seed=17)
    with ctx_for(ac) as c:
        ref = replicated(ac, c, src, smp, "device")
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            out = c.xcorr_shared_source_torch(src, smp, sync=False)
        s.synchronize()
        got = out.cpu().numpy().view(ac.RESULT_DTYPE)
    assert same(ref, got)


def test_refusals_launch_nothing(ac):
    import torch
    lib = ac.lib()
    L = 144000
    src, smp = batch(L, seed=19)
    out = torch.zeros(smp.shape[0] * 64, dtype=torch.uint8, device="cuda:0")
    with ctx_for(ac) as c:
        n0 = c.launch_count()
        # a device base between two elements
        rc = lib.audiosync_cuda_xcorr_shared_source_device(c.handle, 0, src.data_ptr() + 2, smp.data_ptr(), smp.shape[0], L,
                                                           ac.F32, out.data_ptr(), None)
        assert rc == -1 and c.launch_count() == n0
        # no pairs: nothing to do
        rc = lib.audiosync_cuda_xcorr_shared_source_device(c.handle, 0, src.data_ptr(), smp.data_ptr(), 0, L,
                                                           ac.F32, out.data_ptr(), None)
        assert rc == 0 and c.launch_count() == n0
        assert len(c.xcorr_shared_source(src.cpu().numpy(), smp.cpu().numpy()[:0])) == 0
        assert c.launch_count() == n0
    Le = 100001
    src, smp = batch(Le, seed=23)
    res = np.zeros(smp.shape[0], ac.RESULT_DTYPE)
    with ctx_for(ac, phat=True) as c:
        n0 = c.launch_count()
        s, m = src.cpu().numpy(), smp.cpu().numpy()
        rc = lib.audiosync_cuda_xcorr_shared_source(c.handle, s.ctypes.data, m.ctypes.data, smp.shape[0], Le, ac.F32,
                                                    ac.HOST, res.ctypes.data)
        assert rc == -1 and c.launch_count() == n0
        rc = lib.audiosync_cuda_xcorr_shared_source_device(c.handle, 0, src.data_ptr(), smp.data_ptr(), smp.shape[0], Le,
                                                           ac.F32, out.data_ptr(), None)
        assert rc == -1 and c.launch_count() == n0
