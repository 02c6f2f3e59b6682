"""Every source against every sample (audiosync_cuda_xcorr_cross) on the GPU.

Record (s, p) must be, byte for byte, record p of the shared-source call on source s and, through that
call's own contract, the batch call's record for the pair (sources[s], samples[p]).  Both references are
checked on every static length (the reuse path: each source's and each wave's samples' spectra once, the
row kernel from both), on every other kind of plan (one shared-source call per source), in every dtype and
memspace, under PHAT and a lag window, at an odd element offset, over several waves and devices.  The
profile API shows the launches the reuse path promises.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

AUTO, DIRECT = 0, 2
STATIC_LENGTHS = (144000, 288000, 480000, 720000, 960000, 1440000)
# (name, L, forced path, precise): the plans without reuse
OTHER_PATHS = [("radix", 1000000, AUTO, False), ("radix_embedded", 100001, AUTO, False),
               ("single_cta", 4096, AUTO, False), ("direct", 4096, DIRECT, False), ("precise", 24000, AUTO, True)]


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


def cross_batch(L, seed, S=3, P=5):
    """fp32 on cuda:0: S sources [S, 2L] and P samples [P, L].  Sample 0 is cut from source 0 at lag
    +L/3, sample 1 from source 1 (when there is one) at lag -L/5 (zeros shifted in), sample 2 is source
    0 inverted, sample 3 is all zeros; the rest and the other sources are noise."""
    import torch
    g = torch.Generator(device="cuda:0").manual_seed(seed)
    src = torch.randn(S, 2 * L, device="cuda:0", generator=g)
    noise = lambda: 0.3 * torch.randn(L, device="cuda:0", generator=g)   # noqa: E731
    a, b = L // 3, L // 5
    s1 = src[1 if S > 1 else 0]
    rows = [src[0, a:a + L] + noise(),
            torch.cat([torch.zeros(b, device="cuda:0"), s1[:L - b]]) + noise(),
            -src[0, L // 2:L // 2 + L],
            torch.zeros(L, device="cuda:0")]
    rows += [torch.randn(L, device="cuda:0", generator=g) for _ in range(P - 4)]
    return src.contiguous(), torch.stack(rows[:P]).contiguous()


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


def shared_rows(ac, c, src, smp, memspace):
    """S shared-source calls, [S, P] records."""
    if memspace == "host":
        m = smp.cpu().numpy()
        return np.stack([c.xcorr_shared_source(s, m) for s in src.cpu().numpy()])
    return np.stack([c.xcorr_shared_source_torch(s, smp) for s in src])


def replicated(ac, c, src, smp):
    """The batch call on every (source, sample) pair, [S, P] records."""
    S, P = src.shape[0], smp.shape[0]
    sources = src.repeat_interleave(P, dim=0).contiguous()
    samples = smp.repeat(S, 1).contiguous()
    return c.xcorr_batch_torch(sources, samples).reshape(S, P)


def cross(ac, c, src, smp, memspace):
    if memspace == "host":
        return c.xcorr_cross(src.cpu().numpy(), smp.cpu().numpy())
    if memspace == "device_ptr":
        S, P, L = src.shape[0], smp.shape[0], smp.shape[1]
        return c.xcorr_cross_records(src.data_ptr(), S, smp.data_ptr(), P, L, dtype_code(ac, src), ac.DEVICE)
    return c.xcorr_cross_torch(src, smp)


def launches(c):
    p = c.profile_read()
    return {k: p[k][0] for k in ("src_spectrum", "smp_spectrum", "row_fused", "col_fwd")}


def same(a, b):
    return a.shape == b.shape and a.tobytes() == b.tobytes()


def check_records(rec):
    """The planted samples resolve: sample 0 against source 0, the all-zero sample has no coefficient."""
    assert (rec["ret"][:, 3] == -1).all() and np.isnan(rec["coef"][:, 3]).all()
    assert int(rec["ret"][0, 0]) == 0


@pytest.mark.parametrize("L", STATIC_LENGTHS)
def test_static_lengths(ac, L):
    src, smp = cross_batch(L, seed=L)
    with ctx_for(ac, wave=2) as c:
        ref = shared_rows(ac, c, src, smp, "device")
        rep = replicated(ac, c, src, smp)
        c.profile_reset()
        got = cross(ac, c, src, smp, "device")
        n = launches(c)
    assert same(ref, got) and same(rep, got)
    check_records(got)
    assert (int(got["lag"][0, 0]), int(got["lag"][1, 1])) == (L // 3, -(L // 5))
    waves = 3                                            # 5 samples in waves of 2
    assert n["src_spectrum"] == 3 and n["smp_spectrum"] == waves and n["row_fused"] == 3 * waves
    assert n["col_fwd"] == 3 + waves                     # each source's K_A, then one per sample wave


@pytest.mark.parametrize("memspace", ["device", "device_ptr", "host"])
@pytest.mark.parametrize("dt", ["f32", "f64", "s16"])
@pytest.mark.parametrize("phat", [False, True], ids=["none", "phat"])
def test_dtypes_memspaces_and_phat(ac, phat, dt, memspace):
    L = 144000
    src, smp = cross_batch(L, seed=31)
    src, smp = as_dtype(src, dt), as_dtype(smp, dt)
    with ctx_for(ac, phat=phat, wave=2) as c:
        ref = shared_rows(ac, c, src, smp, "host" if memspace == "host" else "device")
        rep = replicated(ac, c, src, smp)
        got = cross(ac, c, src, smp, memspace)
    assert same(ref, got) and same(rep, got)
    check_records(got)


@pytest.mark.parametrize("name,L,path,precise", OTHER_PATHS, ids=[p[0] for p in OTHER_PATHS])
def test_plans_without_reuse(ac, name, L, path, precise):
    src, smp = cross_batch(L, seed=L + 3)
    with ctx_for(ac, path, precise, wave=2) as c:
        ref = shared_rows(ac, c, src, smp, "device")
        rep = replicated(ac, c, src, smp)
        c.profile_reset()
        got = cross(ac, c, src, smp, "device")
        n = launches(c)
        host = cross(ac, c, src, smp, "host")
    assert same(ref, got) and same(rep, got) and same(ref, host)
    check_records(got)
    assert n["src_spectrum"] == 0 and n["smp_spectrum"] == 0


@pytest.mark.parametrize("L", [144000, 24000])
def test_lag_window_excluding_lag_zero(ac, L):
    src, smp = cross_batch(L, seed=37)
    with ctx_for(ac, window=(L // 10, L // 2), wave=2) as c:          # holds +L/3, excludes 0 and -L/5
        ref = shared_rows(ac, c, src, smp, "device")
        rep = replicated(ac, c, src, smp)
        got = cross(ac, c, src, smp, "device")
    assert same(ref, got) and same(rep, got)
    assert int(got["lag"][0, 0]) == L // 3
    assert ((got["lag"] >= L // 10) & (got["lag"] <= L // 2))[got["ret"] == 0].all()


@pytest.mark.parametrize("dt", ["f32", "f64", "s16"])
@pytest.mark.parametrize("L", [144000, 24000])
def test_inputs_at_an_odd_element_offset(ac, L, dt):
    """Sources and samples one element into a buffer: element aligned, not aligned to two elements
    (the register path of K_A)."""
    import torch
    src, smp = cross_batch(L, seed=41)
    src, smp = as_dtype(src, dt), as_dtype(smp, dt)
    sbuf = torch.zeros(src.numel() + 1, dtype=src.dtype, device="cuda:0")
    mbuf = torch.zeros(smp.numel() + 1, dtype=smp.dtype, device="cuda:0")
    sbuf[1:] = src.flatten()
    mbuf[1:] = smp.flatten()
    sv, mv = sbuf[1:].view(src.shape), mbuf[1:].view(smp.shape)
    hs, hm = sbuf.cpu().numpy(), mbuf.cpu().numpy()
    S, P = src.shape[0], smp.shape[0]
    with ctx_for(ac, wave=2) as c:
        ref = shared_rows(ac, c, src, smp, "device")
        assert same(ref, cross(ac, c, sv, mv, "device"))
        host = c.xcorr_cross_records(hs.ctypes.data + hs.itemsize, S, hm.ctypes.data + hm.itemsize, P, L,
                                     dtype_code(ac, src), ac.HOST)
        assert same(ref, host)


def test_host_call_of_several_chunks_transforms_each_source_once(ac):
    """A host-fed call uploads its samples in chunks of about 192 MB (33 F32 samples at 1,440,000
    frames): the later chunks reuse the first one's source spectra."""
    L = 1440000
    src, smp = cross_batch(L, seed=43, S=2, P=70)
    with ctx_for(ac) as c:
        ref = shared_rows(ac, c, src, smp, "host")
        c.profile_reset()
        got = cross(ac, c, src, smp, "host")
        assert launches(c)["src_spectrum"] == 2
    assert same(ref, got)


def test_torch_form_on_a_side_stream(ac):
    import torch
    L = 144000
    src, smp = cross_batch(L, seed=47)
    with ctx_for(ac, wave=2) as c:
        ref = shared_rows(ac, c, src, smp, "device")
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            out = c.xcorr_cross_torch(src, smp, sync=False)
        s.synchronize()
        got = out.cpu().numpy().view(ac.RESULT_DTYPE).reshape(ref.shape)
    assert same(ref, got)


def test_all_devices_of_the_context(ac):
    import torch
    L = 144000
    G = torch.cuda.device_count()
    src, smp = cross_batch(L, seed=53, P=4 + 2 * G)
    with ctx_for(ac, devices=None, wave=2) as c:
        assert c.device_count() == G
        ref = shared_rows(ac, c, src, smp, "host")
        c.profile_reset()
        got = cross(ac, c, src, smp, "host")
        n = launches(c)
    assert same(ref, got)
    assert n["src_spectrum"] == 3 * G                    # every source on every device
    per = [(smp.shape[0] + G - 1 - g) // G for g in range(G)]   # contiguous blocks, the first ones larger
    assert n["smp_spectrum"] == sum((k + 1) // 2 for k in per)
    assert n["row_fused"] == 3 * n["smp_spectrum"]


def test_refusals_write_no_record(ac):
    import torch
    lib = ac.lib()
    L = 144000
    src, smp = cross_batch(L, seed=59)
    S, P = src.shape[0], smp.shape[0]
    sentinel = 0xA5
    out = torch.full((S * P * 64,), sentinel, dtype=torch.uint8, device="cuda:0")
    res = np.zeros((S, P), ac.RESULT_DTYPE)
    res.view(np.uint8)[...] = sentinel
    hs, hm = src.cpu().numpy(), smp.cpu().numpy()

    def untouched():
        torch.cuda.synchronize()
        return bool((out == sentinel).all()) and bool((res.view(np.uint8) == sentinel).all())

    with ctx_for(ac) as c:
        n0 = c.launch_count()
        # a device base between two elements
        rc = lib.audiosync_cuda_xcorr_cross_device(c.handle, 0, src.data_ptr() + 2, S, smp.data_ptr(), P, L, ac.F32,
                                                   out.data_ptr(), None)
        assert rc == -1
        # no sources or no samples: nothing to do
        for ns, npairs in ((0, P), (S, 0)):
            assert lib.audiosync_cuda_xcorr_cross_device(c.handle, 0, src.data_ptr(), ns, smp.data_ptr(), npairs, L,
                                                         ac.F32, out.data_ptr(), None) == 0
            assert lib.audiosync_cuda_xcorr_cross(c.handle, hs.ctypes.data, ns, hm.ctypes.data, npairs, L, ac.F32,
                                                  ac.HOST, res.ctypes.data) == 0
        # a record count that overflows
        big = 1 << 62
        assert lib.audiosync_cuda_xcorr_cross_device(c.handle, 0, src.data_ptr(), big, smp.data_ptr(), 4, L, ac.F32,
                                                     out.data_ptr(), None) == -1
        assert lib.audiosync_cuda_xcorr_cross(c.handle, hs.ctypes.data, 4, hm.ctypes.data, big, L, ac.F32, ac.HOST,
                                              res.ctypes.data) == -1
        # bad dtype, null pointers
        assert lib.audiosync_cuda_xcorr_cross(c.handle, hs.ctypes.data, S, hm.ctypes.data, P, L, 7, ac.HOST,
                                              res.ctypes.data) == -1
        assert lib.audiosync_cuda_xcorr_cross(c.handle, None, S, hm.ctypes.data, P, L, ac.F32, ac.HOST,
                                              res.ctypes.data) == -1
        assert c.launch_count() == n0
        # a lag window with no lag at this length
        c.set_lag_window(L, 2 * L)
        assert lib.audiosync_cuda_xcorr_cross(c.handle, hs.ctypes.data, S, hm.ctypes.data, P, L, ac.F32, ac.HOST,
                                              res.ctypes.data) == -1
        assert lib.audiosync_cuda_xcorr_cross_device(c.handle, 0, src.data_ptr(), S, smp.data_ptr(), P, L, ac.F32,
                                                     out.data_ptr(), None) == -1
        assert c.launch_count() == n0
    # PHAT on a length whose plan cannot weight
    Le = 100001
    src, smp = cross_batch(Le, seed=61)
    hs, hm = src.cpu().numpy(), smp.cpu().numpy()
    with ctx_for(ac, phat=True) as c:
        n0 = c.launch_count()
        assert lib.audiosync_cuda_xcorr_cross(c.handle, hs.ctypes.data, S, hm.ctypes.data, P, Le, ac.F32, ac.HOST,
                                              res.ctypes.data) == -1
        assert lib.audiosync_cuda_xcorr_cross_device(c.handle, 0, src.data_ptr(), S, smp.data_ptr(), P, Le, ac.F32,
                                                     out.data_ptr(), None) == -1
        assert c.launch_count() == n0
    assert untouched()
