"""16-bit PCM (S16) batches on the GPU: every record equals, byte for byte, the F64 call's record on
the doubles s / 32768 -- on every transform path, in precise mode, fed from host or device memory,
through torch tensors, and at any 2-byte-aligned base."""
import os
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "golden"))
sys.path.insert(0, HERE)
from test_pcm_s16_emu import pcm_pair  # noqa: E402

pytestmark = pytest.mark.gpu

STATIC_LENGTHS = (144000, 288000, 480000, 720000, 960000, 1440000)
GEN_LENGTHS = (10007, 24000, 48000, 65536, 100001)      # runtime-radix: 10,007 and 100,001 are embedded
SHORT_LENGTHS = (1000, 4096, 6000)                       # direct / single-CTA under AUTO
AUTO, FFT, DIRECT = 0, 1, 2


@pytest.fixture(scope="module")
def ac():
    import audiosync_cuda
    audiosync_cuda.lib()
    return audiosync_cuda


@pytest.fixture(scope="module")
def ctx(ac):
    c = ac.Context([0])
    yield c
    c.close()


def pairs16(n, L, seed):
    ss, mm = zip(*(pcm_pair(L, seed * 1000 + i) for i in range(n)))
    return np.stack(ss), np.stack(mm)


def widen(x):
    return x.astype(np.float64) / 32768.0


def dev_records(ctx, src, smp):
    """Records of one DEVICE-memspace call (torch tensors on cuda:0, the dtype of the arrays)."""
    import torch
    s = torch.from_numpy(np.ascontiguousarray(src)).cuda()
    m = torch.from_numpy(np.ascontiguousarray(smp)).cuda()
    return ctx.xcorr_batch_torch(s, m)


def assert_same_bytes(got, ref):
    assert got.dtype == ref.dtype and got.shape == ref.shape
    if got.tobytes() != ref.tobytes():
        bad = [i for i in range(len(got)) if got[i].tobytes() != ref[i].tobytes()]
        raise AssertionError("%d of %d records differ, first %d:\n  s16 %s\n  f64 %s"
                             % (len(bad), len(got), bad[0], got[bad[0]], ref[bad[0]]))


def check_s16_equals_f64(ctx, src, smp):
    got = dev_records(ctx, src, smp)
    assert_same_bytes(got, dev_records(ctx, widen(src), widen(smp)))
    return got


def _path_cases():
    out = []
    for L in STATIC_LENGTHS:
        out += [(L, AUTO), (L, FFT)]
    for L in GEN_LENGTHS:
        out += [(L, AUTO), (L, FFT)]
    out += [(24000, DIRECT), (10007, DIRECT)]
    for L in SHORT_LENGTHS:
        out += [(L, AUTO), (L, FFT), (L, DIRECT)]
    return [pytest.param(L, p, id="L%d-%s" % (L, ("auto", "fft", "direct")[p])) for L, p in out]


@pytest.mark.parametrize("L,path", _path_cases())
def test_every_path_s16_equals_f64(ac, L, path):
    with ac.Context([0]) as c:
        c.set_path(path)
        src, smp = pairs16(3, L, L + path)
        rec = check_s16_equals_f64(c, src, smp)
        assert (rec["ret"] == 0).all()


@pytest.mark.parametrize("L", [144000, 1440000])
def test_precise_mode_s16_equals_f64(ac, L):
    with ac.Context([0]) as c:
        c.set_precise(True)
        src, smp = pairs16(2, L, L + 7)
        check_s16_equals_f64(c, src, smp)


@pytest.mark.parametrize("pinned", [True, False], ids=["pinned", "pageable"])
def test_host_memspace_equals_device(ac, ctx, pinned):
    """HOST S16 at 1,440,000 frames over more than one upload chunk (about 22 pairs each) equals the
    DEVICE call, which equals F64."""
    import torch
    L, n = 1440000, 25
    src, smp = pairs16(n, L, 11)
    if pinned:
        hs = torch.from_numpy(src).pin_memory()
        hm = torch.from_numpy(smp).pin_memory()
        ps, pm = hs.data_ptr(), hm.data_ptr()
    else:
        ps, pm = src.ctypes.data, smp.ctypes.data
    host = ctx.xcorr_batch_records(ps, pm, n, L, ac.S16, ac.HOST)
    assert_same_bytes(host, check_s16_equals_f64(ctx, src, smp))
    ctx.host_feed_stats(reset=True)
    ctx.xcorr_batch_records(ps, pm, 2, L, ac.S16, ac.HOST)
    assert ctx.host_feed_stats(reset=True) == (0, 0)          # S16 pairs are not F64 host-feed pairs
    lists = ctx.xcorr_batch(src[:3], smp[:3])
    assert (lists["lags"] == host["lag"][:3]).all() and (lists["rets"] == host["ret"][:3]).all()


def test_host_memspace_multi_device_split(ac):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    L, n = 144000, 9
    src, smp = pairs16(n, L, 12)
    with ac.Context([0, 1]) as c:
        host = c.xcorr_batch_records(src.ctypes.data, smp.ctypes.data, n, L, ac.S16, ac.HOST)
    with ac.Context([0]) as c:
        assert_same_bytes(host, check_s16_equals_f64(c, src, smp))


def test_torch_int16_on_non_default_stream(ac, ctx):
    import torch
    L, n = 144000, 4
    src, smp = pairs16(n, L, 13)
    s = torch.from_numpy(src).cuda()
    m = torch.from_numpy(smp).cuda()
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        out = ctx.xcorr_batch_torch(s, m, sync=False)
    st.synchronize()
    got = out.cpu().numpy().view(ac.RESULT_DTYPE)
    assert_same_bytes(got, dev_records(ctx, widen(src), widen(smp)))


@pytest.mark.parametrize("L", [144000, 24000, 4096, 1000])
def test_odd_element_offset_equals_aligned(ac, ctx, L):
    """Views buf[1:] start 2 bytes past a 4-byte boundary: the kernels take two 2-byte loads per point."""
    import torch
    n = 3
    src, smp = pairs16(n, L, 14)
    bs = torch.zeros(n * 2 * L + 1, dtype=torch.int16, device="cuda")
    bm = torch.zeros(n * L + 1, dtype=torch.int16, device="cuda")
    bs[1:] = torch.from_numpy(src.reshape(-1)).cuda()
    bm[1:] = torch.from_numpy(smp.reshape(-1)).cuda()
    vs, vm = bs[1:].view(n, 2 * L), bm[1:].view(n, L)
    assert vs.data_ptr() % 4 == 2 and vm.data_ptr() % 4 == 2
    aligned = dev_records(ctx, src, smp)
    assert_same_bytes(ctx.xcorr_batch_torch(vs, vm), aligned)
    assert_same_bytes(aligned, dev_records(ctx, widen(src), widen(smp)))


@pytest.mark.parametrize("L", [144000, 24000, 4096, 1000])
def test_edge_values(ac, ctx, L):
    rng = np.random.default_rng(L)
    full = np.where(rng.random(2 * L) < 0.5, -32768, 32767).astype(np.int16)
    src = np.stack([full, np.full(2 * L, 32767, np.int16), full, np.full(2 * L, -32768, np.int16)])
    smp = np.stack([full[5:5 + L], np.full(L, -32768, np.int16), np.zeros(L, np.int16), np.full(L, 1234, np.int16)])
    rec = check_s16_equals_f64(ctx, src, smp)
    assert rec["ret"][2] == -1 and np.isnan(rec["coef"][2])      # all-zero sample: NaN coefficient, as F64
    assert rec["ret"][0] == 0 and rec["success"][0] == 1


def test_quantised_synth_pairs_recover_lag(ac, ctx):
    """Seeded F32 synth pairs quantised to 16 bits (round(x * 32767), clipped) at 1,440,000 frames find
    the F32 pairs' lag."""
    import torch
    L, n = 1440000, 8
    s = torch.empty(n, 2 * L, dtype=torch.float32, device="cuda")
    m = torch.empty(n, L, dtype=torch.float32, device="cuda")
    ctx.synth_pairs(0, 0x5EED, 0, n, L, ac.F32, s.data_ptr(), m.data_ptr())
    ref = ctx.xcorr_batch_torch(s, m)
    q = lambda x: torch.clamp(torch.round(x * 32767), -32768, 32767).to(torch.int16)  # noqa: E731
    got = ctx.xcorr_batch_torch(q(s), q(m))
    assert (got["lag"] == ref["lag"]).all() and (got["success"] == ref["success"]).all() and ref["success"].any()
    assert_same_bytes(got, ctx.xcorr_batch_torch(q(s).double() / 32768.0, q(m).double() / 32768.0))


@pytest.mark.parametrize("L", STATIC_LENGTHS)
def test_one_hot_probes(ac, ctx, L):
    """Closed-form probes (tests/golden/probes.py) quantised at amplitude 16384."""
    import probes as pr
    plan = pr.STATIC_PLANS[L]
    probes = pr.bin_probes(plan, L + 5, n_random=2, dense=False)[:6] + pr.seed_probes(plan, L + 6)[:4]
    srcs, smps = [], []
    for p in probes:
        s, m = p.build(np.float64)
        srcs.append(np.clip(np.round(s * 16384), -32768, 32767).astype(np.int16))
        smps.append(np.clip(np.round(m * 16384), -32768, 32767).astype(np.int16))
    check_s16_equals_f64(ctx, np.stack(srcs), np.stack(smps))


def test_refusals(ac, ctx):
    import torch
    L = 4096
    s = torch.zeros(2, 2 * L, dtype=torch.int16, device="cuda")
    m = torch.zeros(2, L, dtype=torch.int16, device="cuda")
    with pytest.raises(ac.AudiosyncCudaError, match="bad dtype"):
        ctx.synth_pairs(0, 1, 0, 2, L, ac.S16, s.data_ptr(), m.data_ptr())
    hs, hm = np.zeros((2, 2 * L), np.int16), np.zeros((2, L), np.int16)
    out = torch.zeros(2 * ac.RESULT_DTYPE.itemsize, dtype=torch.uint8, device="cuda")
    with pytest.raises(ac.AudiosyncCudaError, match="bad dtype"):
        ctx.xcorr_batch_device(0, s.data_ptr(), m.data_ptr(), 2, L, 3, out.data_ptr())
    for mem, ps, pm in ((ac.HOST, hs.ctypes.data, hm.ctypes.data), (ac.DEVICE, s.data_ptr(), m.data_ptr())):
        with pytest.raises(ac.AudiosyncCudaError, match="bad dtype"):
            ctx.xcorr_batch_records(ps, pm, 2, L, 3, mem)
        with pytest.raises(ac.AudiosyncCudaError, match="bad dtype"):
            ctx.xcorr_batch_ptr(ps, pm, 2, L, 3, mem)
    with pytest.raises(ac.AudiosyncCudaError, match="bad dtype"):
        ac.SessionPool(ctx, 0, 2, L, ac.S16)
