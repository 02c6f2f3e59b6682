"""The reference's UNMODIFIED orchestrator (src/audiosync.c: audiosync_run, the interval loop
of :226-259) driven by fake capture/download threads (oracle/harness/fake_io.c, the reader
protocol of src/ffmpeg_pipe.c), linked

  * against the reference's own src/cross_correlation.c + FFT stand-in  -> audiosync_harness_cpu
  * against libaudiosync_cuda.so, nothing else changed                  -> audiosync_harness_gpu

The second binary has exactly three undefined symbols that resolve into the GPU library:
cross_correlation, fftw_alloc_real, fftw_free -- the drop-in boundary of SURVEY 8b.  Both are
built by oracle/Makefile only where the reference's source checkout exists (REF=...); it is not
part of this repository, and without them the two tests that run them skip.

The two tests after them need no reference build: on the same pairs, the restated loop
(oracle_interval_loop) against the independent NumPy restatement and the generator's injected
lag, and the GPU library's drop-in call, driven through the same schedule, against the restated
loop.  Neither is a check against the reference's own audiosync_run.
"""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, ROOT)
from oracle import capi  # noqa: E402

REF_DIR = os.path.join(ROOT, "oracle", "_ref")
CPU_BIN = os.path.join(REF_DIR, "audiosync_harness_cpu")
GPU_BIN = os.path.join(REF_DIR, "audiosync_harness_gpu")
SEED, L = 0x5EED, 1440000


def _write_pair(tmp_path, pair_id):
    src, smp = capi.synth_pair(SEED, pair_id, L)
    ps, pm = tmp_path / ("src%d.f64" % pair_id), tmp_path / ("smp%d.f64" % pair_id)
    src.astype("<f8").tofile(ps); smp.astype("<f8").tofile(pm)
    return src, smp, str(ps), str(pm)


def _run(binary, ps, pm, debug=0):
    r = subprocess.run([binary, ps, pm, str(debug)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    m = re.search(r"ret=(-?\d+) lag=(-?\d+)", r.stdout)
    assert m, r.stdout
    return int(m.group(1)), int(m.group(2)), r.stderr


@pytest.mark.skipif(not os.path.exists(CPU_BIN), reason="oracle/_ref harness not built (needs the reference's source)")
@pytest.mark.parametrize("pair_id", [0, 3])
def test_cpu_harness_agrees_with_restated_loop(tmp_path, pair_id):
    """Pins oracle_interval_loop (and audiosync_cuda.interval_loop, which mirrors it) on the
    reference's real audiosync_run: same return value and same reported lag."""
    src, smp, ps, pm = _write_pair(tmp_path, pair_id)
    ret, lag, _ = _run(CPU_BIN, ps, pm)
    want = capi.interval_loop(src, smp)
    assert (ret, lag) == (want["final_ret"], want["final_lag"])
    if pair_id % 4 != 3:          # clean pair: accepted at the first interval, lag in ms
        assert ret == 0 and lag == round(capi.synth_true_lag(SEED, pair_id, L) * 1000.0 / 48000.0)
    else:                         # noisy pair: every interval is rejected, lag stays in frames
        assert ret == -1 and lag == capi.synth_true_lag(SEED, pair_id, L)


@pytest.mark.gpu
@pytest.mark.parametrize("pair_id", [0, 3, 5])
def test_unmodified_audiosync_run_on_the_gpu_library(tmp_path, pair_id):
    if not (os.path.exists(CPU_BIN) and os.path.exists(GPU_BIN)):
        pytest.skip("oracle/_ref harness binaries not present")
    _, _, ps, pm = _write_pair(tmp_path, pair_id)
    cpu = _run(CPU_BIN, ps, pm, debug=1)
    gpu = _run(GPU_BIN, ps, pm, debug=1)
    assert gpu[:2] == cpu[:2]
    # the LOG line of src/cross_correlation.c:278 appears once per evaluated interval in both
    pat = re.compile(r"(-?\d+) frames of delay with a confidence of (-?[\d.]+)")
    lc, lg = pat.findall(cpu[2]), pat.findall(gpu[2])
    assert len(lc) == len(lg) >= 1
    for (fc, cc), (fg, cg) in zip(lc, lg):
        assert fc == fg and abs(float(cc) - float(cg)) <= 1e-4


@pytest.mark.parametrize("pair_id", [0, 3, 5])
def test_restated_interval_loop_on_full_length_pairs(pair_id):
    """oracle_interval_loop against the NumPy restatement on every interval it evaluates, and its
    reported (ret, lag) against the injected lag."""
    from oracle import xcorr_numpy as xn
    src, smp = capi.synth_pair(SEED, pair_id, L)
    want = capi.interval_loop(src, smp)
    assert want["n"] >= 1
    for i in range(want["n"]):
        Li = xn.INTERV_SAMPLE[i]
        alt = xn.cross_correlation(src[:2 * Li], smp[:Li])
        assert (want["rets"][i], want["lags"][i]) == (alt["ret"], alt["lag"])
        assert abs(want["coefs"][i] - alt["coef"]) <= 1e-12
    if pair_id % 4 != 3:          # clean pair: accepted at the first interval that finds the lag, lag in ms
        assert want["final_ret"] == 0
        assert want["final_lag"] == round(capi.synth_true_lag(SEED, pair_id, L) * 1000.0 / 48000.0)
    else:                         # noisy pair: every interval is rejected, lag stays in frames
        assert want["n"] == len(xn.INTERV_SAMPLE)
        assert want["final_ret"] == -1 and want["final_lag"] == capi.synth_true_lag(SEED, pair_id, L)


@pytest.mark.gpu
@pytest.mark.parametrize("pair_id", [0, 3, 5])
def test_dropin_interval_schedule_matches_restated_loop(pair_id):
    """The GPU library's cross_correlation, called the way audiosync_run calls it (source in an
    fftw_alloc_real buffer, sample in ordinary host memory) on the interval schedule, against
    oracle_interval_loop: every evaluated interval and the reported (ret, lag)."""
    import audiosync_cuda as ac
    src, smp = capi.synth_pair(SEED, pair_id, L)
    want = capi.interval_loop(src, smp)
    with ac.RealBuffer(2 * L) as buf:
        buf.array[:] = src
        got = ac.interval_loop(None, None, call=lambda n: ac.cross_correlation_ptr(buf.ptr, smp.ctypes.data, n))
    assert (got["n"], got["final_ret"], got["final_lag"]) == (want["n"], want["final_ret"], want["final_lag"])
    assert got["rets"] == want["rets"] and got["lags"] == want["lags"]
    for g, w in zip(got["coefs"], want["coefs"]):
        assert abs(g - w) <= 1e-4
