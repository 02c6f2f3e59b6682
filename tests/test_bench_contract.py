"""bench.py contract checks: the reference arm prints exactly one JSON line on stdout (library
banners must not leak into it) with the keys its readers expect; --steps sets the number of
timed steps, and --dump-outputs writes the same arrays for the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], cwd=ROOT, capture_output=True,
                         text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    return json.loads(out.stdout.strip().splitlines()[-1])


def _dumped(path):
    arrays = {f[:-4]: np.load(os.path.join(path, f)) for f in sorted(os.listdir(path))}
    assert all(a.dtype == np.float64 and a.shape == arrays["pair_id"].shape for a in arrays.values())
    return arrays


def test_reference_arm_dump_outputs_are_reproducible(tmp_path):
    from oracle import capi
    L = 24000
    for run in ("a", "b"):
        line = _bench("--impl", "reference", "--steps", "1", "--warmup", "0", "--sample-len", str(L),
                      "--dump-outputs", str(tmp_path / run))
    a, b = _dumped(tmp_path / "a"), _dumped(tmp_path / "b")
    assert sorted(a) == ["lag", "pair_id"] and len(a["lag"]) >= 8
    assert all(np.array_equal(a[k], b[k]) for k in a)
    seed = line["config"]["seed"]
    assert [int(x) for x in a["lag"]] == [capi.synth_true_lag(seed, int(i), L) for i in a["pair_id"]]


def test_dump_outputs_stays_within_64_mb(tmp_path):
    n = 900000                         # 10 float64 arrays of n rows: 72 MB before sampling
    code = ("import sys, numpy as np; sys.path.insert(0, %r); import bench; "
            "bench.dump_outputs(%r, {'pair_id': range(%d), **{'f%%d' %% i: np.arange(%d) for i in range(9)}})"
            % (ROOT, str(tmp_path), n, n))
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert sum(os.path.getsize(tmp_path / f) for f in os.listdir(tmp_path)) <= 64_000_000
    d = _dumped(tmp_path)
    assert len(d) == 10 and 0 < len(d["pair_id"]) < n
    assert (np.diff(d["pair_id"]) > 0).all() and all(np.array_equal(d["f%d" % i], d["pair_id"]) for i in range(9))


@pytest.mark.gpu
def test_steps_set_the_timed_steps_and_dumps_are_reproducible(tmp_path):
    import audiosync_cuda as ac
    from oracle import capi
    L, n = 144000, 16
    lines = {}
    for steps in (2, 3):
        lines[steps] = _bench("--steps", str(steps), "--warmup", "1", "--pairs", str(n), "--sample-len", str(L),
                              "--no-e2e", "--no-latency", "--no-cpu-baseline", "--dump-outputs", str(tmp_path / str(steps)))
        assert lines[steps]["steps"] == steps
    assert lines[2]["gpu_launches"] * 3 == lines[3]["gpu_launches"] * 2 > 0
    a, b = _dumped(tmp_path / "2"), _dumped(tmp_path / "3")
    assert sorted(a) == sorted(("pair_id",) + ac.RESULT_DTYPE.names)
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k
    seed = lines[3]["config"]["seed"]
    assert [int(x) for x in a["lag"]] == [capi.synth_true_lag(seed, int(i), L) for i in a["pair_id"]]


def test_reference_arm_prints_one_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--sample-len", "144000"], cwd=ROOT, capture_output=True, text=True,
                         timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, out.stdout[:500]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "pairs/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["warmup"] == 0
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["gpu_launches"] == 0


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                          "--steps", "1", "--warmup", "0", "--sample-len", "144000"], cwd=ROOT, env=env,
                         capture_output=True, text=True, timeout=600)
    assert out.returncode == 0 and out.stdout.strip() == ""
