#!/usr/bin/env python3
"""Benchmark of the FFT cross-correlation hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

Metric (BASELINE.json): xcorr pairs/sec at L = 1,440,000 (N = 2,880,000), batched.
A step is one pass of the whole path (forward FFTs, conj-multiply, inverse FFT,
|r| argmax, fold, Pearson) over one batch of device-resident fp32 pairs --
config[3]: 4,096 pairs per GPU.  With N GPUs every rank owns its own 4,096
pairs (pairs are independent: no collective on the data path), so the N = 8 run
is config[4] (32,768 pairs) and scaling is weak.  torch / torch.distributed are
used for device buffers, the barrier and the max-over-ranks only.

The printed JSON line carries, besides the base contract:
  roofline      -- dominant kernel: algorithmic bytes per launch / its average
                   launch duration vs MEASURED_PEAKS.json.  `value` is timed with
                   no per-launch events (the shipped configuration: the stages
                   are chained with programmatic dependent launch); the per-kernel
                   durations come from a second, identical pass of K steps with
                   CUDA events around every launch on its own stream;
                   `kernels` lists all four with their own fractions;
  path_roofline -- the whole path three ways: `frac` with SURVEY 8(d)'s 21*L*4
                   bytes/pair (the survey's accounting), `frac_moved` with the
                   17*L*4 this design moves, `frac_dram` with the DRAM bytes ncu
                   measured (profiles/traffic.json);
  e2e           -- the same metric through the host-facing C-ABI batch call with
                   pinned HOST buffers of the reference ABI's dtype, double (uploads
                   and result download timed); `e2e_variants` adds fp32-pinned and
                   f64-pageable host buffers;
  in_library    -- (N > 1, rank 0) ONE context / one process driving all N devices
                   through audiosync_cuda_xcorr_batch(HOST) and through
                   ..._batch_device per device: north_star's dispatcher, beside the
                   process-per-GPU figure;
  cpu_baseline  -- the reference's CPU path (oracle/_ref, FFT shim) on this box.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "old-audiosync_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

# The CPU legs time the reference's own src/cross_correlation.c.  FFTW3 is not installed, so its
# FFT calls run on the stand-in of oracle/fftw3_shim.c; for TIMING that stand-in is pointed at
# Intel MKL's DFTI (exported by PyTorch's libtorch_cpu.so), an FFTW-class library, one thread per
# transform like FFTW's default plans.  The JSON line names the backend that actually ran.
def _enable_fast_cpu_fft():
    try:
        import importlib.util
        spec = importlib.util.find_spec("torch")
        lib = os.path.join(list(spec.submodule_search_locations)[0], "lib", "libtorch_cpu.so")
        if os.path.exists(lib):
            os.environ.setdefault("ORACLE_FFT_BACKEND", "mkl")
            os.environ.setdefault("ORACLE_MKL_LIB", lib)
    except Exception:
        pass


_enable_fast_cpu_fft()

L_HEADLINE = 1440000
PAIRS_PER_GPU = 4096
SEED = 0x5EED + 4          # seed + config number (SURVEY 8d)
METRIC = "xcorr_pairs_per_sec_L1440000"
UNIT = "pairs/s"

# Algorithmic bytes per pair, in units of U = L * 4 bytes (fp32 device-resident).
# SURVEY 8(d) schedule: 21 U for the whole path.  Per kernel of THIS design:
#   col_fwd   reads 2U (source) + 1U (sample, zero half never read), writes 4U      = 7 U
#   row_fused reads 4U (both planes), writes 2U (product rows, in place)           = 6 U
#   col_inv   reads 2U                                                             = 2 U
#   pearson   reads 2U (the two windows)                                           = 2 U
KERNEL_U = {"col_fwd": 7, "row_fused": 6, "col_inv_argmax": 2, "pearson": 2}
PATH_U = 21          # SURVEY 8(d)'s minimal-pass schedule
MOVED_U = 17         # what this design moves (K_B fuses forward pass 2 with inverse pass 1)


# stdout carries exactly ONE line, the JSON result: everything libraries print to fd 1 (NCCL's
# version banner, for one) is sent to stderr, and the result is written to the saved descriptor.
_RESULT_FD = None


def _claim_stdout():
    global _RESULT_FD
    if _RESULT_FD is None:
        sys.stdout.flush()
        _RESULT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_RESULT_FD, data)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5,
                    help="timed steps (repetitions) of every throughput leg; the latency legs time a fixed "
                         "number of calls and the CPU baseline about 12 s")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--pairs", type=int, default=PAIRS_PER_GPU, help="pairs per GPU per step")
    ap.add_argument("--sample-len", type=int, default=L_HEADLINE)
    ap.add_argument("--e2e-pairs", type=int, default=192)
    ap.add_argument("--wave", type=int, default=0, help="pairs per kernel wave (0 = library default)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-inlib", action="store_true", help="skip the in-library multi-GPU leg (N > 1)")
    ap.add_argument("--inlib-pairs", type=int, default=1024, help="device-resident pairs per GPU in the in-library leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path returned in its last step as DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    return args


DUMP_BYTES = 64_000_000


def dump_outputs(path, arrays):
    """Writes equal-length 1-D arrays as `path`/<name>.npy in float64 (every field of a result
    record, integers included, is exact in float64).  Above DUMP_BYTES in all, a fixed seeded
    sample of the rows is written; `pair_id` says which pairs the rows belong to."""
    import numpy as np
    n = len(arrays["pair_id"])
    keep = (DUMP_BYTES - 1024 * len(arrays)) // (8 * len(arrays))     # 1 KiB per .npy header: headroom
    rows = np.sort(np.random.default_rng(0).choice(n, keep, replace=False)) if n > keep else slice(None)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), np.asarray(a, dtype=np.float64)[rows])


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return float(json.load(open(path))["hbm_gbs"]), "measured"
        except Exception:
            pass
    return 6650.0, "fallback"


class ClockSampler:
    """SM clock, power and throttle reasons sampled (NVML, every 50 ms) while the timed region runs."""

    def __init__(self, index: int):
        self.index, self.on, self.s, self.t, self.h, self.nv = index, False, [], None, None, None

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
        except Exception:
            self.nv = None
            return
        self.on = True
        self.t = threading.Thread(target=self._run, daemon=True)
        self.t.start()

    def _run(self):
        nv = self.nv
        while self.on:
            try:
                self.s.append((nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                               nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0,
                               nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)))
            except Exception:
                break
            time.sleep(0.05)

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        self.on = False
        self.t.join(timeout=2)
        nv = self.nv
        smax = nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM)
        names = {"hw_slowdown": nv.nvmlClocksEventReasonHwSlowdown,
                 "hw_thermal_slowdown": nv.nvmlClocksEventReasonHwThermalSlowdown,
                 "sw_thermal_slowdown": nv.nvmlClocksEventReasonSwThermalSlowdown,
                 "sw_power_cap": nv.nvmlClocksEventReasonSwPowerCap}
        # the first sample can predate the load: drop it when there are others
        s = self.s[1:] if len(self.s) > 2 else self.s
        clk = sorted(x[0] for x in s)
        pw = sorted(x[1] for x in s)
        reasons = sorted(k for k, bit in names.items() if any(x[2] & bit for x in s))
        return {"sm_mhz": statistics.median(clk) if clk else None, "sm_min_mhz": clk[0] if clk else None,
                "sm_max_mhz": smax, "power_w_median": statistics.median(pw) if pw else None,
                "reasons": reasons, "samples": len(s)}


# ------------------------------------------------------------------ reference arm / CPU baseline

def cpu_reference_run(sample_len: int, n_pairs: int, threads: int, seed: int, distinct: int = 0):
    """Times the reference's CPU path on n_pairs seeded pairs with `threads` concurrent callers.

    Uses oracle/_ref (the reference's own src/cross_correlation.c compiled against the
    FFT stand-in; kind "reference") when that build is present, else the restatement
    (kind "port").  Only `distinct` (default: all) different pairs are generated and they
    are cycled through, so a many-second sample does not need gigabytes of inputs.
    Returns (seconds, kind, backend, lags).
    """
    from oracle import capi
    ref = capi.ref_lib()
    kind = "reference" if ref is not None else "port"
    distinct = min(n_pairs, distinct or n_pairs)
    lags = [None] * n_pairs
    inputs = [capi.synth_pair(seed, i, sample_len) for i in range(distinct)]   # outside the timing

    def work(tid):
        for i in range(tid, n_pairs, threads):
            s, p = inputs[i % distinct]
            if ref is not None:
                lags[i] = capi.ref_cross_correlation(s, p)[1]
            else:
                lags[i] = capi.cross_correlation(s, p)["lag"]

    if n_pairs:                       # warm the stand-in's twiddle cache like a long-lived process
        s, p = inputs[0]
        (capi.ref_cross_correlation if ref is not None else capi.cross_correlation)(s, p)
    t0 = time.perf_counter()
    th = [threading.Thread(target=work, args=(t,)) for t in range(threads)]
    [t.start() for t in th]
    [t.join() for t in th]
    dt = time.perf_counter() - t0
    for i in range(n_pairs):
        assert lags[i] == capi.synth_true_lag(seed, i % distinct, sample_len), "CPU reference lost a lag"
    return dt, kind, capi.backend(), lags


def cpu_baseline_sample(sample_len: int, seed: int, target_s: float = 12.0):
    """About `target_s` seconds of the reference's CPU path with every host core busy."""
    cores = os.cpu_count() or 1
    callers = max(1, cores // 2)          # the reference runs two FFT threads per call
    probe = max(callers, 4)
    dt, kind, backend, _ = cpu_reference_run(sample_len, probe, callers, seed)
    rate = probe / dt
    npairs = int(max(2 * callers, min(4096, rate * target_s)))
    npairs -= npairs % callers
    dt, kind, backend, _ = cpu_reference_run(sample_len, npairs, callers, seed, distinct=2 * callers)
    return {"value": npairs / dt, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": "%d pairs (%d distinct, cycled) of the same workload, %d concurrent callers x 2 FFT "
                      "threads, %.1f s wall, FFT backend %s (in place of FFTW3, which is not installed)"
                      % (npairs, min(npairs, 2 * callers), callers, dt, backend)}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    L = args.sample_len
    cores = os.cpu_count() or 1
    # the reference runs two FFT threads per call: nproc/2 concurrent callers use every core
    callers = max(1, cores // 2)
    per_step = max(4 * callers, 8)
    for _ in range(args.warmup):
        cpu_reference_run(L, callers, callers, SEED)
    times = []
    kind = backend = lags = None
    for _ in range(args.steps):
        dt, kind, backend, lags = cpu_reference_run(L, per_step, callers, SEED)
        times.append(dt)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"pair_id": range(per_step), "lag": lags})
    total = sum(times)
    value = per_step * args.steps / total
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
        "data": "synthetic (seeded integer generator, SURVEY 8d)",
        "config": {"workload": "reference CPU path (src/cross_correlation.c) on %d-pair samples of "
                               "config[3]: L=%d, N=%d" % (per_step, L, 2 * L),
                   "sample_len": L, "pairs_per_step": per_step, "seed": SEED},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": "%d pairs/step x %d steps, %d concurrent callers x 2 FFT threads, "
                                   "FFT backend %s (in place of FFTW3, which is not installed)"
                                   % (per_step, args.steps, callers, backend)},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ------------------------------------------------------------------ single-pair latency

def measure_latency(ctx, ac, torch, dev, local, stream, d_src, d_smp, d_res, n, L, reps=200):
    """BASELINE config 3: one L-frame pair per call.

    (i) device-resident fp32 inputs, CUDA events around each call on the launching stream; the
    calls rotate through 16 different resident pairs (276 MB at L = 1.44M > L2), so no call finds
    its inputs in cache.  (ii) the unchanged C signature `cross_correlation(double*, double*, ...)`
    on pinned host doubles: wall clock, upload of 34.56 MB and the 24-byte answer included.
    """
    import numpy as np
    out = {}
    rot = min(16, n)
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for i in range(20 + reps):
        k = i % rot
        if i >= 20:
            ev[i - 20][0].record(stream)
        ctx.xcorr_batch_device(local, d_src.data_ptr() + k * 2 * L * 4, d_smp.data_ptr() + k * L * 4, 1, L,
                               ac.F32, d_res.data_ptr(), stream.cuda_stream)
        if i >= 20:
            ev[i - 20][1].record(stream)
    torch.cuda.synchronize(dev)
    t = sorted(a.elapsed_time(b) * 1e3 for a, b in ev)
    out["device_resident_f32_us"] = {"p50": t[len(t) // 2], "p95": t[int(len(t) * 0.95)], "calls": reps,
                                     "launches_per_call": 4}
    # (ii) drop-in C ABI on host doubles (buffers from the library's pinned fftw_alloc_real)
    lib = ac.lib()
    import ctypes as C
    ps, pm = lib.fftw_alloc_real(2 * L), lib.fftw_alloc_real(L)
    hs = np.ctypeslib.as_array(C.cast(ps, C.POINTER(C.c_double)), shape=(2 * L,))
    hm = np.ctypeslib.as_array(C.cast(pm, C.POINTER(C.c_double)), shape=(L,))
    hs[:] = d_src[: 2 * L].cpu().numpy(); hm[:] = d_smp[:L].cpu().numpy()
    lag, coef = C.c_long(0), C.c_double(0.0)
    wall = []
    for i in range(5 + 30):
        t0 = time.perf_counter()
        rc = lib.cross_correlation(ps, pm, L, C.byref(lag), C.byref(coef))
        if i >= 5:
            wall.append((time.perf_counter() - t0) * 1e3)
    wall.sort()
    out["c_abi_host_f64_ms"] = {"p50": wall[len(wall) // 2], "p95": wall[int(len(wall) * 0.95)], "calls": len(wall),
                                "h2d_bytes_per_call": 3 * L * 8, "ret": rc, "lag": lag.value}
    # (iii) the reference's interval schedule (src/audiosync.c:226-259): six calls on growing
    # prefixes of the same two buffers, with and without interval-schedule residency
    if L == L_HEADLINE:
        sched = {}
        for resident in (False, True):
            lib.audiosync_cuda_set_residency(1 if resident else 0)
            tot = []
            b0 = ac.dropin_stats()[1]
            for rep in range(2 + 10):
                t0 = time.perf_counter()
                for Li in ac.INTERV_SAMPLE:
                    lib.cross_correlation(ps, pm, Li, C.byref(lag), C.byref(coef))
                if rep >= 2:
                    tot.append((time.perf_counter() - t0) * 1e3)
            tot.sort()
            sched["resident" if resident else "full_upload"] = {
                "p50_ms_six_calls": tot[len(tot) // 2],
                "h2d_bytes_six_calls": (ac.dropin_stats()[1] - b0) // 12}
        lib.audiosync_cuda_set_residency(0)
        out["c_abi_interval_schedule"] = sched
        # (iv) the same schedule for many concurrent sessions through the session pool: frames are
        # appended as they "arrive" (each crosses PCIe once, f64le), every interval is ONE batched call
        try:
            ns = 24
            with ac.SessionPool(ctx, local, ns, L, ac.F32) as pool:
                def one_round():
                    prev = 0
                    for Li in ac.INTERV_SAMPLE:
                        for slot in range(ns):
                            lib.audiosync_cuda_pool_append_async(pool._h, slot, ps + 16 * prev, 2 * (Li - prev),
                                                                 pm + 8 * prev, Li - prev)
                        rec = pool.run(0, ns, Li)
                        prev = Li
                    for slot in range(ns):
                        pool.reset(slot)
                    return rec
                one_round()
                t0 = time.perf_counter()
                rec = one_round()
                dt = time.perf_counter() - t0
            out["session_pool_schedule"] = {
                "sessions": ns, "intervals": len(ac.INTERV_SAMPLE), "ms_total": dt * 1e3,
                "ms_per_session_schedule": dt * 1e3 / ns, "h2d_bytes_per_session": 3 * L * 8,
                "h2d_gbs": ns * 3 * L * 8 / dt / 1e9, "slots": "f32 (converted on arrival)",
                "last_interval_lag": int(rec["lag"][0])}
        except Exception as e:          # never let the extra measurement take the bench line down
            out["session_pool_schedule"] = {"error": str(e)[:200]}
    lib.fftw_free(ps); lib.fftw_free(pm)
    return out


# ------------------------------------------------------------------ in-library multi-GPU dispatcher

def measure_in_library(ac, torch, n_dev, L, args, per_gpu_process_value):
    """north_star (3) / SURVEY 8(e): ONE process and ONE context drive all `n_dev` devices.

    (a) device-resident: `inlib_pairs` fp32 pairs per device, generated on each device; every step
        enqueues the whole path on every device through audiosync_cuda_xcorr_batch_device (one
        stream per device, no host synchronisation between devices); time = max over devices of the
        CUDA-event span on that device's stream.  (b) host-facing: one pinned fp32 batch through
        audiosync_cuda_xcorr_batch(memspace=HOST), which shards contiguous pair blocks over the
        devices (one host thread + stream per device) and gathers the records.
    """
    out = {"devices": n_dev}
    npd = args.inlib_pairs
    with ac.Context(list(range(n_dev))) as ctx:
        bufs = []
        for g in range(n_dev):
            dev = torch.device("cuda", g)
            with torch.cuda.device(dev):
                st = torch.cuda.Stream(dev)
                src = torch.empty(npd * 2 * L, dtype=torch.float32, device=dev)
                smp = torch.empty(npd * L, dtype=torch.float32, device=dev)
                res = torch.zeros(npd * ac.RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
                ctx.synth_pairs(g, SEED, g * npd, npd, L, ac.F32, src.data_ptr(), smp.data_ptr(), st.cuda_stream)
                bufs.append((dev, st, src, smp, res))

        # one host thread + one stream per device, as north_star (3) describes (ctypes releases the GIL)
        def drive(g, nsteps, timed):
            dev, st, src, smp, res = bufs[g]
            torch.cuda.set_device(dev)
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            if timed:
                gate.wait()
            a.record(st)
            for _ in range(nsteps):
                ctx.xcorr_batch_device(g, src.data_ptr(), smp.data_ptr(), npd, L, ac.F32, res.data_ptr(), st.cuda_stream)
            b.record(st)
            torch.cuda.synchronize(dev)
            return a.elapsed_time(b)

        from concurrent.futures import ThreadPoolExecutor
        gate = threading.Barrier(n_dev)
        steps = args.steps
        with ThreadPoolExecutor(n_dev) as pool:
            list(pool.map(lambda g: drive(g, max(2, args.warmup), False), range(n_dev)))
            t0 = time.perf_counter()
            spans = list(pool.map(lambda g: drive(g, steps, True), range(n_dev)))
            wall = time.perf_counter() - t0
        ms = max(spans)
        from oracle import capi
        bad = 0
        for g, (dev, st, src, smp, res) in enumerate(bufs):
            r = res.cpu().numpy().view(ac.RESULT_DTYPE)
            bad += sum(1 for i in range(0, npd, max(1, npd // 32))
                       if int(r["lag"][i]) != capi.synth_true_lag(SEED, g * npd + i, L))
        v = n_dev * npd * steps / (ms * 1e-3)
        out["device_resident"] = {"value": v, "unit": UNIT, "pairs_per_gpu": npd, "steps": steps, "ms_max_over_devices": ms,
                                  "wall_ms": wall * 1e3, "lag_mismatches": bad,
                                  "vs_process_per_gpu": v / (n_dev * per_gpu_process_value),
                                  "api": "audiosync_cuda_xcorr_batch_device on every device of one context"}
        # (b) host-facing call, pinned fp32 batch sharded by the library
        ne = min(args.e2e_pairs, npd) * n_dev
        h_src = torch.empty(ne * 2 * L, dtype=torch.float32, pin_memory=True)
        h_smp = torch.empty(ne * L, dtype=torch.float32, pin_memory=True)
        per = ne // n_dev
        for g, (dev, st, src, smp, res) in enumerate(bufs):
            h_src[g * per * 2 * L:(g + 1) * per * 2 * L].copy_(src[: per * 2 * L])
            h_smp[g * per * L:(g + 1) * per * L].copy_(smp[: per * L])
        for dev, *_ in bufs:
            torch.cuda.synchronize(dev)
        o = ctx.xcorr_batch_ptr(h_src.data_ptr(), h_smp.data_ptr(), ne, L, ac.F32, ac.HOST)
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            o = ctx.xcorr_batch_ptr(h_src.data_ptr(), h_smp.data_ptr(), ne, L, ac.F32, ac.HOST)
        dt = time.perf_counter() - t0
        badh = sum(1 for g in range(n_dev) for i in range(0, per, max(1, per // 16))
                   if int(o["lags"][g * per + i]) != capi.synth_true_lag(SEED, g * npd + i, L))
        out["host_batch"] = {"value": ne * reps / dt, "unit": UNIT, "pairs_per_call": ne, "host_dtype": "f32",
                             "host_memory": "pinned", "h2d_gbs_total": ne * 3 * L * 4 * reps / dt / 1e9,
                             "lag_mismatches": badh, "api": "audiosync_cuda_xcorr_batch(memspace=HOST), devices = all"}
    return out


# ------------------------------------------------------------------ our arm

def main():
    args = parse()
    _claim_stdout()
    if args.impl == "reference":
        run_reference_arm(args)
        return

    import numpy as np
    import torch
    import torch.distributed as dist
    import audiosync_cuda as ac

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world > 1:
        # several processes share this host's cores: each library instance gets its share of copy
        # threads (pageable staging / host narrowing; below 8 the library feeds page-locked doubles
        # through the copy engine alone) -- read by the library on first use
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
        os.environ.setdefault("AUDIOSYNC_CUDA_COPY_THREADS",
                              str(max(1, min(12, len(os.sched_getaffinity(0)) * 3 // 4 // max(1, local_world)))))
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    # One process per GPU: run on the CPUs (and allocate pinned host memory on the NUMA node)
    # next to this rank's GPU, as a deployment would; the e2e leg is a PCIe / host-memory number.
    numa = "unbound"
    all_cpus = os.sched_getaffinity(0)
    try:
        import pynvml
        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local))
        numa = "nvml cpu affinity (%d cpus)" % len(os.sched_getaffinity(0))
    except Exception:
        pass

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    L, n = args.sample_len, args.pairs
    U = L * 4
    first_pair, _n = ac.shard_pairs(world * n, world, rank)   # contiguous block split of the pair ids
    assert _n == n
    ctx = ac.Context([local])
    if args.wave:
        ctx.set_wave_pairs(args.wave)
    plan = ctx.describe_plan(L)

    d_src = torch.empty(n * 2 * L, dtype=torch.float32, device=dev)
    d_smp = torch.empty(n * L, dtype=torch.float32, device=dev)
    d_res = torch.zeros(n * ac.RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    # A dedicated (non-default) stream: the library maps a NULL stream handle to its own
    # internal stream, so events recorded on torch's default stream would not bracket the kernels.
    stream = torch.cuda.Stream(dev)
    assert stream.cuda_stream != 0
    ctx.synth_pairs(local, SEED, first_pair, n, L, ac.F32, d_src.data_ptr(), d_smp.data_ptr(),
                    stream.cuda_stream)
    torch.cuda.synchronize(dev)

    def step():
        ctx.xcorr_batch_device(local, d_src.data_ptr(), d_smp.data_ptr(), n, L, ac.F32,
                               d_res.data_ptr(), stream.cuda_stream)

    for _ in range(args.warmup):
        step()
    barrier()
    launches0 = ctx.launch_count()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record(stream)
    for _ in range(args.steps):
        step()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    clocks = sampler.stop() if rank == 0 else None
    launches = ctx.launch_count() - launches0
    res = d_res.cpu().numpy().view(ac.RESULT_DTYPE)      # what the last timed step returned
    if args.dump_outputs:
        everyone = ac.gather_results(res, world * n, dst=0)
        if rank == 0:
            dump_outputs(args.dump_outputs, {"pair_id": range(world * n),
                                             **{f: everyone[f] for f in ac.RESULT_DTYPE.names}})
    # per-kernel durations: the same K steps again, every launch bracketed by CUDA events on its
    # own stream (kept out of the timed region above: the event records sit between the
    # PDL-chained stage launches)
    ctx.profile_enable(True)
    ctx.profile_reset()
    p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    p0.record(stream)
    for _ in range(args.steps):
        step()
    p1.record(stream)
    torch.cuda.synchronize(dev)
    ms_profiled = p0.elapsed_time(p1)
    prof = ctx.profile_read()
    ctx.profile_enable(False)

    # correctness of what was timed: every pair recovers its injected lag
    from oracle import capi   # checker only (synth_true_lag), never the thing measured
    bad = sum(1 for i in range(0, n, max(1, n // 256))
              if int(res["lag"][i]) != capi.synth_true_lag(SEED, first_pair + i, L))
    ok_flags = int(res["success"].sum())

    t = torch.tensor([ms, float(launches), float(bad)], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone(); dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        tsum = t.clone(); dist.all_reduce(tsum, op=dist.ReduceOp.SUM)
        ms, launches, bad = float(tmax[0]), int(tsum[1]), int(tsum[2])
    value = world * n * args.steps / (ms * 1e-3)

    # ---- end to end: host-facing C-ABI batch call on HOST buffers -----------------------------
    # headline: pinned doubles, the dtype the reference ABI's callers hold (f64le from ffmpeg), in
    # the library's default configuration -- LOSSLESS host narrowing: pairs whose doubles are exact
    # images of floats (decoded audio always is; so is the seeded generator's) are converted to fp32
    # by the library's copy threads while others go up as doubles on the copy engine, both at once;
    # every result bit equals the un-narrowed call's (tests/test_gpu_parity.py).  Variants: the same
    # with narrowing off (the doubles cross the link as they are), fp32 pinned, pageable doubles.
    # Uploads, the host-side conversion and the result download are inside the timed region.
    e2e = None
    e2e_variants = {}
    if not args.no_e2e:
        def e2e_leg(tdt, acdt, pinned, ne, reps, narrow=ac.NARROW_LOSSLESS):
            esz = 4 if acdt == ac.F32 else 8
            h_src = torch.empty(ne * 2 * L, dtype=tdt, pin_memory=pinned)
            h_smp = torch.empty(ne * L, dtype=tdt, pin_memory=pinned)
            h_src.copy_(d_src[: ne * 2 * L]); h_smp.copy_(d_smp[: ne * L])     # exact in both dtypes
            torch.cuda.synchronize(dev)
            ctx.set_host_narrowing(narrow)
            out = None
            for _ in range(2):
                out = ctx.xcorr_batch_ptr(h_src.data_ptr(), h_smp.data_ptr(), ne, L, acdt, ac.HOST)
            barrier()
            ctx.host_feed_stats(reset=True)
            t0 = time.perf_counter()
            for _ in range(reps):
                out = ctx.xcorr_batch_ptr(h_src.data_ptr(), h_smp.data_ptr(), ne, L, acdt, ac.HOST)
            torch.cuda.synchronize(dev)
            dt = time.perf_counter() - t0
            fed_direct, fed_narrowed = ctx.host_feed_stats(reset=True)
            ctx.set_host_narrowing(ac.NARROW_LOSSLESS)
            assert all(int(out["lags"][i]) == int(res["lag"][i]) for i in range(ne))
            tt = torch.tensor([dt], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
            del h_src, h_smp
            link_bytes = (ne * reps * 3 * L * esz) if esz == 4 else (fed_direct * 3 * L * 8 + fed_narrowed * 3 * L * 4)
            return {"value": world * ne * reps / float(tt[0]), "unit": UNIT,
                    "h2d_bytes_per_step": ne * 3 * L * esz, "d2h_bytes_per_step": ne * ac.RESULT_DTYPE.itemsize,
                    "pairs_per_step": ne, "host_dtype": "f32" if esz == 4 else "f64",
                    "host_memory": "pinned" if pinned else "pageable", "host_binding": numa,
                    "host_narrowing": (None if esz == 4 else ["off", "lossless", "always"][narrow]),
                    "copy_threads": ac.copy_threads(),
                    "pairs_fed_as_doubles": fed_direct, "pairs_narrowed_on_host": fed_narrowed,
                    "host_gbs_per_gpu": ne * 3 * L * esz * reps / float(tt[0]) / 1e9,
                    "link_gbs_per_gpu": link_bytes / float(tt[0]) / 1e9,
                    "bound": "pcie + host copy threads (%.2f MB of host input per pair)" % (3 * L * esz / 1e6),
                    "api": "audiosync_cuda_xcorr_batch(memspace=HOST)"}
        ne = min(args.e2e_pairs, n)
        reps = args.steps
        e2e = e2e_leg(torch.float64, ac.F64, True, max(1, ne // 2), reps)
        if os.environ.get("E2E_ONLY_HEADLINE") == "1":            # tools/e2e_feed.sh: feed-policy sweeps
            emit({"e2e": e2e, "e2e_variants": {}})
            return
        e2e_variants["f64_pinned_narrowing_off"] = e2e_leg(torch.float64, ac.F64, True, max(1, ne // 2), reps, narrow=ac.NARROW_OFF)
        e2e_variants["f32_pinned"] = e2e_leg(torch.float32, ac.F32, True, ne, reps)
        e2e_variants["f64_pageable"] = e2e_leg(torch.float64, ac.F64, False, max(1, ne // 4), reps)
        e2e_variants["f64_pageable_narrowing_off"] = e2e_leg(torch.float64, ac.F64, False, max(1, ne // 4), reps, narrow=ac.NARROW_OFF)

    # ---- config 3: single-pair latency at this length (rank 0 only) --------------------------
    latency = None
    if rank == 0 and not args.no_latency:
        latency = measure_latency(ctx, ac, torch, dev, local, stream, d_src, d_smp, d_res, n, L)

    # ---- north_star (3): the in-library dispatcher -- one process, one context, all N devices --
    in_library = None
    if world > 1 and not args.no_inlib:
        # the other ranks must wait on the HOST: an NCCL barrier is a kernel spinning on their GPUs,
        # which rank 0 is about to drive -- a gloo group keeps the devices free
        host_group = dist.new_group(backend="gloo")
        barrier()
        torch.cuda.synchronize(dev)
        dist.barrier(group=host_group)
        if rank == 0:
            try:
                in_library = measure_in_library(ac, torch, world, L, args, value / world)
            except Exception as e:                  # never let the extra leg take the bench line down
                in_library = {"error": str(e)[:300]}
        dist.barrier(group=host_group)
        barrier()

    if rank == 0:
        peak, peak_kind = measured_peaks()
        # dominant kernel by device time inside the timed region
        dom = max(KERNEL_U, key=lambda k: prof.get(k, (0, 0.0))[1])
        n_launch, tot_ms = prof[dom]
        pairs_per_launch = n * args.steps / max(1, n_launch)
        alg_bytes = KERNEL_U[dom] * U * pairs_per_launch
        avg_ms = tot_ms / max(1, n_launch)
        achieved = alg_bytes / (avg_ms * 1e-3) / 1e9
        traffic = None
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
                if dom in tj and tj[dom].get("bytes_per_pair"):
                    traffic = tj[dom]["bytes_per_pair"] * pairs_per_launch
            except Exception:
                traffic = None
        total_kernel_ms = sum(v[1] for v in prof.values())
        shares = {k: round(v[1] / total_kernel_ms, 4) for k, v in prof.items() if v[1] > 0}
        tj = {}
        if os.path.exists(tpath):
            try:
                tj = json.load(open(tpath))
            except Exception:
                tj = {}
        kernels = {}
        for k, u in KERNEL_U.items():
            nl, tm = prof.get(k, (0, 0.0))
            if nl == 0 or tm <= 0:
                continue
            us_pair = 1e3 * tm / (n * args.steps)
            ach = u * U / (us_pair * 1e-6) / 1e9
            kernels[k] = {"us_per_pair": round(us_pair, 3), "alg_bytes_per_pair": u * U, "achieved_gbs": round(ach, 1),
                          "frac": round(ach / peak, 4),
                          "dram_bytes_per_pair_ncu": tj.get(k, {}).get("bytes_per_pair")}
        dram_pair = sum(v.get("bytes_per_pair", 0) for k, v in tj.items() if k in KERNEL_U) or None
        pairs_s_gpu = value / world
        path_achieved = PATH_U * U * pairs_s_gpu / 1e9
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic (seeded integer "
            "generator, SURVEY 8d; generated on device)",
            "config": {"workload": "config[3]: %d pairs/GPU of L=%d frames (N=%d real points), "
                                   "device-resident fp32, whole path incl. argmax + Pearson" % (n, L, 2 * L),
                       "sample_len": L, "pairs_per_gpu": n, "total_pairs": world * n, "plan": plan, "seed": SEED,
                       "inputs_larger_than_l2": bool(n * 3 * L * 4 > 126e6),
                       "input_bytes_per_gpu": n * 3 * L * 4, "sharding": "contiguous pair blocks, no collective"},
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_kind": peak_kind,
                         "alg_bytes_per_launch": alg_bytes, "avg_launch_ms": avg_ms,
                         "launches": n_launch, "bytes_per_pair": KERNEL_U[dom] * U,
                         "kernel_time_shares": shares,
                         "traffic_source": "constant from profiles/traffic.json (one ncu --set full capture), not measured in this run",
                         "measured_in": "second pass of the same %d steps with CUDA events around every launch "
                                        "(%.1f ms vs %.1f ms for the timed, event-free pass)" % (args.steps, ms_profiled, ms),
                         "kernels": kernels},
            "path_roofline": {"bytes_per_pair": PATH_U * U, "achieved": path_achieved, "peak": peak,
                              "unit": "GB/s", "frac": path_achieved / peak, "per_gpu": True,
                              "accounting": "frac: SURVEY 8(d)'s 21*U schedule (the survey's accounting); frac_moved: the "
                                            "17*U this design moves; frac_dram: DRAM bytes per pair measured by ncu",
                              "bytes_moved_per_pair": MOVED_U * U,
                              "frac_moved": MOVED_U * U * pairs_s_gpu / 1e9 / peak,
                              "dram_bytes_per_pair_ncu": dram_pair,
                              "frac_dram": (dram_pair * pairs_s_gpu / 1e9 / peak) if dram_pair else None},
            "e2e": e2e, "e2e_variants": e2e_variants, "gpu_launches": launches, "clocks": clocks,
            "check": {"lag_mismatches": bad, "success_flags": ok_flags, "pairs_checked_per_rank": min(n, 256)},
        }
        if latency is not None:
            line["latency"] = latency
        if in_library is not None:
            line["in_library"] = in_library
        if world == 1 and not args.no_cpu_baseline:
            os.sched_setaffinity(0, all_cpus)      # the CPU leg gets every host core back
            line["cpu_baseline"] = cpu_baseline_sample(L, SEED)
        emit(line)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
