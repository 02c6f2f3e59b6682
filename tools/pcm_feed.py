"""16-bit PCM (S16) against F32 / F64 at L = 1,440,000 on one GPU: host-fed and device-resident rates.

    python tools/pcm_feed.py [--host-pairs 96] [--host-seconds 3] [--rounds 2] [--device-pairs 4096]

Host-fed legs (audiosync_cuda_xcorr_batch_results, HOST memspace, page-locked inputs): S16, F32,
F64 with LOSSLESS host narrowing and F64 with narrowing OFF, alternated, each run `--rounds` times
for at least `--host-seconds` by calling the batch of `--host-pairs` pairs over and over.  All four
hold the same audio: int16 samples s, and s / 32768 as floats and doubles.

Device-resident legs (audiosync_cuda_xcorr_batch_device): `--device-pairs` seeded F32 synth pairs and
their 16-bit quantisation round(x * 32767) (clipped), alternated after a warm-up; then one profiled
run of each for the per-kernel times.

Every S16 record (host-fed and device-resident) is compared byte for byte with the F64 record of
the widened values s / 32768; the mismatch count is reported.  Prints the card name, power limit
and max SM clock of the same run and one JSON line.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "old-audiosync_b200"))

L = 1440000
SEED = 0x5EED


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def host_inputs(torch, n, rng):
    """Page-locked int16 / float32 / float64 copies of n pairs: sample = source from a random lag plus noise."""
    s16 = torch.empty((n, 2 * L), dtype=torch.int16).pin_memory()
    m16 = torch.empty((n, L), dtype=torch.int16).pin_memory()
    for i in range(n):
        src = np.clip(np.round(rng.normal(0, 6000, 2 * L)), -32768, 32767)
        lag = int(rng.integers(0, L))
        s16[i] = torch.from_numpy(src.astype(np.int16))
        m16[i] = torch.from_numpy(np.clip(src[lag:lag + L] + np.round(rng.normal(0, 1500, L)), -32768, 32767).astype(np.int16))
    f32 = [(x.to(torch.float32) / 32768.0).pin_memory() for x in (s16, m16)]
    f64 = [(x.to(torch.float64) / 32768.0).pin_memory() for x in (s16, m16)]
    return (s16, m16), f32, f64


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--host-pairs", type=int, default=96)
    ap.add_argument("--host-seconds", type=float, default=3.0)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--device-pairs", type=int, default=4096)
    ap.add_argument("--device-reps", type=int, default=5)
    args = ap.parse_args()

    import torch
    import audiosync_cuda as ac
    if not torch.cuda.is_available():
        raise SystemExit("pcm_feed.py measures on a CUDA device; none is visible")
    info = card()
    print("card:", info, flush=True)
    out = {"L": L, "card": info}
    mismatches = 0

    def same(a, b):
        return sum(int(a[i].tobytes() != b[i].tobytes()) for i in range(len(a)))

    # ---------------------------------------------------------------- host-fed
    n = args.host_pairs
    (s16, m16), f32, f64 = host_inputs(torch, n, np.random.default_rng(SEED))
    legs = {
        "s16": (s16, m16, ac.S16, ac.NARROW_LOSSLESS),
        "f32": (f32[0], f32[1], ac.F32, ac.NARROW_LOSSLESS),
        "f64_lossless": (f64[0], f64[1], ac.F64, ac.NARROW_LOSSLESS),
        "f64_off": (f64[0], f64[1], ac.F64, ac.NARROW_OFF),
    }
    host = {k: [] for k in legs}
    recs = {}
    with ac.Context([0]) as ctx:
        for k, (s, m, dt, mode) in legs.items():     # warm-up: plans, staging buffers, copy threads
            ctx.set_host_narrowing(mode)
            recs[k] = ctx.xcorr_batch_records(s.data_ptr(), m.data_ptr(), n, L, dt, ac.HOST)
        for _ in range(args.rounds):
            for k, (s, m, dt, mode) in legs.items():
                ctx.set_host_narrowing(mode)
                ctx.host_feed_stats(reset=True)
                calls, t0 = 0, time.perf_counter()
                while True:
                    r = ctx.xcorr_batch_records(s.data_ptr(), m.data_ptr(), n, L, dt, ac.HOST)
                    calls += 1
                    dt_s = time.perf_counter() - t0
                    if dt_s >= args.host_seconds:
                        break
                host[k].append(round(calls * n / dt_s, 1))
                if k == "s16":
                    mismatches += same(r, recs["f64_off"])
                if k == "f64_lossless":
                    out["f64_lossless_feed"] = ctx.host_feed_stats()
                print("host %-13s %8.1f pairs/s  (%d calls of %d pairs, %.2f s)" % (k, host[k][-1], calls, n, dt_s), flush=True)
        mismatches += same(recs["s16"], recs["f64_off"]) + same(recs["f64_lossless"], recs["f64_off"])
    out["host_pairs_per_s"] = host
    out["host_batch_pairs"] = n
    del s16, m16, f32, f64, legs

    # ---------------------------------------------------------- device-resident
    nd = args.device_pairs
    dev = torch.device("cuda", 0)
    src = torch.empty((nd, 2 * L), dtype=torch.float32, device=dev)
    smp = torch.empty((nd, L), dtype=torch.float32, device=dev)
    res = torch.empty(nd * ac.RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
    stream = torch.cuda.Stream(dev)                   # torch work and the library's kernels in one stream order
    with ac.Context([0]) as ctx, torch.cuda.stream(stream):
        st = stream.cuda_stream
        ctx.synth_pairs(0, SEED, 0, nd, L, ac.F32, src.data_ptr(), smp.data_ptr(), st)
        q_src = torch.empty((nd, 2 * L), dtype=torch.int16, device=dev)
        q_smp = torch.empty((nd, L), dtype=torch.int16, device=dev)
        for p0 in range(0, nd, 256):                  # in slices: the fp32 temporaries of the whole batch would not fit
            for x, y in ((src, q_src), (smp, q_smp)):
                y[p0:p0 + 256] = torch.clamp(torch.round(x[p0:p0 + 256] * 32767), -32768, 32767).to(torch.int16)
        arms = {"f32": (src, smp, ac.F32), "s16": (q_src, q_smp, ac.S16)}

        def run(k):
            s, m, dt = arms[k]
            ctx.xcorr_batch_device(0, s.data_ptr(), m.data_ptr(), nd, L, dt, res.data_ptr(), st)

        for k in arms:
            run(k)
        stream.synchronize()
        dev_rate = {k: [] for k in arms}
        for _ in range(args.device_reps):
            for k in arms:
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                stream.synchronize()
                e0.record(stream)
                run(k)
                e1.record(stream)
                e1.synchronize()
                dev_rate[k].append(round(nd / (e0.elapsed_time(e1) / 1e3), 1))
        print("device pairs/s:", dev_rate, flush=True)
        kern = {}
        for k in arms:
            ctx.profile_enable(True)
            ctx.profile_reset()
            run(k)
            prof = ctx.profile_read()
            ctx.profile_enable(False)
            kern[k] = {name: round(ms * 1e3 / nd, 3) for name, (cnt, ms) in prof.items() if cnt}
        print("device us/pair by kernel:", kern, flush=True)
        # S16 records of the timed pairs against F64 on the widened values, in slices that fit beside the inputs
        run("s16")
        stream.synchronize()
        got = res.cpu().numpy().view(ac.RESULT_DTYPE).copy()
        del src, smp, arms
        torch.cuda.empty_cache()
        step = 256
        ref_res = torch.empty(step * ac.RESULT_DTYPE.itemsize, dtype=torch.uint8, device=dev)
        for p0 in range(0, nd, step):
            c = min(step, nd - p0)
            ws, wm = q_src[p0:p0 + c].double() / 32768.0, q_smp[p0:p0 + c].double() / 32768.0
            ctx.xcorr_batch_device(0, ws.data_ptr(), wm.data_ptr(), c, L, ac.F64, ref_res.data_ptr(), st)
            stream.synchronize()
            mismatches += same(got[p0:p0 + c], ref_res[: c * ac.RESULT_DTYPE.itemsize].cpu().numpy().view(ac.RESULT_DTYPE))
    out["device_pairs"] = nd
    out["device_pairs_per_s"] = dev_rate
    out["device_us_per_pair"] = kern
    out["mismatches_vs_f64"] = mismatches
    out["card_after"] = card()
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
