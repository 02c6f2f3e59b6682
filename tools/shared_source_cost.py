"""Cost of one source against many samples on one GPU: the batch call on the source replicated per pair
and the shared-source call, alternated on the same samples.

    python tools/shared_source_cost.py [--rounds 2] [--reps 3] [--out shared_source_cost.json]

Legs:
  device-resident F32 (xcorr_batch_device / xcorr_shared_source_device, seeded synth samples):
    4,096 pairs at 1,440,000 frames and 512 at 144,000 (static plans: the source is transformed once
    per call), 512 at 1,000,000 (runtime-radix plan: every pair reads the one source); and F64, 512
    pairs at 480,000 (the fp64 sample-only column kernel, at 60 registers against its sibling's 58);
  host-fed from page-locked memory (xcorr_batch_results / xcorr_shared_source, HOST) at 1,440,000
    frames: F32, S16 and F64 (the replicated F64 arm with host narrowing off, which the shared call
    equals by contract).
After a warm-up of both arms, each leg alternates replicated and shared `--rounds` times, each timed
over `--reps` calls ending in a device synchronise (whole-path pairs/s); then one profiled call of
each arm gives the per-kernel device time per pair (profile API: CUDA events around every launch).
Both arms' record bytes are compared.  Prints the card name, power limit and max SM clock of the same
run and one JSON line per leg.
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
sys.path.insert(0, ROOT)

SEED = 0x5EED
DEVICE_LEGS = (("f32", 1440000, 4096), ("f32", 144000, 512), ("f32", 1000000, 512), ("f64", 480000, 512))
HOST_LEGS = (("f32", 1440000, 128), ("s16", 1440000, 128), ("f64", 1440000, 64))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def alternate(calls, n, rounds, reps, sync):
    rates = {k: [] for k in calls}
    for k in calls:                                  # warm-up: plans, modules, workspaces
        calls[k]()
        sync()
    for _ in range(rounds):
        for k in calls:
            t0 = time.perf_counter()
            for _ in range(reps):
                calls[k]()
            sync()
            rates[k].append(n * reps / (time.perf_counter() - t0))
    return rates


def kernels(c, call, n):
    c.profile_reset()
    c.profile_enable(True)
    call()
    prof = c.profile_read()
    c.profile_enable(False)
    return {k: round(ms * 1000.0 / n, 3) for k, (cnt, ms) in prof.items() if cnt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import audiosync_cuda as ac
    gpu = card()
    print("card:", gpu, flush=True)
    lines = []

    def report(line):
        r = line["pairs_per_s"]
        line["shared_over_replicated"] = round(sum(r["shared"]) / sum(r["replicated"]), 4)
        line["pairs_per_s"] = {k: [round(x) for x in v] for k, v in r.items()}
        print(json.dumps(line), flush=True)
        lines.append(line)

    for dt, L, n in DEVICE_LEGS:
        c = ac.Context([0])
        tdt, code = (torch.float64, ac.F64) if dt == "f64" else (torch.float32, ac.F32)
        srcs = torch.empty(n, 2 * L, dtype=tdt, device="cuda:0")
        smp = torch.empty(n, L, dtype=tdt, device="cuda:0")
        c.synth_pairs(0, SEED, 0, n, L, code, srcs.data_ptr(), smp.data_ptr())
        c.synchronize(0)
        src = srcs[0].clone()
        srcs.copy_(src.expand(n, 2 * L))                  # the replicated arm's input
        res = {k: torch.empty(n * 64, dtype=torch.uint8, device="cuda:0") for k in ("replicated", "shared")}
        calls = {"replicated": lambda: c.xcorr_batch_device(0, srcs.data_ptr(), smp.data_ptr(), n, L, code,
                                                            res["replicated"].data_ptr()),
                 "shared": lambda: c.xcorr_shared_source_device(0, src.data_ptr(), smp.data_ptr(), n, L, code,
                                                                res["shared"].data_ptr())}
        rates = alternate(calls, n, args.rounds, args.reps, lambda: c.synchronize(0))
        kern = {k: kernels(c, f, n) for k, f in calls.items()}
        c.synchronize(0)
        report(dict(leg="device", dtype=dt, L=L, pairs=n, card=gpu, plan=c.describe_plan(L),
                    records_equal=bool(torch.equal(res["replicated"], res["shared"])), pairs_per_s=rates,
                    us_per_pair=kern))
        c.close()
        del srcs, smp, src, res
        torch.cuda.empty_cache()

    rng = np.random.default_rng(SEED)
    for dt, L, n in HOST_LEGS:
        c = ac.Context([0])
        c.set_host_narrowing(ac.NARROW_OFF)
        code = {"f32": ac.F32, "s16": ac.S16, "f64": ac.F64}[dt]
        src32 = rng.standard_normal(2 * L).astype(np.float32)
        smp32 = np.stack([src32[(97 * i) % L:(97 * i) % L + L] for i in range(n)])
        smp32 += 0.3 * rng.standard_normal(smp32.shape).astype(np.float32)
        if dt == "s16":
            conv = lambda a: np.clip(np.round(a * 6000), -32768, 32767).astype(np.int16)   # noqa: E731
        else:
            conv = lambda a: a.astype(np.float64 if dt == "f64" else np.float32)          # noqa: E731
        pinned = lambda a: torch.from_numpy(np.ascontiguousarray(a)).pin_memory()   # noqa: E731
        src = pinned(conv(src32))
        srcs = pinned(np.broadcast_to(conv(src32), (n, 2 * L)))
        smp = pinned(conv(smp32))
        out = {k: np.zeros(n, ac.RESULT_DTYPE) for k in ("replicated", "shared")}
        lib = ac.lib()

        def ok(rc):
            if rc != 0:
                raise RuntimeError(ac.last_error())
        calls = {"replicated": lambda: ok(lib.audiosync_cuda_xcorr_batch_results(c.handle, srcs.data_ptr(), smp.data_ptr(), n, L,
                                                                                 code, ac.HOST, out["replicated"].ctypes.data)),
                 "shared": lambda: ok(lib.audiosync_cuda_xcorr_shared_source(c.handle, src.data_ptr(), smp.data_ptr(), n, L,
                                                                             code, ac.HOST, out["shared"].ctypes.data))}
        rates = alternate(calls, n, args.rounds, args.reps, lambda: None)   # host calls return synchronised
        kern = {k: kernels(c, f, n) for k, f in calls.items()}
        report(dict(leg="host_pinned", dtype=dt, L=L, pairs=n, card=gpu, plan=c.describe_plan(L),
                    records_equal=out["replicated"].tobytes() == out["shared"].tobytes(), pairs_per_s=rates,
                    us_per_pair=kern))
        c.close()
        del src, srcs, smp
    if args.out:
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
