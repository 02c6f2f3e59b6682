"""Cost of the runner-up records on one GPU: the batch call and the runner-up call alternated on the
same device-resident pairs.

    python tools/runner_up_cost.py [--rounds 2] [--reps 3] [--out profiles/runner_up_cost.json]

Legs (seeded F32 synth pairs on the device): 4,096 pairs at 1,440,000 frames (static plan), 512 at
1,000,000 (runtime-radix plan) and 512 at 48,000.  Per leg, after a warm-up of both variants, they
alternate `--rounds` times, each timed over `--reps` calls ending in a device synchronise (whole path);
the batch variant is audiosync_cuda_xcorr_batch_device, the other audiosync_cuda_xcorr_runner_up_device
at min_separation 48.  Then one profiled call of each gives the per-kernel device time per pair (profile
API: CUDA events around every launch), and the runner-up call's records are compared byte for byte with
the batch call's.  Prints the card name, power limit and max SM clock of the same run and one JSON line
per leg and variant.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "old-audiosync_b200"))
sys.path.insert(0, ROOT)

SEED = 0x5EED
LEGS = ((1440000, 4096), (1000000, 512), (48000, 512))
D = 48


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


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
    for L, n in LEGS:
        variants = ("batch", "runner_up")
        src = torch.empty(n * 2 * L, dtype=torch.float32, device="cuda:0")
        smp = torch.empty(n * L, dtype=torch.float32, device="cuda:0")
        res = {k: torch.empty(n * 64, dtype=torch.uint8, device="cuda:0") for k in variants}
        ru = torch.empty(n * 64, dtype=torch.uint8, device="cuda:0")
        c = ac.Context([0])
        c.synth_pairs(0, SEED, 0, n, L, ac.F32, src.data_ptr(), smp.data_ptr())
        c.synchronize(0)

        def call(k):
            if k == "batch":
                c.xcorr_batch_device(0, src.data_ptr(), smp.data_ptr(), n, L, ac.F32, res[k].data_ptr())
            else:
                c.xcorr_runner_up_device(0, src.data_ptr(), smp.data_ptr(), n, L, ac.F32, D, res[k].data_ptr(),
                                         ru.data_ptr())

        for k in variants:                               # warm-up: plans, modules, workspaces
            call(k)
            c.synchronize(0)
        rates = {k: [] for k in variants}
        for _ in range(args.rounds):
            for k in variants:
                t0 = time.perf_counter()
                for _ in range(args.reps):
                    call(k)
                c.synchronize(0)
                rates[k].append(n * args.reps / (time.perf_counter() - t0))
        kern = {}
        for k in variants:
            c.profile_reset()
            c.profile_enable(True)
            call(k)
            prof = c.profile_read()
            c.profile_enable(False)
            c.synchronize(0)
            kern[k] = {kk: round(ms * 1000.0 / n, 3) for kk, (cnt, ms) in prof.items() if cnt}
        same = bool(torch.equal(res["batch"], res["runner_up"]))
        base = sum(rates["batch"])
        for k in variants:
            line = dict(L=L, pairs=n, call=k, min_separation=D if k == "runner_up" else None, card=gpu,
                        plan=c.describe_plan(L), records_equal_batch=same,
                        pairs_per_s=[round(r) for r in rates[k]],
                        over_batch=round(sum(rates[k]) / base, 4), us_per_pair=kern[k])
            print(json.dumps(line), flush=True)
            lines.append(line)
        c.close()
        del src, smp, res, ru
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
