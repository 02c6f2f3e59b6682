"""Cost of the correlation export on one GPU: no export, a +-48,000-lag range and the full range,
alternated on the same device-resident pairs.

    python tools/corr_cost.py [--rounds 2] [--reps 3] [--out corr_cost.json]

Legs (seeded F32 synth pairs on the device): 4,096 pairs at 1,440,000 frames (static plan), 512 at
1,000,000 (runtime-radix plan), 512 at 48,000 and 512 at 24,000 in precise mode.  Per leg, after a
warm-up of every variant, the variants alternate `--rounds` times, each timed over `--reps` calls
ending in a device synchronise (whole path: transform, export, Pearson); the no-export variant is
audiosync_cuda_xcorr_batch_device, the others audiosync_cuda_xcorr_correlation_device into a device
array.  Then one profiled call of each gives the per-kernel device time per pair (profile API: CUDA
events around every launch) and the records of every variant are compared byte for byte.  Prints the
card name, power limit and max SM clock of the same run and one JSON line per leg and variant.
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
LEGS = ((1440000, 4096, False), (1000000, 512, False), (48000, 512, False), (24000, 512, True))


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
    for L, n, precise in LEGS:
        W48 = min(48000, L - 1)
        variants = {"none": None, "pm48000": (-W48, W48), "full": (-L, L - 1)}
        src = torch.empty(n * 2 * L, dtype=torch.float32, device="cuda:0")
        smp = torch.empty(n * L, dtype=torch.float32, device="cuda:0")
        res = {k: torch.empty(n * 64, dtype=torch.uint8, device="cuda:0") for k in variants}
        c = ac.Context([0])
        c.set_precise(precise)
        c.synth_pairs(0, SEED, 0, n, L, ac.F32, src.data_ptr(), smp.data_ptr())
        c.synchronize(0)
        # one export array, as large as the largest range needs (the full range at 1.44M: 94 GB for
        # 4,096 pairs) -- the calls are split into batches of `per` pairs whose rows fit in 8 GB
        per = max(1, min(n, (8 << 30) // (8 * 2 * L)))
        corr = torch.empty(per * 2 * L, dtype=torch.float64, device="cuda:0")

        def call(k):
            rng = variants[k]
            for p0 in range(0, n, per):
                m = min(per, n - p0)
                s = src.data_ptr() + p0 * 2 * L * 4
                q = smp.data_ptr() + p0 * L * 4
                r = res[k].data_ptr() + p0 * 64
                if rng is None:
                    c.xcorr_batch_device(0, s, q, m, L, ac.F32, r)
                else:
                    c.xcorr_correlation_device(0, s, q, m, L, ac.F32, rng[0], rng[1], r, corr.data_ptr())

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
        same = all(bool(torch.equal(res["none"], res[k])) for k in variants)
        base = sum(rates["none"])
        for k, rng in variants.items():
            line = dict(L=L, pairs=n, precise=precise, export=k, lags=list(rng) if rng else None, card=gpu,
                        plan=c.describe_plan(L), records_equal_no_export=same,
                        pairs_per_s=[round(r) for r in rates[k]],
                        over_no_export=round(sum(rates[k]) / base, 4), us_per_pair=kern[k])
            print(json.dumps(line), flush=True)
            lines.append(line)
        c.close()
        del src, smp, res, corr
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
