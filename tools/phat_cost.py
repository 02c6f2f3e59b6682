"""Cost of PHAT weighting on one GPU: NONE and PHAT alternated on the same device-resident pairs.

    python tools/phat_cost.py [--rounds 2] [--reps 5] [--out phat_cost.json]

Legs (audiosync_cuda_xcorr_batch_device, seeded F32 synth pairs, one context per weighting):
4,096 pairs at 1,440,000 frames (static plan), 512 pairs at 1,000,000 (runtime-radix plan) and 512
pairs at 48,000 (runtime-radix columns, static rows).  Per length, after a warm-up of both modes,
NONE and PHAT alternate `--rounds` times, each timed over `--reps` calls ending in a device
synchronise; then one profiled call of each gives the per-kernel device time per pair (profile API:
CUDA events around every launch).  Prints the card name, power limit and max SM clock of the same run
and one JSON line per leg.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "old-audiosync_b200"))

SEED = 0x5EED
LEGS = ((1440000, 4096), (1000000, 512), (48000, 512))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return q.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import audiosync_cuda as ac
    gpu = card()
    print("card:", gpu, flush=True)
    lines = []
    ctxs = {w: ac.Context([0]) for w in (ac.WEIGHT_NONE, ac.WEIGHT_PHAT)}
    ctxs[ac.WEIGHT_PHAT].set_weighting(ac.WEIGHT_PHAT)
    names = {ac.WEIGHT_NONE: "none", ac.WEIGHT_PHAT: "phat"}
    for L, n in LEGS:
        src = torch.empty(n * 2 * L, dtype=torch.float32, device="cuda:0")
        smp = torch.empty(n * L, dtype=torch.float32, device="cuda:0")
        res = torch.empty(n * 64, dtype=torch.uint8, device="cuda:0")
        ctxs[ac.WEIGHT_NONE].synth_pairs(0, SEED, 0, n, L, ac.F32, src.data_ptr(), smp.data_ptr())
        ctxs[ac.WEIGHT_NONE].synchronize(0)

        def call(w):
            ctxs[w].xcorr_batch_device(0, src.data_ptr(), smp.data_ptr(), n, L, ac.F32, res.data_ptr())

        for w in ctxs:                                   # warm-up: plans, modules, workspaces
            call(w)
            ctxs[w].synchronize(0)
        rates = {w: [] for w in ctxs}
        for _ in range(args.rounds):
            for w in ctxs:
                t0 = time.perf_counter()
                for _ in range(args.reps):
                    call(w)
                ctxs[w].synchronize(0)
                rates[w].append(n * args.reps / (time.perf_counter() - t0))
        kern = {}
        for w, c in ctxs.items():
            c.profile_reset()
            c.profile_enable(True)
            call(w)
            prof = c.profile_read()
            c.profile_enable(False)
            kern[names[w]] = {k: round(ms * 1000.0 / n, 3) for k, (cnt, ms) in prof.items() if cnt}
        line = dict(L=L, pairs=n, card=gpu, plan_none=ctxs[ac.WEIGHT_NONE].describe_plan(L),
                    plan_phat=ctxs[ac.WEIGHT_PHAT].describe_plan(L),
                    pairs_per_s={names[w]: [round(r) for r in v] for w, v in rates.items()},
                    us_per_pair=kern)
        print(json.dumps(line), flush=True)
        lines.append(line)
        del src, smp, res
        torch.cuda.empty_cache()
    for c in ctxs.values():
        c.close()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
