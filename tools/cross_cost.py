"""Cost of many sources against many samples on one GPU: the batch call on every (source, sample) pair,
one shared-source call per source, and one cross call, alternated on the same seeded samples.

    python tools/cross_cost.py [--rounds 2] [--reps 3] [--out profiles/cross_cost.json]

Legs, device-resident F32, S = 8 sources against P = 512 samples (4,096 combinations):
  1,440,000 and 144,000 frames (static plans: the cross call transforms each source and each sample
  once), 1,000,000 frames (runtime-radix plan: the cross call runs the shared-source call per source,
  so no gain is expected).
After a warm-up of every arm, each leg alternates the three arms `--rounds` times, each timed over `--reps`
calls ending in a device synchronise (whole-path pairs/s); then one profiled call of each arm gives the
per-kernel device time per pair (profile API: CUDA events around every launch).  The record bytes of the
three arms are compared.  Prints the card name, power limit and max SM clock of the same run and one JSON
line per leg.
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
LEGS = ((1440000, 8, 512), (144000, 8, 512), (1000000, 8, 512))


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
    for L, S, P in LEGS:
        n = S * P
        c = ac.Context([0])
        # seeded synth pairs: sources from the first S pairs, samples from the first P
        srcs = torch.empty(P, 2 * L, dtype=torch.float32, device="cuda:0")
        smp = torch.empty(P, L, dtype=torch.float32, device="cuda:0")
        c.synth_pairs(0, SEED, 0, P, L, ac.F32, srcs.data_ptr(), smp.data_ptr())
        c.synchronize(0)
        src = srcs[:S].clone()
        del srcs
        rep_src = src.repeat_interleave(P, dim=0)         # pair s * P + p = (source s, sample p)
        rep_smp = smp.repeat(S, 1)
        res = {k: torch.empty(n * 64, dtype=torch.uint8, device="cuda:0") for k in ("replicated", "shared", "cross")}

        def shared():
            for s in range(S):
                c.xcorr_shared_source_device(0, src[s].data_ptr(), smp.data_ptr(), P, L, ac.F32,
                                             res["shared"].data_ptr() + s * P * 64)
        calls = {"replicated": lambda: c.xcorr_batch_device(0, rep_src.data_ptr(), rep_smp.data_ptr(), n, L, ac.F32,
                                                            res["replicated"].data_ptr()),
                 "shared": shared,
                 "cross": lambda: c.xcorr_cross_device(0, src.data_ptr(), S, smp.data_ptr(), P, L, ac.F32,
                                                       res["cross"].data_ptr())}
        rates = alternate(calls, n, args.rounds, args.reps, lambda: c.synchronize(0))
        kern = {k: kernels(c, f, n) for k, f in calls.items()}
        c.synchronize(0)
        line = dict(leg="device", dtype="f32", L=L, sources=S, samples=P, pairs=n, card=gpu, plan=c.describe_plan(L),
                    records_equal={"cross_vs_shared": bool(torch.equal(res["cross"], res["shared"])),
                                   "cross_vs_replicated": bool(torch.equal(res["cross"], res["replicated"]))},
                    pairs_per_s={k: [round(x) for x in v] for k, v in rates.items()},
                    cross_over_shared=round(sum(rates["cross"]) / sum(rates["shared"]), 4),
                    cross_over_replicated=round(sum(rates["cross"]) / sum(rates["replicated"]), 4),
                    us_per_pair=kern)
        print(json.dumps(line), flush=True)
        lines.append(line)
        c.close()
        del src, smp, rep_src, rep_smp, res
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
