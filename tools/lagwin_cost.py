"""Cost of the lag window on one GPU: unwindowed and windowed calls alternated on the same pairs.

    python tools/lagwin_cost.py [--rounds 2] [--reps 5] [--out lagwin_cost.json]

Legs (audiosync_cuda_xcorr_batch_device, seeded F32 synth pairs): 4,096 pairs at 1,440,000 frames
(static plan), 512 pairs at 1,000,000 (runtime-radix plan) and 512 pairs at 48,000.  Windows, with
W = min(48,000, L / 10):
  full     [-L, L-1]: must be the unwindowed call (same kernels, same record bytes)
  around   [lag0 - W, lag0 + W] around the true lag of pair 0
  exclude  [-L, -L + 2W], below every synth lag (they lie in [-L/2, L/2]): the global peak is
           outside, the threshold's worst case
  phat     `around` under PHAT weighting, against unwindowed PHAT
Per leg, after a warm-up of every context, each window alternates with its unwindowed twin
`--rounds` times, each timed over `--reps` calls ending in a device synchronise; then one profiled
call of each gives the per-kernel device time per pair (profile API: CUDA events around every
launch).  Prints the card name, power limit and max SM clock of the same run and one JSON line per
leg and window.
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
    from oracle import xcorr_numpy as xn
    gpu = card()
    print("card:", gpu, flush=True)
    lines = []
    for L, n in LEGS:
        W = min(48000, L // 10)
        lag0 = xn.synth_true_lag(SEED, 0, L)
        windows = {"full": (-L, L - 1, False), "around": (lag0 - W, lag0 + W, False),
                   "exclude": (-L, -L + 2 * W, False), "phat": (lag0 - W, lag0 + W, True)}
        src = torch.empty(n * 2 * L, dtype=torch.float32, device="cuda:0")
        smp = torch.empty(n * L, dtype=torch.float32, device="cuda:0")
        res = {k: torch.empty(n * 64, dtype=torch.uint8, device="cuda:0") for k in ("base", "win")}
        for name, (lo, hi, phat) in windows.items():
            base, win = ac.Context([0]), ac.Context([0])
            for c in (base, win):
                c.set_weighting(ac.WEIGHT_PHAT if phat else ac.WEIGHT_NONE)
            win.set_lag_window(lo, hi)
            base.synth_pairs(0, SEED, 0, n, L, ac.F32, src.data_ptr(), smp.data_ptr())
            base.synchronize(0)
            ctxs = {"base": base, "win": win}

            def call(k):
                ctxs[k].xcorr_batch_device(0, src.data_ptr(), smp.data_ptr(), n, L, ac.F32, res[k].data_ptr())

            for k in ctxs:                               # warm-up: plans, modules, workspaces
                call(k)
                ctxs[k].synchronize(0)
            rates = {k: [] for k in ctxs}
            for _ in range(args.rounds):
                for k in ctxs:
                    t0 = time.perf_counter()
                    for _ in range(args.reps):
                        call(k)
                    ctxs[k].synchronize(0)
                    rates[k].append(n * args.reps / (time.perf_counter() - t0))
            kern = {}
            for k, c in ctxs.items():
                c.profile_reset()
                c.profile_enable(True)
                call(k)
                prof = c.profile_read()
                c.profile_enable(False)
                c.synchronize(0)
                kern[k] = {kk: round(ms * 1000.0 / n, 3) for kk, (cnt, ms) in prof.items() if cnt}
            same = bool(torch.equal(res["base"], res["win"]))
            ratio = sum(rates["win"]) / sum(rates["base"])
            line = dict(L=L, pairs=n, window=name, lags=[lo, hi], phat=phat, card=gpu,
                        plan=win.describe_plan(L), records_equal_unwindowed=same,
                        pairs_per_s={k: [round(r) for r in v] for k, v in rates.items()},
                        windowed_over_unwindowed=round(ratio, 4), us_per_pair=kern)
            print(json.dumps(line), flush=True)
            lines.append(line)
            for c in ctxs.values():
                c.close()
        del src, smp, res
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
