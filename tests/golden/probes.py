"""Closed-form PROBE inputs for the transform kernels -- TEST INFRASTRUCTURE.

The white-noise pairs of the parity suite see the correlation r only through one tall peak, so
one frequency bin (about 1/M of that peak) can be wrong without moving the record.  These probes
make every bin class and every output position observable and need no FFT to check:

with the sample one-hot at `a` (0 <= a < L), the reference's results[j] (j < 2L, FFTW's
unnormalised c2r, N = 2L) is exactly

    r[j] = N * source[(j + a) mod 2L]

for every plan, embedded ones included (those correlate the periodically extended source, and
a + j < 3L).  So the expected record is an O(N) fp64 computation on the probe's own fp32-rounded
values.  Families:

  A  bin probes: a spike of height 1 at source position p plus a tone A cos(2 pi k n / N + phi),
     A = 0.25, phi putting the tone at pi/2 at p -- a phase error d in bin k moves the peak by
     A d N, an amplitude error moves the second peak.  Bins are chosen from the plan's
     M1 x M2 split (bin k = k1 + M1 k2): DC, 1, M-1, Nyquist, M/2 +- 1, row 0, row M1/2, rows
     1 and M1/2-1 with their partners, both ends of a split-phase stripe, and seeded random bins.
  B  position probes: one spike whose output lands on 0, 1, L-1, L, L+1, 2L-1, both outputs of
     one packed point, the first and last column of a column tile, and (embedded plans) where
     it recurs at j + 2L inside the padded transform.
  C  second-peak placement: spikes h > g > f (g - f = 1e-3 g) with g in the same thread, warp,
     CTA as h, in an earlier or later column tile, or at r[0].
  D  signed seed: r[0] < 0 with |r[0]| above the true answer (ratios 0.5, 0.99, 1.01), a
     negative r[0] whose neighbours r[+-1] are nearly as large, and a positive r[0] that ties.

Every array is built in fp64 from a few integers, rounded once to fp32, and the expectation is
computed from the rounded values, so the same probes are rebuilt bit for bit anywhere.
"""
from __future__ import annotations

import os
import re
import sys
from dataclasses import dataclass, field

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
from oracle import xcorr_numpy as xn  # noqa: E402

TONE_A = 0.25

# Bound on |kernel - closed form| of peak and second, relative to N * sum(|spike|) (+ A for a
# tone).  The fp32 kernels land within ~3e-7 of it on every bin class; a bin that is not split,
# multiplied or merged at all shows up at ~0.15.
TOL_F32 = 2e-6
TOL_F64 = 1e-9


@dataclass(frozen=True)
class Plan:
    """Four-step split of the packed length M = M1 * M2 (M = L unless embedded)."""
    L: int
    M: int
    M1: int
    M2: int
    row: tuple            # row radices, DIF pass order
    ct: int = 16          # columns per inverse-column tile
    embedded: bool = False


# fft_plan.h: the static plans of the interval schedule
STATIC_PLANS = {
    144000: Plan(144000, 144000, 300, 480, (4, 8, 15)),
    288000: Plan(288000, 288000, 300, 960, (4, 16, 15)),
    480000: Plan(480000, 480000, 400, 1200, (5, 16, 15)),
    720000: Plan(720000, 720000, 600, 1200, (5, 16, 15)),
    960000: Plan(960000, 960000, 400, 2400, (10, 16, 15)),
    1440000: Plan(1440000, 1440000, 600, 2400, (10, 16, 15)),
}


def parse_plan(L: int, desc: str) -> Plan:
    """Plan of a runtime-radix description ("fft L=.. M=.. M1=.. M2=.. col=.. row=.. tile=..")."""
    m = re.search(r"M=(\d+) M1=(\d+) M2=(\d+) col=[0-9x]+ row=([0-9x]+) (?:padded|plain) tile=(\d+)", desc)
    assert m, desc
    M, M1, M2 = int(m.group(1)), int(m.group(2)), int(m.group(3))
    row = tuple(int(x) for x in m.group(4).split("x"))
    return Plan(L, M, M1, M2, row, int(m.group(5)), "embedded" in desc)


def single_cta_plan(L: int) -> Plan:
    """The single-CTA kernel (fft_small.cuh): one 'row' of M = L points, 256 threads."""
    return Plan(L, L, 1, L, (L,), ct=1)


def row_freq_of_pos(plan: Plan, e: int) -> int:
    """Bin held at position e of a row after the forward DIF passes (RadixList::freq_of_pos)."""
    k, stride, weight = 0, plan.M2, 1
    for r in plan.row:
        stride //= r
        d = e // stride
        e -= d * stride
        k += d * weight
        weight *= r
    return k


@dataclass
class Probe:
    """source = sum of spikes (output position j, height h) + optional tone; sample = one-hot at a."""
    name: str
    L: int
    a: int
    spikes: list = field(default_factory=list)    # [(j, h)] -> source[(j + a) mod 2L] += h
    tone_k: int = -1                              # real bin of the tone (-1: none)
    tone_p: int = 0                               # source position where the tone is at pi/2

    def build(self, dtype=np.float32):
        L, N = self.L, 2 * self.L
        src = np.zeros(N, np.float64)
        if self.tone_k >= 0:
            k = self.tone_k
            # DC and Nyquist have no phase: a plain constant / alternating tone there
            phi = 0.0 if k in (0, L) else np.pi / 2 - 2 * np.pi * ((k * self.tone_p) % N) / N
            src += TONE_A * np.cos(2 * np.pi * ((k * np.arange(N, dtype=np.int64)) % N) / N + phi)
        for j, h in self.spikes:
            src[(j + self.a) % N] += h
        smp = np.zeros(L, np.float64)
        smp[self.a] = 1.0
        return src.astype(np.float32).astype(dtype), smp.astype(dtype)

    def scale(self) -> float:
        """N * sum |spike| (+ A): the size the kernel's rounding errors are relative to."""
        return 2.0 * self.L * (sum(abs(h) for _, h in self.spikes) + (TONE_A if self.tone_k >= 0 else 0.0))

    def expect(self, idx=None, arrays=None, tol=TOL_F32):
        """The record the reference computes for this probe, in closed form (see module doc).
        `tied`: every index whose |r| is within tol * scale() of the peak's, above or below -- a tie
        no transform of that precision can resolve; `idx` evaluates the record at one of them
        instead of the argmax.  A larger |r| that the argmax rule passes over (a negative r[0])
        is no tie."""
        src, smp = self.build(np.float64) if arrays is None else (np.asarray(a, np.float64) for a in arrays)
        N = 2 * self.L
        r = N * np.roll(src, -self.a)
        best = xn.max_abs_index(r)
        mag = np.abs(r)
        tied = [int(i) for i in np.flatnonzero(np.abs(mag - mag[best]) <= tol * self.scale())]
        idx = best if idx is None else idx
        mag[idx] = -1.0
        second = float(np.nanmax(mag))
        peak = float(r[idx])
        lag, wx, wy = xn.windows(src, smp, idx)
        coef = xn.pearson(wx, wy)
        out = dict(raw_index=idx, peak=peak, second=second, lag=int(lag), coef=coef,
                   ret=-1 if coef != coef else 0, tied=tied)
        out.update(xn.peak_quality(src, smp, idx, peak, second))
        return out


def _a(rng, L, near=False):
    """Sample position: seeded; `near`: small, so that j + a stays below L (no wrap of the source)."""
    if near:
        return int(rng.integers(0, min(L, 97)))
    return int(rng.integers(0, L))


def bin_probes(plan: Plan, seed: int, n_random: int = 16, dense: bool = True):
    """Family A.  `dense`: every class with several members; otherwise one bin per class."""
    L, M, M1, M2 = plan.L, plan.M, plan.M1, plan.M2
    rng = np.random.default_rng(seed)
    bins = {"dc": 0, "1": 1, "M-1": M - 1, "nyquist": M, "M/2-1": M // 2 - 1, "M/2": M // 2, "M/2+1": M // 2 + 1}
    if M1 > 1:
        k2s = [1, M2 // 2 - 1, M2 // 2, M2 // 2 + 1, M2 - 1] if dense else [M2 // 2]
        for k2 in k2s:
            bins["row0-k2=%d" % k2] = M1 * k2
        if M1 % 2 == 0:
            for k2 in ([0, 1, M2 // 2, M2 - 1] if dense else [1]):
                bins["row%d-k2=%d" % (M1 // 2, k2)] = M1 // 2 + M1 * k2
        rows = [1, M1 - 1, M1 // 2 - 1, M1 - (M1 // 2 - 1)] if dense else [1, M1 // 2 - 1]
        for k1 in sorted(set(r for r in rows if 0 < r < M1 and 2 * r != M1)):
            for k2 in ([0, M2 // 3, M2 - 1] if dense else [M2 // 3]):
                bins["row%d-k2=%d" % (k1, k2)] = k1 + M1 * k2
        # split phase of the two-row branch: position e = d0 * S0 + e1 of row k1a pairs with M2-1-e
        # of row M1-k1a; stripes e1 = 0 .. S0-1 of the first and last d0
        S0 = M2 // plan.row[0]
        k1a = 2 if M1 > 4 else 1
        for e in ([0, S0 - 1, (plan.row[0] - 1) * S0, M2 - 1] if dense else [S0 - 1]):
            bins["stripe-e=%d" % e] = k1a + M1 * row_freq_of_pos(plan, e)
            bins["stripe-partner-e=%d" % e] = (M1 - k1a) + M1 * row_freq_of_pos(plan, M2 - 1 - e)
    for i in range(n_random):
        bins["rand%d" % i] = int(rng.integers(0, M + 1))
    out = []
    for name, k in bins.items():
        if plan.M != plan.L:
            k = k % (L + 1)               # embedded: a bin of the padded transform is no bin of N = 2L
        p = int(rng.integers(0, 2 * L))
        a = _a(rng, L)
        out.append(Probe("A:%s(k=%d)" % (name, k), L, a, [((p - a) % (2 * L), 1.0)], tone_k=k, tone_p=p))
    return out


def _packed_j(plan: Plan, n1: int, n2: int, odd: int) -> int:
    return 2 * (n1 * plan.M2 + n2) + odd


def position_probes(plan: Plan, seed: int):
    """Family B: one spike, output position j; alternating sign."""
    L = plan.L
    rng = np.random.default_rng(seed)
    js = {"0": 0, "1": 1, "L-1": L - 1, "L": L, "L+1": L + 1, "2L-1": 2 * L - 1}
    q = int(rng.integers(1, L - 1))
    js["even"], js["odd"] = 2 * q, 2 * q + 1
    if plan.M1 > 1:
        ntiles = (plan.M2 + plan.ct - 1) // plan.ct
        for t in (0, 1, ntiles - 1):
            n1 = int(rng.integers(0, plan.M1))
            for c, tag in ((0, "first"), (plan.ct - 1, "last")):
                n2 = min(t * plan.ct + c, plan.M2 - 1)
                for odd in (0, 1):
                    j = _packed_j(plan, n1, n2, odd)
                    if j < 2 * L:
                        js["tile%d-%s-col%s" % (t, tag, "-odd" if odd else "")] = j
    out = []
    for i, (name, j) in enumerate(js.items()):
        h = 1.0 if i % 2 == 0 or j == 0 else -1.0
        out.append(Probe("B:%s(j=%d)" % (name, j), L, _a(rng, L), [(j, h)]))
    # the spike recurs at j + 2L inside an embedded transform when j + a stays below L
    for j in (1, 2, L - 200):
        out.append(Probe("B:recur(j=%d)" % j, L, _a(rng, L, near=True), [(j, -0.5)]))
    return out


def second_probes(plan: Plan, seed: int):
    """Family C: peak h = 1, second g = 0.75, third f = g (1 - 1e-3); g placed relative to h."""
    L = plan.L
    rng = np.random.default_rng(seed)
    h, g, f = 1.0, 0.75, 0.75 * (1 - 1e-3)
    M1, M2, ct = plan.M1, plan.M2, plan.ct
    ntiles = (M2 + ct - 1) // ct

    def at(n1, n2, odd):
        return _packed_j(plan, n1 % M1, n2 % M2, odd)

    out = []
    for rep in range(2):
        n1 = int(rng.integers(1, max(2, M1 - 1)))
        t = int(rng.integers(1, max(2, ntiles - 1)))
        n2 = min(t * ct + int(rng.integers(0, max(1, ct - 1))), M2 - 2)
        jh = at(n1, n2, 0)
        places = {
            "same-thread": jh + 1,
            "same-warp": at(n1, n2 + 1, rep),
            "same-cta": at(n1 + M1 // 2, n2, 1 - rep),
            "earlier-cta": at(n1, n2 - ct, rep) if n2 >= ct else at(n1, 0, 1),
            "later-cta": at(n1, min(n2 + ct, M2 - 1), rep),
            "r0": 0,
        }
        for name, jg in places.items():
            if jg >= 2 * L or jg == jh:
                continue
            jf = at(int(rng.integers(0, M1)), int(rng.integers(0, M2)), rep)
            while jf in (jh, jg) or jf >= 2 * L:
                jf = (jf + 7) % (2 * L)
            sg = -1.0 if rep else 1.0
            out.append(Probe("C:%s-%d(jh=%d,jg=%d)" % (name, rep, jh, jg), L, _a(rng, L),
                             [(jh, h if rep == 0 else -h), (jg, g * sg), (jf, f)]))
    return out


def seed_probes(plan: Plan, seed: int):
    """Family D: r[0] = -1 against a true answer of 0.5 / 0.99 / 1.01 in various places."""
    L = plan.L
    rng = np.random.default_rng(seed)
    M1, M2, ct = plan.M1, plan.M2, plan.ct
    places = {"same-thread": 1, "2L-1": 2 * L - 1, "mid": (L + 5001) % (2 * L) or 1}
    if M1 > 1:
        places["same-warp"] = _packed_j(plan, 0, 1, 0)
        places["same-cta"] = _packed_j(plan, M1 // 2, ct // 2, 1)
        places["later-cta"] = _packed_j(plan, int(rng.integers(0, M1)), M2 - 1, 0)
    else:   # single CTA: the seed thread's own later items (n = 0 mod 256)
        places["seed-thread"] = 2 * 256 * ((L // 2 - 1) // 256)
    out = []
    for name, j in places.items():
        j = min(j, 2 * L - 1)
        for ratio in (0.5, 0.99, 1.01):
            noise = [(int(rng.integers(2, 2 * L - 1)), 0.01 * (i + 1)) for i in range(3)]
            spikes = [(0, -1.0), (j, ratio * (-1.0 if ratio > 1 else 1.0))]
            spikes += [s for s in noise if s[0] not in (0, j)]
            out.append(Probe("D:neg-seed-%s-%.2f(j=%d)" % (name, ratio, j), L, _a(rng, L), spikes))
    # inverted low-passed audio: r[0] < 0 with r[1], r[-1] nearly as large
    out.append(Probe("D:neg-shoulders-left", L, _a(rng, L), [(0, -1.0), (1, -0.97), (2 * L - 1, -0.98)]))
    out.append(Probe("D:neg-shoulders-right", L, _a(rng, L), [(0, -1.0), (1, -0.98), (2 * L - 1, -0.97), (2, -0.9)]))
    # a positive r[0] keeps index 0 on a tie (strict '>'); the tied entry is the second peak
    out.append(Probe("D:pos-seed-tie", L, _a(rng, L), [(0, 1.0), (2 * L - 1, -1.0), (L // 2, 0.5)]))
    return out


def all_probes(plan: Plan, seed: int, dense: bool = True):
    return (bin_probes(plan, seed, 16 if dense else 4, dense) + position_probes(plan, seed + 1)
            + second_probes(plan, seed + 2) + seed_probes(plan, seed + 3))


def resolve_tie(probe: Probe, exp: dict, raw_index: int, tol: float = TOL_F32) -> dict:
    """The expected record at `raw_index` when it is tied with the peak within the rounding floor
    (an exact tie no transform can resolve: either index is right), else `exp`.  `exp` and `tol`
    must come from the same expect(tol=...)."""
    if raw_index != exp["raw_index"] and raw_index in exp["tied"]:
        return probe.expect(raw_index, tol=tol)
    return exp


def check(probe: Probe, exp: dict, raw_index: int, peak: float, second: float, tol: float = TOL_F32):
    """'' if (raw_index, peak, second) match the closed form, else a one-line description."""
    bound = tol * probe.scale()
    errs = []
    if raw_index != exp["raw_index"]:
        errs.append("raw_index %d != %d" % (raw_index, exp["raw_index"]))
    if not abs(peak - exp["peak"]) <= bound:
        errs.append("peak %.9g vs %.9g (err %.2e of scale)" % (peak, exp["peak"], abs(peak - exp["peak"]) / probe.scale()))
    if not abs(second - exp["second"]) <= bound:
        errs.append("second %.9g vs %.9g (err %.2e of scale)" % (second, exp["second"],
                                                                abs(second - exp["second"]) / probe.scale()))
    return "" if not errs else "%s L=%d a=%d: %s" % (probe.name, probe.L, probe.a, "; ".join(errs))


def error_of(probe: Probe, exp: dict, peak: float, second: float) -> float:
    """max(|peak error|, |second error|) / scale."""
    return max(abs(peak - exp["peak"]), abs(second - exp["second"])) / probe.scale()
