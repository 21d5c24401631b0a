"""Gap-affine 2-piece throughput: reads with one long indel each, end to end through wfagpu_align_affine2p with CIGAR,
the single-piece (4, 4, 2) rate on the same pairs for context, and a parity sample against the exact 2-piece DP.
Prints one JSON line with the card's name and power limit.

  workload a: 8192 x 10 kbp pairs, 5 % error plus one 100 .. 500 bp insertion or deletion, (4, 4, 2, 24, 1)
  workload b: 100000 x 1 kbp pairs, the same errors and penalties

usage: affine2p_probe.py [--reps N] [--sample N] [--small]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "wfa-gpu_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import wfagpu  # noqa: E402
from affine2p_ref import cost_ok, gotoh2p  # noqa: E402

BASES = np.frombuffer(b"ACGT", np.uint8)
PEN = (4, 4, 2, 24, 1)


def indel_reads(seed, n, length, err, lo=100, hi=500):
    """Pattern = text with err / 3 substitutions, deletions and insertions each, plus one insertion or deletion of
    lo .. hi bases (alternating) at a random position."""
    rng = np.random.default_rng(seed)
    pairs = []
    for i in range(n):
        text = BASES[rng.integers(0, 4, length)]
        r = rng.random(length)
        read = text.copy()
        sub = r < err / 3
        read[sub] = BASES[rng.integers(0, 4, int(sub.sum()))]
        keep = ~((r >= err / 3) & (r < 2 * err / 3))
        ins = (r >= 2 * err / 3) & (r < err)
        reps = keep.astype(np.int64) + ins
        out = np.repeat(read, reps)
        ends = np.cumsum(reps) - 1
        out[ends[ins]] = BASES[rng.integers(0, 4, int(ins.sum()))]
        L = int(rng.integers(lo, hi + 1))
        at = int(rng.integers(0, max(1, len(out) - L)))
        if i % 2 == 0:
            out = np.concatenate([out[:at], BASES[rng.integers(0, 4, L)], out[at:]])
        else:
            out = np.concatenate([out[:at], out[at + L:]])
        pairs.append((out.tobytes().decode(), text.tobytes().decode()))
    return pairs


def timed(pairs, pen, reps):
    """pen: five values (2-piece) or three (single piece).  -> aligner, pairs per second (median of reps calls)."""
    a = wfagpu.Aligner()
    for p, t in pairs:
        a.add_sequences(p, t)
    a.initialize_parameters(*pen[:3])
    a.options.compute_cigar = True
    a.options.max_error = 3000
    times = []
    for r in range(reps + 1):                   # the first call warms up the device and the provisioning
        a.reset_results()
        t0 = time.perf_counter()
        a.align(affine2p=pen if len(pen) == 5 else None)
        dt = time.perf_counter() - t0
        if r:
            times.append(dt)
    assert a.run_stats()["failed_pairs"] == 0
    return a, len(pairs) / statistics.median(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sample", type=int, default=8)
    ap.add_argument("--small", action="store_true", help="tiny sizes (a dry run of the script)")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    card = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"
    out = {"card": card, "penalties": list(PEN)}
    lib = wfagpu.load()
    for name, n, length in (("a_10kbp", 8192, 10000), ("b_1kbp", 100000, 1000)):
        if args.small:
            n, length = 64, min(length, 1000)
        pairs = indel_reads(0xA2F0 + length, n, length, 0.05)
        a, rate2 = timed(pairs, PEN, args.reps)
        mean2 = float(np.mean(a.errors()))
        rng = np.random.default_rng(7)
        idx = rng.choice(n, size=min(args.sample, n), replace=False)
        bad = 0
        for i in idx:
            p, t = pairs[i]
            s = gotoh2p(p, t, *PEN)
            bad += a.error(int(i)) != s or not cost_ok(lib, p, t, PEN, s, a.cigar(int(i)))
        del a
        a1, rate1 = timed(pairs, PEN[:3], args.reps)
        mean1 = float(np.mean(a1.errors()))
        del a1
        out[name] = {"pairs": n, "affine2p_aln_per_s": round(rate2, 1), "single_piece_4_4_2_aln_per_s": round(rate1, 1),
                     "mean_affine2p_score": round(mean2, 2), "mean_single_piece_score": round(mean1, 2),
                     "parity_sample": int(len(idx)), "parity_mismatches": int(bad)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
