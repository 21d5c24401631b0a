"""Ends-free throughput: reads aligned inside flanked windows of the text, end to end through wfagpu_align_span, and the
same pairs aligned globally for context, plus a parity sample against the exact ends-free DP.  Prints one JSON line
with the card's name and power limit.

  workload 1: 8192 x 10 kbp reads at 5 % error, windows of 10 kbp + 500 bp flanks, span (0, 0, 500, 500), CIGAR
  workload 2: 100000 x 150 bp reads, 16 bp flanks, span (0, 0, 16, 16), CIGAR

usage: endsfree_probe.py [--reps N] [--sample N] [--small]"""
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
from endsfree_ref import gotoh_span, span_cost_ok  # noqa: E402

BASES = np.frombuffer(b"ACGT", np.uint8)


def windows(seed, n, length, flank, err):
    """Reads with err / 3 substitutions, deletions and insertions each, inside text windows of length + 2 flank."""
    rng = np.random.default_rng(seed)
    pairs = []
    for _ in range(n):
        core = BASES[rng.integers(0, 4, length)]
        r = rng.random(length)
        read = core.copy()
        sub = r < err / 3
        read[sub] = BASES[rng.integers(0, 4, int(sub.sum()))]
        keep = ~((r >= err / 3) & (r < 2 * err / 3))
        ins = (r >= 2 * err / 3) & (r < err)
        reps = keep.astype(np.int64) + ins
        out = np.repeat(read, reps)
        # the second copy of every inserted base becomes a random base
        ends = np.cumsum(reps) - 1
        out[ends[ins]] = BASES[rng.integers(0, 4, int(ins.sum()))]
        text = np.concatenate([BASES[rng.integers(0, 4, flank)], core, BASES[rng.integers(0, 4, flank)]])
        pairs.append((out.tobytes().decode(), text.tobytes().decode()))
    return pairs


def timed(pairs, span, reps):
    a = wfagpu.Aligner()
    for p, t in pairs:
        a.add_sequences(p, t)
    a.initialize_parameters(2, 3, 1)
    a.options.compute_cigar = True
    a.options.max_error = 2000
    times = []
    for r in range(reps + 1):                   # the first call warms up the device and the provisioning
        a.reset_results()
        t0 = time.perf_counter()
        a.align(ends_free=span)
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
    out = {"card": card}
    for name, n, length, flank in (("reads_10kbp_in_windows", 8192, 10000, 500), ("short_reads_150bp", 100000, 150, 16)):
        if args.small:
            n, length = 64, min(length, 1000)
        pairs = windows(0xEF10 + length, n, length, flank, 0.05)
        span = (0, 0, flank, flank)
        a, ef_rate = timed(pairs, span, args.reps)
        rng = np.random.default_rng(7)
        bad = 0
        lib = wfagpu.load()
        idx = rng.choice(n, size=min(args.sample, n), replace=False)
        for i in idx:
            p, t = pairs[i]
            s = gotoh_span(p, t, 2, 3, 1, span)
            bad += a.error(int(i)) != s or not span_cost_ok(lib, p, t, 2, 3, 1, span, s, a.cigar(int(i)))
        mean_score = float(np.mean(a.errors()))
        _, gl_rate = timed(pairs, None, args.reps)
        out[name] = {"pairs": n, "span": list(span), "ends_free_aln_per_s": round(ef_rate, 1),
                     "global_aln_per_s": round(gl_rate, 1), "mean_ends_free_score": round(mean_score, 2),
                     "parity_sample": int(len(idx)), "parity_mismatches": int(bad)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
