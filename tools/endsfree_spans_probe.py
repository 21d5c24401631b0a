"""Per-pair ends-free spans on a mixed batch: 100 000 x 150 bp reads in windows with 16 bp flanks, span (0, 0, 16, 16),
plus 64 x 10 kbp reads with the text fully free, span (0, 0, 10**6, 10**6); CIGAR.  Times one wfagpu_align_spans call over
all pairs against the same pairs split by span into two wfagpu_align_span calls, and checks that both give the same
scores and CIGARs.  Prints one JSON line with the card's name and power limit.

usage: endsfree_spans_probe.py [--reps N] [--small]"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "wfa-gpu_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import wfagpu  # noqa: E402
from endsfree_probe import windows  # noqa: E402

FREE = 10 ** 6


def aligner(pairs):
    a = wfagpu.Aligner()
    for p, t in pairs:
        a.add_sequences(p, t)
    a.initialize_parameters(2, 3, 1)
    a.options.compute_cigar = True
    a.options.max_error = 2000
    return a


def timed(calls, reps):
    """calls: [(aligner, ends_free)], run back to back; -> median seconds of the whole set"""
    times = []
    for r in range(reps + 1):                   # the first round warms up the device and the provisioning
        for a, _ in calls:
            a.reset_results()
        t0 = time.perf_counter()
        for a, ef in calls:
            a.align(ends_free=ef)
        dt = time.perf_counter() - t0
        if r:
            times.append(dt)
    for a, _ in calls:
        assert a.run_stats()["failed_pairs"] == 0
    return statistics.median(times)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--small", action="store_true", help="tiny sizes (a dry run of the script)")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    card = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"
    n_short, n_long, long_len = (2000, 4, 2000) if args.small else (100000, 64, 10000)
    short = windows(0x5B10, n_short, 150, 16, 0.05)
    long_ = windows(0x5B11, n_long, long_len, 500, 0.05)
    spans = [(0, 0, 16, 16)] * n_short + [(0, 0, FREE, FREE)] * n_long
    mixed = aligner(short + long_)
    a_short, a_long = aligner(short), aligner(long_)
    t_one = timed([(mixed, spans)], args.reps)
    t_two = timed([(a_short, (0, 0, 16, 16)), (a_long, (0, 0, FREE, FREE))], args.reps)
    same = (mixed.errors() == a_short.errors() + a_long.errors() and mixed.cigars() == a_short.cigars() + a_long.cigars())
    n = n_short + n_long
    print(json.dumps({"card": card, "pairs": n, "one_per_pair_call_aln_per_s": round(n / t_one, 1),
                      "two_calls_split_by_span_aln_per_s": round(n / t_two, 1), "one_call_s": round(t_one, 4),
                      "two_calls_s": round(t_two, 4), "same_results": bool(same)}))


if __name__ == "__main__":
    main()
