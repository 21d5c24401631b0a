"""What coordinates cost: the DESIGN.md §9 ends-free workloads end to end through Aligner.align in three modes --
score only, score only with coordinates (origin rows), and CIGAR with coordinates (traceback) -- median of N calls after
a warm-up call, and whether both coordinate modes agree.  Prints one JSON line with the card's name and power limit.

  reads_10kbp_in_windows: 8192 x 10 kbp reads at 5 % error in windows with 500 bp flanks, span (0, 0, 500, 500)
  reads_10kbp_free_text:  the same pairs, the whole text free (span (0, 0, 10**6, 10**6))
  short_reads_150bp:      100000 x 150 bp reads, 16 bp flanks, span (0, 0, 16, 16)

usage: endsfree_coords_probe.py [--reps N] [--small]"""
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

MODES = {"score_only": (False, False), "score_only_coords": (False, True), "cigar_coords": (True, True)}


def timed(a, span, cigar, coords, reps):
    a.options.compute_cigar = cigar
    times = []
    for r in range(reps + 1):                   # the first call warms up the device and the provisioning
        a.reset_results()
        t0 = time.perf_counter()
        a.align(ends_free=span, coords=coords)
        dt = time.perf_counter() - t0
        if r:
            times.append(dt)
    assert a.run_stats()["failed_pairs"] == 0
    return statistics.median(times), (a.coords() if coords else None)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--small", action="store_true", help="tiny sizes (a dry run of the script)")
    args = ap.parse_args()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True)
    card = q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"
    out = {"card": card, "reps": args.reps}
    for name, n, length, flank, span in (("reads_10kbp_in_windows", 8192, 10000, 500, (0, 0, 500, 500)),
                                         ("reads_10kbp_free_text", 8192, 10000, 500, (0, 0, 10 ** 6, 10 ** 6)),
                                         ("short_reads_150bp", 100000, 150, 16, (0, 0, 16, 16))):
        if args.small:
            n, length = 64, min(length, 1000)
        pairs = windows(0xEF10 + length, n, length, flank, 0.05)     # the pairs of tools/endsfree_probe.py
        a = wfagpu.Aligner()
        for p, t in pairs:
            a.add_sequences(p, t)
        a.initialize_parameters(2, 3, 1)
        a.options.max_error = 2000
        res, coords = {"pairs": n, "span": list(span)}, {}
        for mode, (cigar, want) in MODES.items():
            dt, coords[mode] = timed(a, span, cigar, want, args.reps)
            res[mode + "_ms"] = round(dt * 1e3, 2)
            res[mode + "_aln_per_s"] = round(n / dt, 1)
        res["coords_agree"] = coords["score_only_coords"] == coords["cigar_coords"]
        out[name] = res
    print(json.dumps(out))


if __name__ == "__main__":
    main()
