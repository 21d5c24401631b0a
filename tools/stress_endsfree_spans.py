"""Randomised sweep of per-pair ends-free spans on the GPU: every round (tests/newpath_cases.py) gets a span per pair from a
cycle of shapes (zero, partly free, clamped, len - 1 / len / len + 1, fully free, the round's own span) and is aligned
in one wfagpu_align_spans call with CIGAR.  Every pair's score must equal the exact ends-free DP under its span, its
CIGAR must pass wfagpu_check_result_span, and no pair may fail.  Prints one JSON line; exit code 1 on any mismatch.

usage: stress_endsfree_spans.py [--seed S] [--rounds N] [--scale F]"""
import argparse
import json
import os
import sys
from multiprocessing import Pool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "wfa-gpu_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import newpath_cases as cases  # noqa: E402
import wfagpu  # noqa: E402
from endsfree_ref import gotoh_span, span_cost_ok  # noqa: E402
from endsfree_spans_check import mixed_spans  # noqa: E402


def _dp(job):
    p, t, pen, span = job
    return gotoh_span(p, t, *pen, span)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seed", type=int, default=20261024)
    ap.add_argument("--rounds", type=int, default=20)
    ap.add_argument("--scale", type=float, default=0.5)
    args = ap.parse_args()
    lib = wfagpu.load()
    pairs_total, bad = 0, []
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        for r in range(args.rounds):
            rd = cases.ef_round(args.seed + r, scale=args.scale)
            ps, pen = rd["pairs"], rd["pen"]
            spans = [rd["span"] if j % 5 == 4 else mixed_spans(p, t, j + r) for j, (p, t) in enumerate(ps)]
            a = wfagpu.Aligner()
            for p, t in ps:
                assert a.add_sequences(p, t)
            assert a.initialize_parameters(*pen)
            a.options.compute_cigar = True
            a.options.max_error = rd["budget"]
            a.set_batch_size(rd["batch"])
            a.align(ends_free=spans)
            if a.run_stats()["failed_pairs"]:
                bad.append((r, "failed pairs"))
            want = pool.map(_dp, [(p, t, pen, sp) for (p, t), sp in zip(ps, spans)], chunksize=2)
            for i, ((p, t), sp, s) in enumerate(zip(ps, spans, want)):
                if a.error(i) != s or not span_cost_ok(lib, p, t, *pen, sp, s, a.cigar(i)):
                    bad.append((r, i, list(pen), list(sp), a.error(i), s))
            pairs_total += len(ps)
    print(json.dumps({"seed": args.seed, "rounds": args.rounds, "pairs": pairs_total, "mismatches": len(bad),
                      "first": bad[:5]}))
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
