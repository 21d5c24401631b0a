"""Aligns the ends-free test batches and writes {config: {"scores": [...], "cigars": [...]}} as JSON to argv[1].
Run in a subprocess with WFAGPU_* variables that select a kernel variant (read once when the device opens);
EF_MAX_ERROR sets the first pass's budget (small: pairs are re-dispatched), EF_BATCH the batch size."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "wfa-gpu_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import wfagpu  # noqa: E402
from endsfree_ref import window_pairs  # noqa: E402

# 150 bp (warp per pair), 1 kbp (CTA per pair), 5 kbp; plus pairs with 'N' (byte-compare kernel) and tiny ones
SPANS = [(0, 0, 20, 20), (40, 40, 0, 0), (0, 30, 25, 0), (3, 7, 11, 2), (5000, 5000, 5000, 5000), (10 ** 6,) * 4]
CONFIGS = [((2, 3, 1), s, True) for s in SPANS] + [((2, 3, 1), (0, 0, 20, 20), False), ((2, 3, 1), (3, 7, 11, 2), False)]
CONFIGS += [(pen, s, True) for pen in ((1, 0, 1), (2, 24, 9), (4, 6, 2)) for s in ((0, 0, 20, 20), (0, 30, 25, 0))]


def batch():
    pairs = window_pairs(0xEF01, [(24, 150, 16, 0.05), (9, 1000, 100, 0.05), (3, 5000, 300, 0.03)])
    for i in (0, 1, 2, 25, 26):
        p, t = pairs[i]
        pairs.append((p[:30] + "N" + p[31:], t[:50] + "NN" + t[52:]))
    pairs += [("", "ACGT"), ("ACGT", ""), ("A", "C"), ("A", "A"), ("ACGTACGTAC", "TTTTTTTTTT"), ("A", "A" * 40)]
    # several target diagonals finish at the same score: the lowest one wins
    pairs += [("AC", "ACAC"), ("ACAC", "AC"), ("ACGT" * 5, "ACGT" * 9), ("ACGT" * 9, "ACGT" * 5)]
    return pairs


def key(pen, span, cigar):
    return "%d,%d,%d|%s|%s" % (pen + (",".join(map(str, span)), "cigar" if cigar else "score"))


def run(pairs, pen, span, cigar, max_error=400, batch_size=0):
    a = wfagpu.Aligner()
    for p, t in pairs:
        assert a.add_sequences(p, t)
    assert a.initialize_parameters(*pen)
    a.options.compute_cigar = cigar
    a.options.max_error = max_error
    if batch_size:
        a.set_batch_size(batch_size)
    a.align(ends_free=span)
    st = a.run_stats()
    assert st["failed_pairs"] == 0, st
    return dict(scores=a.errors(), cigars=a.cigars() if cigar else None)


if __name__ == "__main__":
    pairs = batch()
    me, bs = int(os.environ.get("EF_MAX_ERROR", "400")), int(os.environ.get("EF_BATCH", "0"))
    out = {key(pen, span, cigar): run(pairs, pen, span, cigar, me, bs) for pen, span, cigar in CONFIGS}
    with open(sys.argv[1], "w") as f:
        json.dump(out, f)
