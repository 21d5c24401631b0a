"""Aligns the gap-affine 2-piece test batches and writes {config: {"scores": [...], "cigars": [...]}} as JSON to argv[1].
Run in a subprocess with WFAGPU_* variables that select a kernel variant (read once when the device opens);
AP_MAX_ERROR sets the first pass's budget (small: pairs are re-dispatched), AP_BATCH the batch size."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "wfa-gpu_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import wfagpu  # noqa: E402
from affine2p_ref import indel_pairs  # noqa: E402

# minimap2-like, a WFA2-lib-like long-read set, o1 = 0, the pieces swapped; identical pieces (single-piece equality)
PENALTIES = [(4, 4, 2, 24, 1), (19, 39, 3, 81, 1), (2, 0, 2, 6, 1), (4, 24, 1, 4, 2), (2, 3, 1, 3, 1), (4, 6, 2, 6, 2)]
CONFIGS = [(pen, True) for pen in PENALTIES] + [((4, 4, 2, 24, 1), False), ((2, 3, 1, 3, 1), False)]


def batch():
    # 150 bp (warp per pair), 1 kbp (CTA per pair), 5 kbp; one 50 .. 500 bp indel per pair
    pairs = indel_pairs(0xA2C1, [(24, 150, 0.05, 20, 50), (9, 1000, 0.05, 50, 300), (3, 5000, 0.03, 100, 500)])
    for i in (0, 1, 2, 25, 26):
        p, t = pairs[i]
        pairs.append((p[:30] + "N" + p[31:], t[:50] + "NN" + t[52:]))
    pairs += [("", "ACGT"), ("ACGT", ""), ("", ""), ("A", "C"), ("A", "A"), ("ACGTACGTAC", "TTTTTTTTTT"), ("A", "A" * 40)]
    # ties between the pieces and between gap placements
    pairs += [("AC", "ACAC"), ("ACAC", "AC"), ("ACGT" * 5, "ACGT" * 9), ("ACGT" * 9, "ACGT" * 5), ("A" * 30, "A" * 50)]
    return pairs


def key(pen, cigar):
    return "%s|%s" % (",".join(map(str, pen)), "cigar" if cigar else "score")


def run(pairs, pen, cigar, max_error=600, batch_size=0, single=False):
    """single: the plain single-piece wfagpu_align with (x, o1, e1) instead of the 2-piece call."""
    a = wfagpu.Aligner()
    for p, t in pairs:
        assert a.add_sequences(p, t)
    assert a.initialize_parameters(*pen[:3])
    a.options.compute_cigar = cigar
    a.options.max_error = max_error
    if batch_size:
        a.set_batch_size(batch_size)
    a.align() if single else a.align(affine2p=pen)
    st = a.run_stats()
    assert st["failed_pairs"] == 0, st
    return dict(scores=a.errors(), cigars=a.cigars() if cigar else None)


if __name__ == "__main__":
    pairs = batch()
    me, bs = int(os.environ.get("AP_MAX_ERROR", "600")), int(os.environ.get("AP_BATCH", "0"))
    out = {key(pen, cigar): run(pairs, pen, cigar, me, bs) for pen, cigar in CONFIGS}
    with open(sys.argv[1], "w") as f:
        json.dump(out, f)
