"""Aligns the per-pair span test jobs and writes {job: {...}} as JSON to argv[1]: the per-pair call (wfagpu_align_spans)
with CIGAR and coordinates, score only with coordinates, and with CIGAR alone; every pair alone through wfagpu_align_span
with its span (argv[2] == "alone"); the reference calls a job's spans must reproduce byte for byte (one batch span for n
equal spans, wfagpu_align for all-zero spans); and the check_correctness counts of wfagpu_launch_alignments_spans.  Run
in a subprocess with WFAGPU_* variables that select a kernel variant; EF_MAX_ERROR sets the first pass's budget (small:
pairs are re-dispatched), EF_BATCH the batch size (cuts the span array mid-chunk)."""
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "wfa-gpu_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import newpath_cases as cases  # noqa: E402
import wfagpu  # noqa: E402
from endsfree_ref import mutate, rand_seq, window_pairs  # noqa: E402

BIG = 10 ** 6


def mixed_spans(p, t, i):
    """The i-th of a cycle of span shapes: zero, partly free, clamped, len - 1 / len / len + 1, fully free."""
    pl, tl = len(p), len(t)
    return [(0, 0, 0, 0), (0, 0, 16, 16), (pl + 1, 3, 0, tl + 1), (max(0, pl - 1), 0, tl, max(0, tl - 1)),
            (0, 0, 0, 0), (3, 1, 0, 5), (BIG,) * 4, (0, pl + 1, max(0, tl - 1), 0), (pl, pl, tl, tl)][i % 9]


def _reads_in_windows(seed, n, length, flank, err):
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        core = rand_seq(rng, length)
        a, b = int(rng.integers(0, flank + 1)), int(rng.integers(0, flank + 1))
        out.append((mutate(rng, core, err), rand_seq(rng, a) + core + rand_seq(rng, b)))
    return out


def jobs():
    """-> {name: (pairs, pen, spans, reference, max_error, batch)}; reference: "span" (all spans equal), "global" (all
    zero) or None"""
    me, bs = int(os.environ.get("EF_MAX_ERROR", "400")), int(os.environ.get("EF_BATCH", "0"))
    out = {}
    reads = _reads_in_windows(0x5A11, 40, 150, 16, 0.04) + window_pairs(0x5A12, [(12, 300, 40, 0.08)])
    reads += [("", ""), ("", "ACG"), ("ACG", ""), ("A", "C"), ("AC", "ACAC"), ("ACAC", "AC")]
    out["mixed"] = (reads, (2, 3, 1), [mixed_spans(p, t, i) for i, (p, t) in enumerate(reads)], None, me, bs)
    # a fully free 2 kbp pair among 150 bp reads with 16 bp flanks: the reads' own reach is far narrower than the batch's
    wide = _reads_in_windows(0x5A13, 1, 2000, 400, 0.03)
    out["wide"] = (reads[:40] + wide, (4, 6, 2), [(0, 0, 16, 16)] * 40 + [(0, 0, BIG, BIG)], None, me, bs)
    for i in range(4):
        rd = cases.ef_round(20261023 + i, scale=0.3)
        ps = rd["pairs"]
        spans = [rd["span"] if j % 5 == 4 else mixed_spans(p, t, j + i) for j, (p, t) in enumerate(ps)]
        out["sweep|%d" % i] = (ps, rd["pen"], spans, None, min(me, rd["budget"]), bs or rd["batch"])
    out["uniform"] = (reads, (2, 3, 1), [(5, 7, 16, 16)] * len(reads), "span", me, bs)
    out["zeros"] = (reads, (2, 3, 1), [(0, 0, 0, 0)] * len(reads), "global", me, bs)
    # pairs with N (byte-compare kernel) and one pair longer than the int16 offsets of the shared-memory tiers
    rng = np.random.default_rng(0x5A14)
    withn = []
    for p, t in reads[:12]:
        at = int(rng.integers(len(p))) if p else 0
        withn.append((p[:at] + "N" + p[at + 1:], t))
    out["n_pairs"] = (withn + reads[12:20], (2, 3, 1), [mixed_spans(p, t, i) for i, (p, t) in enumerate(withn + reads[12:20])],
                      None, me, bs)
    big = window_pairs(0x10A7, [(1, 33000, 300, 0.01)])
    out["long"] = (big + reads[:8], (2, 3, 1), [(0, 0, 300, 300)] + [mixed_spans(p, t, i) for i, (p, t) in enumerate(reads[:8])],
                   None, me, bs)
    return out


def _aligner(pairs, pen, cigar, max_error, batch):
    a = wfagpu.Aligner()
    for p, t in pairs:
        assert a.add_sequences(p, t)
    assert a.initialize_parameters(*pen)
    a.options.compute_cigar = cigar
    a.options.max_error = max_error
    if batch:
        a.set_batch_size(batch)
    return a


def align(pairs, pen, spans, cigar, coords, max_error, batch, ends_free="spans"):
    a = _aligner(pairs, pen, cigar, max_error, batch)
    if ends_free == "spans":
        a.align(ends_free=spans, coords=coords)
    elif ends_free == "span":
        a.align(ends_free=spans[0], coords=coords)
    else:
        a.align(coords=coords)
    assert a.run_stats()["failed_pairs"] == 0
    return dict(scores=a.errors(), cigars=a.cigars() if cigar else None, coords=a.coords() if coords else None)


def checked(pairs, pen, spans, cigar, max_error, batch):
    a = _aligner(pairs, pen, cigar, max_error, batch)
    sp = wfagpu.spans_of(spans, len(pairs))
    a.L.wfagpu_launch_alignments_spans(a.s.sequences_buffer, a.s.sequences_buffer_len, a.s.sequences_metadata,
                                       a.s.results, a.options, cigar, True, sp, None)
    st = a.run_stats()
    return [st["checked"], st["incorrect"], st["failed_pairs"]]


if __name__ == "__main__":
    with_alone = len(sys.argv) > 2 and sys.argv[2] == "alone"
    res = {}
    for name, (pairs, pen, spans, ref, me, bs) in jobs().items():
        r = dict(cigar=align(pairs, pen, spans, True, True, me, bs),
                 score=align(pairs, pen, spans, False, True, me, bs),
                 plain=align(pairs, pen, spans, True, False, me, bs),
                 check=[checked(pairs, pen, spans, c, me, bs) for c in (True, False)])
        if ref:
            r["ref"] = dict(cigar=align(pairs, pen, spans, True, True, me, bs, ref),
                            score=align(pairs, pen, spans, False, True, me, bs, ref))
        if with_alone:
            alone = [[align([pt], pen, [sp], c, True, me, 0, "span") for c in (True, False)]
                     for pt, sp in zip(pairs, spans)]
            r["alone"] = dict(cigar=dict(scores=[c["scores"][0] for c, _ in alone], cigars=[c["cigars"][0] for c, _ in alone],
                                         coords=[c["coords"][0] for c, _ in alone]),
                              score=dict(scores=[s["scores"][0] for _, s in alone], coords=[s["coords"][0] for _, s in alone]))
        res[name] = r
    with open(sys.argv[1], "w") as f:
        json.dump(res, f)
