"""Aligns the coordinate test jobs three ways -- the plain ends-free call with CIGAR, and align(coords=True) score only
and with CIGAR -- and writes {job: {"plain": ..., "score": ..., "cigar": ...}} as JSON to argv[1].  Run in a subprocess
with WFAGPU_* variables that select a kernel variant (read once when the device opens); EF_MAX_ERROR sets the first
pass's budget (small: pairs are re-dispatched), EF_BATCH the batch size."""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "wfa-gpu_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

import endsfree_check  # noqa: E402
import newpath_cases as cases  # noqa: E402
import wfagpu  # noqa: E402
from endsfree_ref import mutate, rand_seq, window_pairs  # noqa: E402

SWEEP_SEED, SWEEP_ROUNDS = 20261022, 4
BIG = 10 ** 6


def _edge_pairs():
    rng = np.random.default_rng(0xC0DE)
    # 200-base patterns against 260-base texts, so that the spans below sit on the clamp edges of every pair
    out = window_pairs(0xC0DE, [(6, 200, 30, 0.05)])
    out = [(p[:200].ljust(200, "A"), t[:260].ljust(260, "C")) for p, t in out]
    core = rand_seq(rng, 200)
    out += [(core, rand_seq(rng, 30) + core + rand_seq(rng, 30)),       # score 0 with a free text
            (core, core + rand_seq(rng, 60)), (core, rand_seq(rng, 60) + core),
            ("ACGT" * 50, "ACGT" * 65), (mutate(rng, core, 0.1), rand_seq(rng, 17) + core + rand_seq(rng, 43))]
    return out


def jobs():
    """-> {name: (pairs, pen, span or None, max_error, batch)}"""
    me, bs = int(os.environ.get("EF_MAX_ERROR", "400")), int(os.environ.get("EF_BATCH", "0"))
    out = {}
    pairs = endsfree_check.batch()
    for pen, span, _ in endsfree_check.CONFIGS:
        out["batch|" + endsfree_check.key(pen, span, False)] = (pairs, pen, span, me, bs)
    out["batch|global"] = (pairs, (2, 3, 1), None, me, bs)
    for i in range(SWEEP_ROUNDS):
        rd = cases.ef_round(SWEEP_SEED + i, scale=0.3)
        out["sweep|%d" % i] = (rd["pairs"], rd["pen"], rd["span"], min(me, rd["budget"]), bs or rd["batch"])
    edges = _edge_pairs()
    for span in [(200, 200, 0, 0), (199, 199, 0, 0), (0, 0, 260, 260), (0, 0, 259, 259), (0, 0, BIG, BIG), (BIG,) * 4,
                 (200, 0, 0, 260), (0, 199, 259, 0), (1, 1, 1, 1)]:
        out["edge|" + ",".join(map(str, span))] = (edges, (2, 3, 1), span, me, bs)
    out["edge|global"] = (edges, (4, 6, 2), None, me, bs)
    # one pair longer than the int16 offsets of the shared-memory tiers (int32 rings in global memory)
    out["long"] = (window_pairs(0x10A6, [(1, 33000, 400, 0.01)]), (2, 3, 1), (0, 0, 400, 400), me, bs)
    return out


def align(pairs, pen, span, cigar, coords, max_error, batch):
    a = wfagpu.Aligner()
    for p, t in pairs:
        assert a.add_sequences(p, t)
    assert a.initialize_parameters(*pen)
    a.options.compute_cigar = cigar
    a.options.max_error = max_error
    if batch:
        a.set_batch_size(batch)
    a.align(ends_free=span, coords=coords)
    assert a.run_stats()["failed_pairs"] == 0
    return dict(scores=a.errors(), cigars=a.cigars() if cigar else None, coords=a.coords() if coords else None)


if __name__ == "__main__":
    res = {}
    for name, (pairs, pen, span, me, bs) in jobs().items():
        res[name] = dict(plain=align(pairs, pen, span, True, False, me, bs),
                         score=align(pairs, pen, span, False, True, me, bs),
                         cigar=align(pairs, pen, span, True, True, me, bs))
    with open(sys.argv[1], "w") as f:
        json.dump(res, f)
