"""Per-pair ends-free spans (DESIGN.md §9): a pair aligned inside a batch whose widest start row W is larger than its own
runs on a step table widened by that W, but the kernel clamps every window to the pair's own reach
[-pb - r(d), tb + r(d)] and NULLs only the pair's own prologue.  The CPU model of that (tests/endsfree_spans_model.py,
every cell the kernel does not write poisoned) must give such a pair the score, k_begin, k_end, origin and CIGAR that
tests/endsfree_model.py and tests/endsfree_origin_model.py give the pair alone, and the ends-free DP -- and must not when
the clamp is one diagonal too narrow on either side."""
import os
from multiprocessing import Pool

import pytest

import endsfree_model as model
import endsfree_origin_model as origin_model
import endsfree_spans_model as spans_model
import newpath_cases as cases
import test_endsfree_model as base
from endsfree_ref import clamp, gotoh_span

ROUNDS = 24
KEYS = ("finished", "distance", "k_begin", "k_end", "cigar")


def mixed_spans(p, t, i):
    """The i-th of a cycle of span shapes for one pair: zero, partly free, clamped, len - 1 / len / len + 1, fully free."""
    pl, tl = len(p), len(t)
    return [(0, 0, 0, 0), (0, 0, 8, 8), (pl + 1, 3, 0, tl + 1), (max(0, pl - 1), 0, tl, max(0, tl - 1)),
            (pl, pl, tl, tl), (3, 1, 0, 5), (cases.BIG,) * 4, (0, pl + 1, tl - 1 if tl else 0, 0)][i % 8]


def batch_width(pairs, spans):
    return max(max(clamp(sp, len(p), len(t))[0], clamp(sp, len(p), len(t))[2]) for (p, t), sp in zip(pairs, spans))


def _same(a, b):
    return all(a[k] == b[k] for k in KEYS)


def _narrow_differs(oracle, p, t, pen, span, W, trim):
    try:
        return not _same(spans_model.align(oracle, p, t, *pen, span, W, trim=trim), model.align(oracle, p, t, *pen, span))
    except AssertionError:          # the model's traceback left the computed cells: also a wrong kernel
        return True


@pytest.mark.parametrize("pen", base.PENALTIES[:5])
def test_pair_in_a_wider_batch_equals_the_pair_alone(oracle, pen):
    pairs = base.pairs_for(pen)
    spans = [mixed_spans(p, t, i) for i, (p, t) in enumerate(pairs)]
    W = batch_width(pairs, spans)
    for (p, t), span in zip(pairs, spans):
        alone = model.align(oracle, p, t, *pen, span)
        assert alone["finished"] and alone["distance"] == gotoh_span(p, t, *pen, span), (p, t, span)
        g = origin_model.align(oracle, p, t, *pen, span)
        for w in (W, W + 37):
            m = spans_model.align(oracle, p, t, *pen, span, w)
            assert _same(m, alone), (p, t, span, w, m, alone)
            assert m["k_origin"] == g["k_origin"] == alone["k_begin"], (p, t, span, w)


def test_a_batch_span_equals_the_unclamped_kernel(oracle):
    # every pair of a batch with one span: the clamp is the pair's own reach of the same step table (no narrower than the
    # unclamped window wherever a cell can be non-NULL), down to the pruning's dmax = s
    for pen in base.PENALTIES[:3]:
        for p, t in base.pairs_for(pen)[:6]:
            for span in base.SPANS:
                W = max(clamp(span, len(p), len(t))[0], clamp(span, len(p), len(t))[2])
                alone = model.align(oracle, p, t, *pen, span)
                for dmax in (-1, alone["distance"], alone["distance"] + 2):
                    assert _same(spans_model.align(oracle, p, t, *pen, span, W, dmax=dmax),
                                 model.align(oracle, p, t, *pen, span, dmax=dmax)), (p, t, span, dmax)


_oracle = None


def _round_job(job):
    global _oracle
    p, t, pen, span, W = job
    from oracle import Oracle
    if _oracle is None:
        _oracle = Oracle()
    m = spans_model.align(_oracle, p, t, *pen, span, W)
    alone = model.align(_oracle, p, t, *pen, span)
    g = origin_model.align(_oracle, p, t, *pen, span)
    return (_same(m, alone) and m["finished"] and m["distance"] == gotoh_span(p, t, *pen, span) and
            m["k_origin"] == g["k_origin"] == m["k_begin"])


def test_mixed_spans_on_random_rounds_match_the_dp():
    jobs = []
    for seed in range(ROUNDS):
        rd = cases.ef_round(0x5A4 + seed, scale=0.3)
        ps = rd["pairs"]
        spans = [rd["span"] if i % 9 == 8 else mixed_spans(p, t, i + seed) for i, (p, t) in enumerate(ps)]
        W = batch_width(ps, spans)
        jobs += [(p, t, rd["pen"], sp, W) for (p, t), sp in zip(ps, spans)]
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        res = pool.map(_round_job, jobs, chunksize=4)
    bad = [j[:4] for j, ok in zip(jobs, res) if not ok]
    assert not bad, bad[:3]
    assert sum(1 for j in jobs if j[4] > max(clamp(j[3], len(j[0]), len(j[1]))[::2])) > len(jobs) // 2


@pytest.mark.parametrize("trim", [(1, 0), (0, 1)])
def test_a_clamp_one_diagonal_too_narrow_is_caught(oracle, trim):
    # leading free bases followed by a gap: the optimal path runs on the edge of the pair's own reach
    pen = (2, 3, 1)
    p, t = "ACGTTGCA" + "GATTACA" * 3, "TT" + "GATTACA" * 3
    hits = 0
    for span in ((8, 0, 0, 0), (0, 0, 2, 0), (8, 0, 2, 0), (0, 0, 0, 0)):
        for W in (max(span[0], span[2]), 40):
            hits += _narrow_differs(oracle, p, t, pen, span, W, trim)
    for p, t in base.pairs_for(pen):
        for i in range(8):
            hits += _narrow_differs(oracle, p, t, pen, mixed_spans(p, t, i), 60, trim)
    assert hits > 0
