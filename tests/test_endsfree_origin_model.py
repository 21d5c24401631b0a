"""The CPU model of the score-only kernel's origin rows (tests/endsfree_origin_model.py), with every origin cell the
kernel never writes poisoned, must finish where tests/endsfree_model.py finishes and give its traceback's k_begin on
every case of
tests/test_endsfree_model.py and on the random rounds of tests/newpath_cases.py -- tie pairs and score-0 pairs
included.  This is the rule the GPU's score-only coordinates are checked against."""
import os
from multiprocessing import Pool

import numpy as np
import pytest

import endsfree_model as model
import endsfree_origin_model as origin_model
import newpath_cases as cases
import test_endsfree_model as base
from endsfree_ref import window_pairs

ROUNDS = 40


def _begins(oracle, p, t, pen, span, **kw):
    """-> (traceback model, origin model) after checking that both finish alike and start on the same diagonal."""
    m = model.align(oracle, p, t, *pen, span, cigar=False, **kw)
    g = origin_model.align(oracle, p, t, *pen, span, **kw)
    assert (g["finished"], g["distance"], g["k_end"]) == (m["finished"], m["distance"], m["k_end"]), (p, t, pen, span, kw)
    assert g["k_origin"] == m["k_begin"], (p, t, pen, span, kw, g["k_origin"], m["k_begin"])
    return m, g


def _same_begin(oracle, p, t, pen, span, **kw):
    return _begins(oracle, p, t, pen, span, **kw)[0]


@pytest.mark.parametrize("pen", base.PENALTIES)
def test_origin_equals_the_traceback_begin(oracle, pen):
    for p, t in base.pairs_for(pen):
        for span in base.SPANS:
            assert _same_begin(oracle, p, t, pen, span)["finished"]


@pytest.mark.parametrize("pen", [(2, 3, 1), (4, 6, 2), (5, 3, 2), (1, 0, 1)])
def test_origin_is_exact_under_range_pruning(oracle, pen):
    # the cases of test_range_pruning_is_exact: pruned cells hold poisoned origins as well as poisoned values
    rng = np.random.default_rng(sum(pen))
    pairs = window_pairs(int(rng.integers(1 << 30)), [(6, 120, 12, 0.1), (3, 60, 30, 0.3)]) + base.TINY
    for span in ((0, 0, 12, 12), (12, 12, 0, 0), (0, 12, 12, 0), (3, 1, 0, 5), (10 ** 6,) * 4):
        for p, t in pairs:
            s = _same_begin(oracle, p, t, pen, span)["distance"]
            for dmax in (s, s + 1, s + 3, 3 * s + 7):
                assert _same_begin(oracle, p, t, pen, span, dmax=dmax)["finished"]


def test_origin_on_ties_and_score_zero(oracle):
    # score-0 finishes on two diagonals (the lowest wins) and tandem repeats where gap placements tie
    for p, t, span in [("AC", "ACAC", (0, 0, 2, 2)), ("ACAC", "AC", (2, 2, 0, 0)), ("ACGT" * 5, "ACGT" * 9, (0, 0, 9, 9)),
                       ("ACGTACGT", "ACGACGTACGT", (0, 0, 0, 0)), ("AAAA", "AAAAAAAAAA", (0, 0, 3, 3)),
                       ("GATTACA", "GATTACA", (10 ** 6,) * 4)]:
        m = _same_begin(oracle, p, t, (2, 3, 1), span)
        assert m["finished"]


_oracle = None


def _round_job(job):
    global _oracle
    p, t, pen, span = job
    from oracle import Oracle
    if _oracle is None:
        _oracle = Oracle()
    m = model.align(_oracle, p, t, *pen, span, cigar=False)
    g = origin_model.align(_oracle, p, t, *pen, span)
    return m["finished"] and (g["finished"], g["distance"], g["k_end"]) == (True, m["distance"], m["k_end"]), \
        g["k_origin"], m["k_begin"]


def test_origin_equals_the_traceback_begin_on_random_rounds():
    jobs = []
    for seed in range(ROUNDS):
        rd = cases.ef_round(0x5EED + seed, scale=0.3)
        jobs += [(p, t, rd["pen"], rd["span"]) for p, t in rd["pairs"]]
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        res = pool.map(_round_job, jobs, chunksize=4)
    for (p, t, pen, span), (fin, k_origin, k_begin) in zip(jobs, res):
        assert fin and k_origin == k_begin, (pen, span, p, t, k_origin, k_begin)
    assert sum(1 for (fin, ko, kb) in res if ko != 0) > len(res) // 4     # most begins are off diagonal 0
