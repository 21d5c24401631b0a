"""The CPU model of the ends-free kernel path (tests/endsfree_model.py) against the exact ends-free DP, the oracle and
the library's host decoder; and the exactness of the range pruning with poisoned pruned cells."""
import numpy as np
import pytest

import endsfree_model as model
from endsfree_ref import gotoh_span, ops_to_cigar_span, span_cost_ok, window_pairs

PENALTIES = [(2, 3, 1), (1, 0, 1), (2, 24, 9), (4, 6, 2), (5, 3, 2), (3, 1, 4), (2, 10, 5), (6, 4, 2)]
F = 8
SPANS = [(0, 0, F, F), (F, F, 0, 0), (0, F, F, 0), (3, 1, 0, 5), (0, 2, 7, 0), (60, 60, 60, 60), (10 ** 6,) * 4]
TINY = [("", ""), ("", "ACG"), ("ACG", ""), ("A", "C"), ("A", "A"), ("G", "ACGTA"), ("AC", "ACAC"), ("ACAC", "AC")]


def pairs_for(pen):
    return window_pairs(0xEF00 + sum(pen), [(6, 40, F, 0.15)]) + TINY


@pytest.mark.parametrize("pen", PENALTIES)
def test_model_equals_the_dp_and_its_cigars_cost_the_score(oracle, lib, pen):
    for p, t in pairs_for(pen):
        for span in SPANS:
            m = model.align(oracle, p, t, *pen, span)
            s = gotoh_span(p, t, *pen, span)
            assert m["finished"] and m["distance"] == s, (p, t, span, m["distance"], s)
            # consumes both sequences, costs the score under the span
            assert span_cost_ok(lib, p, t, *pen, span, s, m["cigar"]), (p, t, span, m["cigar"])
            # the library's host decoder prints the model's text from the model's op stream
            assert ops_to_cigar_span(lib, p, t, m["k_begin"], m["ops"]) == m["cigar"], (p, t, span)


@pytest.mark.parametrize("pen", PENALTIES[:4])
def test_model_with_zero_span_equals_the_oracle(oracle, pen):
    for p, t in pairs_for(pen):
        r = oracle.align(p, t, *pen, 4000)
        m = model.align(oracle, p, t, *pen, (0, 0, 0, 0))
        assert (m["distance"], m["cigar"]) == (r["distance"], r["cigar"]), (p, t)


def test_lowest_finishing_diagonal_wins(oracle):
    # "AC" ends the text's first and second copy at score 0: k = 0 and k = 2 both finish, k = 0 wins
    m = model.align(oracle, "AC", "ACAC", 2, 3, 1, (0, 0, 2, 2))
    assert (m["distance"], m["k_begin"], m["k_end"], m["cigar"]) == (0, 0, 0, "2M2I")
    m = model.align(oracle, "ACAC", "AC", 2, 3, 1, (2, 2, 0, 0))
    assert (m["distance"], m["k_begin"], m["k_end"], m["cigar"]) == (0, -2, -2, "2D2M")


@pytest.mark.parametrize("pen", [(2, 3, 1), (4, 6, 2), (5, 3, 2), (1, 0, 1)])
def test_range_pruning_is_exact(oracle, pen):
    # Cells with d + e * dist(k, [kt - te, kt + pe]) > dmax are never computed; the model poisons them, so a read of
    # one would corrupt the result.  Every pair must come out with the unpruned score, path and CIGAR down to
    # dmax = s, and must not finish with dmax = s - 1.
    rng = np.random.default_rng(sum(pen))
    pairs = window_pairs(int(rng.integers(1 << 30)), [(6, 120, 12, 0.1), (3, 60, 30, 0.3)]) + TINY
    for span in ((0, 0, 12, 12), (12, 12, 0, 0), (0, 12, 12, 0), (3, 1, 0, 5), (10 ** 6,) * 4):
        for p, t in pairs:
            full = model.align(oracle, p, t, *pen, span)
            s = full["distance"]
            for dmax in (s, s + 1, s + 3, int(1.2 * s) + 2, 3 * s + 7):
                m = model.align(oracle, p, t, *pen, span, dmax=dmax)
                assert (m["finished"], m["distance"], m["k_begin"], m["k_end"], m["cigar"]) == (
                    True, s, full["k_begin"], full["k_end"], full["cigar"]), (p, t, span, dmax)
            if s > 0:
                assert not model.align(oracle, p, t, *pen, span, dmax=s - 1)["finished"], (p, t, span)
