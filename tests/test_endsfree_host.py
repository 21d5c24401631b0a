"""Ends-free alignment, host side (no GPU): the exact DP the GPU tests check against, the span cost rule of
wfagpu_check_result_span and the CIGAR text of wfagpu_ops_to_cigar_span."""
import numpy as np
import pytest

from endsfree_ref import gotoh_span, gotoh_span_cells, ops_to_cigar_span, rand_seq, mutate, span_cost_ok, window_pairs

PENALTIES = [(2, 3, 1), (1, 0, 1), (2, 24, 9), (4, 6, 2), (5, 3, 2), (3, 1, 4), (2, 10, 5), (6, 4, 2)]
INS, SUB, DEL = 1, 2, 3


def test_dp_with_zero_span_equals_the_oracle(oracle):
    rng = np.random.default_rng(11)
    for x, o, e in PENALTIES[:4]:
        for _ in range(12):
            c = rand_seq(rng, int(rng.integers(1, 300)))
            p, t = mutate(rng, c, 0.1), c
            r = oracle.align(p, t, x, o, e, 20000, cigar=False)
            assert r["finished"]
            assert gotoh_span(p, t, x, o, e, (0, 0, 0, 0)) == r["distance"]


@pytest.mark.parametrize("pen", PENALTIES)
def test_dp_equals_the_cell_by_cell_statement(pen):
    rng = np.random.default_rng(sum(pen))
    pairs = window_pairs(int(rng.integers(1 << 30)), [(6, 20, 6, 0.15)])
    pairs += [("", ""), ("", "ACG"), ("ACG", ""), ("A", "C"), ("A", "A"), ("G", "ACGTA")]
    spans = [(0, 0, 0, 0), (0, 0, 6, 6), (6, 6, 0, 0), (0, 6, 6, 0), (3, 1, 0, 5), (40, 40, 40, 40), (10 ** 6,) * 4]
    for p, t in pairs:
        for span in spans:
            assert gotoh_span(p, t, *pen, span) == gotoh_span_cells(p, t, *pen, span), (p, t, span)


def test_free_flanks_cost_nothing():
    rng = np.random.default_rng(3)
    core = rand_seq(rng, 200)
    t = rand_seq(rng, 50) + core + rand_seq(rng, 50)
    assert gotoh_span(core, t, 2, 3, 1, (0, 0, 50, 50)) == 0
    assert gotoh_span(core, t, 2, 3, 1, (0, 0, 49, 50)) == 3 + 1
    assert gotoh_span(core, t, 2, 3, 1, (0, 0, 0, 0)) == 2 * (3 + 50)
    assert gotoh_span("", "ACGT", 2, 3, 1, (0, 0, 1, 2)) == 3 + 1
    assert gotoh_span("", "ACGT", 2, 3, 1, (0, 0, 2, 2)) == 0


def test_check_result_span_accepts_and_rejects(lib):
    p, t = "ACGTACGT", "TTACGTACGTGG"
    assert span_cost_ok(lib, p, t, 2, 3, 1, (0, 0, 2, 2), 0, "2I8M2I")
    assert span_cost_ok(lib, p, t, 2, 3, 1, (0, 0, 0, 0), 10, "2I8M2I")
    assert span_cost_ok(lib, p, t, 2, 3, 1, (0, 0, 1, 2), 4, "2I8M2I")          # leading run longer than its allowance
    assert not span_cost_ok(lib, p, t, 2, 3, 1, (0, 0, 1, 2), 0, "2I8M2I")
    assert not span_cost_ok(lib, p, t, 2, 3, 1, (0, 0, 2, 2), 0, "1I8M3I")      # not an alignment of p with t
    assert not span_cost_ok(lib, p, t, 2, 3, 1, (2, 2, 0, 0), 0, "2I8M2I")      # pattern allowances do not cover I
    assert span_cost_ok(lib, t, p, 2, 3, 1, (2, 2, 0, 0), 0, "2D8M2D")
    assert span_cost_ok(lib, "ACGAACGT", t, 2, 3, 1, (0, 0, 2, 2), 2, "2I3M1X4M2I")
    assert not span_cost_ok(lib, p, t, 2, 3, 1, (0, 0, 2, 2), 0, "2I8M1I1I")    # only the last run is trailing
    assert span_cost_ok(lib, p, t, 2, 3, 1, (0, 0, 2, 2), 4, "2I8M1I1I")
    # one run both leading and trailing uses both allowances
    assert span_cost_ok(lib, "", "ACGTA", 2, 3, 1, (0, 0, 2, 3), 0, "5I")
    assert span_cost_ok(lib, "", "ACGTA", 2, 3, 1, (0, 0, 2, 2), 4, "5I")
    assert span_cost_ok(lib, "", "", 2, 3, 1, (0, 0, 0, 0), 0, "")
    assert not span_cost_ok(lib, p, t, 2, 3, 1, (-1, 0, 2, 2), 0, "2I8M2I")


def test_ops_to_cigar_span(lib):
    # score 0: leading run, match, trailing run
    assert ops_to_cigar_span(lib, "ACGT", "TTACGTTT", 2, []) == "2I4M2I"
    assert ops_to_cigar_span(lib, "TTACGTTT", "ACGT", -2, []) == "2D4M2D"
    assert ops_to_cigar_span(lib, "", "ACG", 1, []) == "3I"                         # leading and trailing join
    # the leading free run joins a gap of the same letter that opens on the start cell
    assert ops_to_cigar_span(lib, "AC", "GGTAC", 2, [INS, SUB]) == "3I2M"
    # the trailing free run joins the last gap through its delimiter
    assert ops_to_cigar_span(lib, "AC", "ACGG", 0, [INS, SUB]) == "2M2I"
    # a mismatch keeps them apart
    assert ops_to_cigar_span(lib, "ACGA", "TACGTG", 1, [SUB]) == "1I3M1X1I"
    # a gap inside the path
    assert ops_to_cigar_span(lib, "ACGTTT", "GACGT", 1, [DEL, DEL, SUB]) == "1I4M2D"
