"""Gap-affine 2-piece on the host: the row DP against a cell-by-cell statement and the single-piece DP, the CIGAR
validator wfagpu_check_result_affine2p on hand cases, and the step table against a restatement of its rules."""
import numpy as np
import pytest

import affine2p_model
from affine2p_ref import cost_ok, gotoh2p, gotoh2p_cells, indel_pairs, step_table
from endsfree_ref import gotoh_span, mutate, rand_seq

PENALTIES = [(4, 4, 2, 24, 1), (19, 39, 3, 81, 1), (2, 3, 1, 3, 1), (4, 6, 4, 20, 2), (2, 0, 2, 6, 1),
             (4, 24, 1, 4, 2), (1, 0, 1, 5, 1), (3, 2, 3, 12, 1), (5, 1, 5, 0, 3)]
TINY = [("", ""), ("", "ACG"), ("ACG", ""), ("A", "C"), ("A", "A"), ("G", "ACGTA"), ("ACGTA", "G"), ("AC", "ACAC")]


def small_pairs(seed):
    rng = np.random.default_rng(seed)
    out = []
    for n in (12, 25, 40):
        t = rand_seq(rng, n)
        p = mutate(rng, t, 0.15)
        at = int(rng.integers(0, len(p) + 1))
        out.append((p[:at] + rand_seq(rng, 9) + p[at:], t))
        out.append((p[:at] + p[at + 9:], t))
    return out + TINY


@pytest.mark.parametrize("pen", PENALTIES)
def test_row_dp_equals_cells(pen):
    for p, t in small_pairs(sum(pen)):
        assert gotoh2p(p, t, *pen) == gotoh2p_cells(p, t, *pen), (p, t)


@pytest.mark.parametrize("pen", [(2, 3, 1), (4, 6, 2), (1, 0, 1), (19, 39, 3)])
def test_identical_pieces_equal_single_piece(pen):
    x, o, e = pen
    for p, t in small_pairs(7) + indel_pairs(3, [(4, 300, 0.05, 50, 80)]):
        assert gotoh2p(p, t, x, o, e, o, e) == gotoh_span(p, t, x, o, e, (0, 0, 0, 0)), (p, t)


@pytest.mark.parametrize("pen", PENALTIES)
def test_swapped_pieces_give_equal_scores(pen):
    x, o1, e1, o2, e2 = pen
    for p, t in small_pairs(11) + indel_pairs(5, [(2, 300, 0.05, 50, 80)]):
        assert gotoh2p(p, t, x, o1, e1, o2, e2) == gotoh2p(p, t, x, o2, e2, o1, e1), (p, t)


def test_two_pieces_beat_both_single_pieces_on_indel_pairs():
    # a pair with short indels and one long indel needs both pieces in one alignment
    x, o1, e1, o2, e2 = pen = (4, 4, 2, 24, 1)
    pairs = indel_pairs(0xA2, [(12, 1000, 0.05, 50, 500)])
    strict = 0
    for p, t in pairs:
        s2 = gotoh2p(p, t, *pen)
        s1a = gotoh_span(p, t, x, o1, e1, (0, 0, 0, 0))
        s1b = gotoh_span(p, t, x, o2, e2, (0, 0, 0, 0))
        assert s2 <= min(s1a, s1b), (s2, s1a, s1b)
        strict += s2 < min(s1a, s1b)
    assert strict > len(pairs) // 2, (strict, len(pairs))


def test_validator_hand_cases(lib):
    pen = (4, 4, 2, 24, 1)                       # a gap of L costs min(4 + 2L, 24 + L): the crossover is L = 20
    t = "ACGT" * 10                              # 40 bases
    # piece 1 cheaper: a 3-base insertion costs 4 + 6 = 10
    assert cost_ok(lib, t[:20] + "TTT" + t[20:], t, pen, 10, "20M3D20M")
    assert cost_ok(lib, t[:20] + t[23:], t, pen, 10, "20M3I17M")
    # piece 2 cheaper: a 30-base deletion costs min(64, 54) = 54
    assert cost_ok(lib, t[:5] + t[35:], t, pen, 54, "5M30I5M")
    # the crossover: 20 bases cost 44 under either piece
    assert cost_ok(lib, t[:10] + t[30:], t, pen, 44, "10M20I10M")
    assert cost_ok(lib, t[:10] + t[29:], t, pen, 4 + 2 * 19, "10M19I11M")
    assert cost_ok(lib, t[:10] + t[31:], t, pen, 24 + 21, "10M21I9M")
    # mismatches cost x
    assert cost_ok(lib, "AAGT", "ACGT", pen, 4, "1M1X2M")
    # a wrong score, a CIGAR that does not match the sequences, one that does not consume them, malformed text
    assert not cost_ok(lib, t[:5] + t[35:], t, pen, 64, "5M30I5M")
    assert not cost_ok(lib, "AAGT", "ACGT", pen, 0, "4M")
    assert not cost_ok(lib, "ACGT", "ACGT", pen, 0, "3M")
    assert not cost_ok(lib, "ACGT", "ACGT", pen, 0, "4Q")
    # invalid penalties
    assert not cost_ok(lib, "ACGT", "ACGT", (4, 4, 2, 24, 0), 0, "4M")


def _check_table(lib, pen, max_steps, max_dist):
    d_end, tab, _ = step_table(lib, pen, max_steps, max_dist)
    ns, kinds = affine2p_model.steps(*pen, max_steps, max_dist)
    assert d_end == len(ns), (pen, max_steps, d_end, len(ns))
    assert [(n, k) for _, n, k in tab] == list(zip(ns.tolist(), kinds.tolist())), pen
    return d_end


@pytest.mark.parametrize("pen", PENALTIES)
def test_step_table_follows_the_rules(lib, pen):
    # unlimited by the budget, then cut off by it
    assert _check_table(lib, pen, 10 ** 6, 600) == 600
    d_cut = _check_table(lib, pen, 40, 10 ** 5)
    assert d_cut < 10 ** 5
    _, tab, _ = step_table(lib, pen, 40, 10 ** 5)
    assert sum(k == 2 for _, _, k in tab) == 40 - 2            # the step count starts at 1 and stops at max_steps - 1


@pytest.mark.parametrize("pen", [(2, 3, 1), (4, 6, 2), (19, 39, 3), (1, 0, 1), (4, 4, 2)])
def test_identical_pieces_give_the_single_piece_table(lib, pen):
    import ctypes as C
    import wfagpu
    x, o, e = pen
    for max_steps, max_dist in ((10 ** 6, 500), (30, 10 ** 5)):
        d2, tab2, u2 = step_table(lib, (x, o, e, o, e), max_steps, max_dist)
        tab1 = (wfagpu.Step * (max_dist + 1))()
        u1 = C.c_uint64()
        d1 = lib.wfagpu_build_step_table(x, o, e, max_steps, max_dist, 0, tab1, C.byref(u1))
        assert (d1, u1.value) == (d2, u2)
        assert [(tab1[d].row_off, tab1[d].n, tab1[d].kind) for d in range(d1)] == tab2


def test_step_table_rejects_invalid_penalties(lib):
    for pen in ((0, 4, 2, 24, 1), (4, 4, 0, 24, 1), (4, 4, 2, 24, 0), (4, -1, 2, 24, 1), (4, 4, 2, -1, 1)):
        assert step_table(lib, pen, 100, 100)[0] == -1, pen
