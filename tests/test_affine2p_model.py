"""The CPU model of the gap-affine 2-piece kernel path (tests/affine2p_model.py) against the exact 2-piece DP, the
CIGAR validator and, with identical pieces, the single-piece oracle; and the exactness of the pruning with poisoned
pruned cells."""
import pytest

import affine2p_model as model
from affine2p_ref import cost_ok, gotoh2p, indel_pairs
from test_affine2p_host import PENALTIES, TINY, small_pairs


def pairs_for(pen):
    return small_pairs(0xA200 + sum(pen)) + indel_pairs(sum(pen), [(3, 200, 0.05, 50, 90)])


@pytest.mark.parametrize("pen", PENALTIES)
def test_model_equals_the_dp_and_its_cigars_cost_the_score(lib, pen):
    for p, t in pairs_for(pen):
        m = model.align(p, t, *pen)
        s = gotoh2p(p, t, *pen)
        assert m["finished"] and m["distance"] == s, (p, t, m["distance"], s)
        assert cost_ok(lib, p, t, pen, s, m["cigar"]), (p, t, m["cigar"])


@pytest.mark.parametrize("pen", [(2, 3, 1), (4, 6, 2), (1, 0, 1), (2, 24, 9)])
def test_identical_pieces_equal_the_oracle(oracle, pen):
    x, o, e = pen
    for p, t in small_pairs(sum(pen)) + indel_pairs(1, [(2, 200, 0.05, 50, 90)]):
        r = oracle.align(p, t, x, o, e, 4000)
        m = model.align(p, t, x, o, e, o, e)
        assert (m["distance"], m["cigar"]) == (r["distance"], r["cigar"]), (p, t)


@pytest.mark.parametrize("pen", [(4, 4, 2, 24, 1), (2, 0, 2, 6, 1), (4, 24, 1, 4, 2), (19, 39, 3, 81, 1)])
def test_pruning_is_exact(pen):
    # Cells with d + min(e1, e2) * |k - kt| > dmax are never computed; the model poisons them, so a read of one would
    # corrupt the result.  Every pair keeps its unpruned score and CIGAR down to dmax = s, and does not finish at s - 1.
    for p, t in indel_pairs(sum(pen) + 1, [(4, 150, 0.1, 20, 40)]) + TINY:
        full = model.align(p, t, *pen)
        s = full["distance"]
        for dmax in (s, s + 1, s + 3, int(1.2 * s) + 2, 3 * s + 7):
            m = model.align(p, t, *pen, dmax=dmax)
            assert (m["finished"], m["distance"], m["cigar"]) == (True, s, full["cigar"]), (p, t, dmax)
        if s > 0:
            assert not model.align(p, t, *pen, dmax=s - 1)["finished"], (p, t)
