"""The pairs of the byte-compare GPU tests and the premise they rest on, checked on the CPU: every original is flagged by
the packer and no twin is, a twin is its original under a one-to-one map onto ACGT, and the oracle's result (score,
CIGAR text, whether the band finishes) does not change under any of the 24 relabellings of ACGT."""
import itertools
import random

import pytest

import byte_compare_cases as bc

GROUPS = sorted(bc.GROUPS)


@pytest.fixture(scope="module")
def groups():
    return {g: bc.GROUPS[g]() for g in GROUPS}


@pytest.mark.parametrize("group", GROUPS)
def test_originals_are_flagged_and_twins_are_not(oracle, groups, group):
    pairs, twins = groups[group]
    assert len(pairs) == len(twins) and pairs
    for (p, t), tw in zip(pairs, twins):
        assert bc.pair_flagged(p, t), (p[:40], t[:40])
        if max(len(p), len(t)) < 1 << 15:
            # the packer's rule is the oracle's below 32768 bases (above, the oracle flags every sequence)
            assert oracle.has_N(p) or oracle.has_N(t)
        if tw is None:
            continue
        assert not bc.pair_flagged(*tw)
        if max(len(p), len(t)) < 1 << 15:
            assert not (oracle.has_N(tw[0]) or oracle.has_N(tw[1]))


@pytest.mark.parametrize("group", GROUPS)
def test_twins_are_one_to_one_relabellings_onto_acgt(groups, group):
    pairs, twins = groups[group]
    for (p, t), tw in zip(pairs, twins):
        if tw is None:
            assert len(set(p + t)) > 4
            continue
        tp, tt = tw
        assert set(tp + tt) <= set("ACGT")
        assert (len(tp), len(tt)) == (len(p), len(t))
        m = {}
        for a, b in zip(p + t, tp + tt):
            assert m.setdefault(a, b) == b, (a, b, m)
        assert len(set(m.values())) == len(m)


def test_the_groups_cover_the_edge_shapes(groups):
    pairs = groups["short"][0] + groups["mid"][0]
    have = set(pairs)
    assert {("N", "N"), ("", "N"), ("N", "")} <= have
    assert ("N" * 150, "N" * 150) in have and ("N" * 40, "N" * 47) in have
    assert any("N" not in p + t for p, t in pairs)                       # flagged through a YTGC-like group
    assert sum(tw is None for tw in groups["short"][1] + groups["mid"][1]) >= 5
    # an N at every position of a group, and in the final partial group
    for length in (9, 10, 11, 151):
        at = [s.index("N") for p, t in pairs for s in (p, t) if len(s) == length and s.count("N") == 1]
        assert {i % 4 for i in at} == {0, 1, 2, 3} and {0, length - 1} <= set(at)
        assert any(i >= length - length % 4 for i in at)
    assert max(len(t) for t in groups["long"][0][0]) >= 1 << 15


PENS = [(2, 3, 1), (4, 6, 2), (1, 0, 1), (5, 3, 2)]


def test_oracle_results_do_not_depend_on_the_labels(oracle, groups):
    rng = random.Random(24)
    twins = [tw for tw in groups["short"][1] + groups["mid"][1] if tw and len(tw[0]) + len(tw[1]) <= 2400]
    sample = rng.sample(twins, 12)
    for tp, tt in sample:
        pen = rng.choice(PENS)
        band, window = rng.choice([(10, 64), (25, 128)])
        ref = None
        for perm in itertools.permutations("ACGT"):
            m = dict(zip("ACGT", perm))
            p, t = "".join(m[c] for c in tp), "".join(m[c] for c in tt)
            got = [oracle.align(p, t, *pen, 4000), oracle.align(p, t, *pen, 300, band=band, window=window)]
            got = [(r["finished"], r["distance"], r["cigar"]) for r in got]
            ref = ref or got
            assert got == ref, (perm, pen, band, window)
        assert ref[0][0]
