"""Shared helpers for the parity tests."""
import wfagpu


def synth_aligner(specs, seed=0xB2000000):
    """specs: list of (n, length, err_lo, err_hi). Returns a filled Aligner."""
    a = wfagpu.Aligner()
    for i, (n, length, lo, hi) in enumerate(specs):
        a.add_synthetic(seed + i, n, length, lo, hi)
    return a


def non_acgt_pairs():
    """The pairs of test_gpu_parity.py::test_non_acgt_pairs_match_cpu_wfa_scores: every third one with 1-6 'N' in
    each sequence.  -> (pairs, indices of the pairs that were given an 'N')"""
    import random
    rng = random.Random(77)
    a = synth_aligner([(300, 800, 0.02, 0.10), (40, 3000, 0.05, 0.05)], 0xB2000077)
    pairs, dirty = [], []
    for i in range(a.num_pairs):
        p, t = a.pair(i)
        if i % 3 == 0:
            p, t = list(p), list(t)
            for s in (p, t):
                for _ in range(rng.randint(1, 6)):
                    s[rng.randrange(len(s))] = "N"
            p, t = "".join(p), "".join(t)
            dirty.append(i)
        pairs.append((p, t))
    return pairs, dirty


def cpu_wfa_scores(name):
    """Stored exact gap-affine scores of a test workload (tests/golden/cpu_wfa_scores.json, made by
    tests/golden/make_cpu_wfa_scores.py)."""
    import json
    import os
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "cpu_wfa_scores.json")) as f:
        return json.load(f)[name]


def assert_cpu_wfa_scores(name, got, lo=0):
    """Scores `got` of pairs [lo, lo + len(got)) of workload `name` equal the stored exact scores: element by element
    where the scores are stored, otherwise on the stored sample and through the digest of the whole list."""
    import hashlib
    import numpy as np
    g = cpu_wfa_scores(name)
    got = [int(s) for s in got]
    if "scores" in g:
        assert got == g["scores"][lo:lo + len(got)]
        return
    assert lo == 0 and len(got) == g["n"]
    k = g["every"]
    assert got[::k] == g["sample"]
    assert hashlib.sha256(np.asarray(got, dtype="<i4").tobytes()).hexdigest() == g["sha256"]


def pairs_of(a, idx=None):
    idx = range(a.num_pairs) if idx is None else idx
    return [a.pair(i) for i in idx]


def check_against_oracle(oracle, a, x, o, e, max_steps, cigar, sample=None, big_budget=None):
    """Compare every (or sampled) pair of a finished Aligner run with the oracle.

    The GPU library re-dispatches over-budget pairs, so its final answer must equal
    the oracle run with a budget large enough to finish (big_budget)."""
    idx = list(range(a.num_pairs)) if sample is None else sample
    bad = []
    for i in idx:
        p, t = a.pair(i)
        r = oracle.align(p, t, x, o, e, max_steps, cigar=cigar)
        if not r["finished"]:
            r = oracle.align(p, t, x, o, e, big_budget or 8 * max_steps + 64, cigar=cigar)
            assert r["finished"]
        if a.error(i) != r["distance"]:
            bad.append((i, "score", a.error(i), r["distance"]))
        elif cigar and a.cigar(i) != r["cigar"]:
            bad.append((i, "cigar", a.cigar(i)[:80], r["cigar"][:80]))
    return bad
