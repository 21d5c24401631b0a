"""The CPU models of the ends-free and 2-piece kernel paths (tests/endsfree_model.py, tests/affine2p_model.py) against
their exact DPs on seeded random draws of penalties, spans and pairs (tests/newpath_cases.py), and every model CIGAR
through the library's validator at the model's score.  The GPU sweeps take their CIGAR bytes from these models, so the
models must hold across the whole drawn space, not only on the named penalty sets."""
import os
from multiprocessing import Pool

import pytest

import newpath_cases as cases
from affine2p_ref import cost_ok
from endsfree_ref import span_cost_ok
from newpath_sweep import reference

ROUNDS = 40


def _jobs(kind):
    out = []
    for seed in range(ROUNDS):
        rd = cases.ef_round(0x5EED + seed, scale=0.3) if kind == "ef" else cases.ap_round(0x5EED + seed, scale=0.3)
        out += [(kind, p, t, rd["pen"], rd.get("span")) for p, t in rd["pairs"]]
    return out


@pytest.mark.parametrize("kind", ["ef", "ap"])
def test_models_equal_the_dps_on_random_draws(lib, kind):
    jobs = _jobs(kind)
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        refs = pool.map(reference, jobs, chunksize=4)
    pens = {j[3] for j in jobs}
    assert len(pens) >= ROUNDS // 2, pens                 # most rounds draw a different penalty set
    for (k, p, t, pen, span), (s, fin, ms, mc) in zip(jobs, refs):
        assert fin and ms == s, (pen, span, p, t, ms, s)
        ok = span_cost_ok(lib, p, t, *pen, span, s, mc) if kind == "ef" else cost_ok(lib, p, t, pen, s, mc)
        assert ok, (pen, span, p, t, s, mc)


def test_draws_reach_the_named_regimes():
    # the regimes the fixed GPU batches never reach: deep mismatch rings, gcd > 1, o2 = 0, dominated and deep pieces,
    # equal extensions, crossover indels, clamp-edge and fully free spans, the smallest budgets
    ef = [cases.ef_round(s) for s in range(400)]
    ap = [cases.ap_round(s) for s in range(400)]
    ef_pens = {r["pen"] for r in ef}
    ap_pens = {r["pen"] for r in ap}
    assert {(9, 1, 1), (12, 0, 2), (5, 3, 2), (3, 1, 4)} <= ef_pens
    assert {(4, 6, 4, 20, 2), (5, 1, 5, 0, 3), (2, 3, 1, 5, 2), (3, 2, 2, 10, 2), (4, 4, 2, 120, 1), (4, 120, 1, 4, 2)} <= ap_pens
    assert any(cases.dominated(p) and p[1:3] != p[3:] for p in ap_pens)
    spans = [r["span"] for r in ef]
    assert sum(cases.BIG in s for s in spans) > 100 and sum(0 in s for s in spans) > 100
    # a side equal to a pair's length or one less (the clamp edges)
    assert sum(any(v in (len(p), len(p) - 1, len(t), len(t) - 1) and v > 0 for v in r["span"] for p, t in r["pairs"])
               for r in ef) > 100
    lens = {len(p) for r in ef for p, _ in r["pairs"]} | {len(t) for r in ef for _, t in r["pairs"]}
    assert {0, 1} <= lens and max(lens) > 3000
    assert {r["budget"] for r in ef + ap} == set(cases.BUDGETS)
    xs = [r for r in ap if cases.crossover(r["pen"])]
    assert xs
    for r in xs[:20]:
        c = cases.crossover(r["pen"])
        gaps = {abs(len(p) - len(t)) for p, t in r["pairs"]}
        assert {int(c) - 1, int(c), int(c) + 1} & gaps, (r["pen"], c)
