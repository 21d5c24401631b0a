"""Randomised GPU sweep of the ends-free (kind "ef") and gap-affine 2-piece (kind "ap") paths: one round aligns one
seeded batch (tests/newpath_cases.py) through the public API and checks every pair against the CPU references:
  * the score equals the exact DP (`gotoh_span`, `gotoh2p`);
  * the CIGAR aligns both sequences at that cost (`wfagpu_check_result_span`, `wfagpu_check_result_affine2p`);
  * the CIGAR text equals the CPU model of the kernel path (`endsfree_model`, `affine2p_model`) byte for byte;
  * run_stats()["failed_pairs"] == 0;
and, on the GPU results alone:
  * ends-free: pattern and text swapped with (pb, pe) <-> (tb, te) give the same scores;
  * 2-piece: the pieces swapped give the same scores; identical pieces print the bytes of plain `wfagpu_align`; a
    dominated second piece (o2 >= o1, e2 >= e1) gives the scores of plain `wfagpu_align` with (x, o1, e1).

Round r of seed S uses the cases of seed S + r, so `<tool> 1 <S + r>` re-runs that round alone.
NEWPATH_REF_CACHE=<dir> keeps the CPU references per round seed there (the same seed under another kernel variant
reuses them); NEWPATH_BATCH=<n> overrides the drawn batch size (small batches for two workers per GPU)."""
import json
import os
import sys
import time
from multiprocessing import Pool

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for _d in ("oracle", os.path.join("wfa-gpu_b200", "python"), "tests"):
    if os.path.join(ROOT, _d) not in sys.path:
        sys.path.insert(0, os.path.join(ROOT, _d))

import newpath_cases as cases  # noqa: E402

_oracle = None


def reference(job):
    """(kind, p, t, pen, span) -> (DP score, model finished, model score, model CIGAR); runs in a pool worker."""
    global _oracle
    kind, p, t, pen, span = job
    if kind == "ef":
        import endsfree_model
        from endsfree_ref import gotoh_span
        from oracle import Oracle
        if _oracle is None:
            _oracle = Oracle()
        s = gotoh_span(p, t, *pen, span)
        m = endsfree_model.align(_oracle, p, t, *pen, span, max_steps=s + 8)
    else:
        import affine2p_model
        from affine2p_ref import gotoh2p
        s = gotoh2p(p, t, *pen)
        m = affine2p_model.align(p, t, *pen, max_steps=s + 8)
    return s, bool(m["finished"]), int(m["distance"]), m["cigar"]


def gpu_align(pairs, pen, cigar, budget, batch, span=None, affine2p=None):
    """-> (scores, cigars or None, failed_pairs) of one call of the public API."""
    import wfagpu
    a = wfagpu.Aligner()
    for p, t in pairs:
        assert a.add_sequences(p, t)
    assert a.initialize_parameters(*pen[:3])
    a.options.compute_cigar = cigar
    a.options.max_error = budget
    a.set_batch_size(batch)
    a.align(ends_free=span, affine2p=affine2p)
    out = (a.errors(), a.cigars() if cigar else None, a.run_stats()["failed_pairs"])
    a.destroy()
    return out


def _references(pool, kind, seed, rd):
    path = os.environ.get("NEWPATH_REF_CACHE")
    f = os.path.join(path, "%s_%d.json" % (kind, seed)) if path else None
    if f and os.path.exists(f):
        with open(f) as fh:
            return [tuple(r) for r in json.load(fh)]
    span = rd.get("span")
    jobs = [(kind, p, t, rd["pen"], span) for p, t in rd["pairs"]]
    # longest first: the pool's tail is not one 3 kbp pair
    order = sorted(range(len(jobs)), key=lambda i: -len(jobs[i][1]) - len(jobs[i][2]))
    got = pool.map(reference, [jobs[i] for i in order], chunksize=1)
    refs = [None] * len(jobs)
    for i, r in zip(order, got):
        refs[i] = r
    if f:
        os.makedirs(path, exist_ok=True)
        with open(f + ".tmp", "w") as fh:
            json.dump(refs, fh)
        os.replace(f + ".tmp", f)
    return refs


def check_round(pool, kind, seed):
    """Align round `seed` on the GPU and check it.  -> (pairs, list of mismatch descriptions)."""
    import wfagpu
    from affine2p_ref import cost_ok
    from endsfree_ref import span_cost_ok
    lib = wfagpu.load()
    rd = cases.ef_round(seed) if kind == "ef" else cases.ap_round(seed)
    pairs, pen, budget, cigar = rd["pairs"], rd["pen"], rd["budget"], rd["cigar"]
    span = rd.get("span")
    batch = int(os.environ.get("NEWPATH_BATCH", "0")) or rd["batch"]
    where = "seed=%d pen=%s span=%s budget=%d batch=%d cigar=%d" % (seed, pen, span, budget, batch, cigar)
    bad = []
    if kind == "ef":
        scores, cigars, failed = gpu_align(pairs, pen, cigar, budget, batch, span=span)
    else:
        scores, cigars, failed = gpu_align(pairs, pen, cigar, budget, batch, affine2p=pen)
    if failed:
        bad.append("%s: failed_pairs=%d" % (where, failed))
    refs = _references(pool, kind, seed, rd)
    for i, ((p, t), (s, fin, ms, mc)) in enumerate(zip(pairs, refs)):
        what = "%s pair=%d plen=%d tlen=%d" % (where, i, len(p), len(t))
        if not fin or ms != s:
            bad.append("%s: CPU model %s/%d != DP %d" % (what, fin, ms, s))
        if scores[i] != s:
            bad.append("%s: score %d != DP %d" % (what, scores[i], s))
            continue
        if cigar:
            ok = (span_cost_ok(lib, p, t, *pen, span, s, cigars[i]) if kind == "ef"
                  else cost_ok(lib, p, t, pen, s, cigars[i]))
            if not ok:
                bad.append("%s: CIGAR %s... does not cost %d" % (what, cigars[i][:60], s))
            if cigars[i] != mc:
                bad.append("%s: CIGAR %s... != model %s..." % (what, cigars[i][:60], mc[:60]))
    # metamorphic checks: GPU against GPU
    if kind == "ef":
        pb, pe, tb, te = span
        sw, _, _ = gpu_align([(t, p) for p, t in pairs], pen, False, budget, batch, span=(tb, te, pb, pe))
        for i, (a, b) in enumerate(zip(scores, sw)):
            if a != b:
                bad.append("%s pair=%d: swapped pattern / text score %d != %d" % (where, i, b, a))
    else:
        x, o1, e1, o2, e2 = pen
        sw, _, _ = gpu_align(pairs, (x, o2, e2), False, budget, batch, affine2p=(x, o2, e2, o1, e1))
        for i, (a, b) in enumerate(zip(scores, sw)):
            if a != b:
                bad.append("%s pair=%d: swapped pieces score %d != %d" % (where, i, b, a))
        if (o1, e1) == (o2, e2):
            one = gpu_align(pairs, pen, cigar, budget, batch)
            if one[:2] != (scores, cigars):
                bad.append("%s: identical pieces differ from the single-piece bytes" % where)
        elif cases.dominated(pen):
            one, _, _ = gpu_align(pairs, pen, False, budget, batch)
            for i, (a, b) in enumerate(zip(scores, one)):
                if a != b:
                    bad.append("%s pair=%d: dominated piece 2: score %d != single-piece %d" % (where, i, a, b))
    return len(pairs), bad


def main(kind, argv):
    """usage: <tool> <seconds|rounds> [seed]: `60s` runs rounds for 60 seconds, `12` runs 12 rounds."""
    if len(argv) < 2:
        print(__doc__)
        return 2
    limit = argv[1]
    seconds = float(limit[:-1]) if limit.endswith("s") else None
    rounds_max = None if seconds is not None else int(limit)
    seed0 = int(argv[2]) if len(argv) > 2 else 12345
    # the pool forks before this process opens a CUDA context
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        t0 = time.time()
        rounds = pairs_total = bad_total = 0
        while (rounds < rounds_max) if rounds_max is not None else (time.time() - t0 < seconds):
            n, bad = check_round(pool, kind, seed0 + rounds)
            rounds += 1
            pairs_total += n
            bad_total += len(bad)
            for b in bad[:5]:
                print("MISMATCH", b, flush=True)
    env = {k: v for k, v in os.environ.items() if k.startswith("WFAGPU_")}
    print(f"rounds={rounds} pairs={pairs_total} mismatches={bad_total} seed={seed0} env={env}")
    return 1 if bad_total else 0
