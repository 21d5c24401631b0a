"""The ends-free and 2-piece paths on the GPU beyond their fixed batches: the randomised sweeps of
tools/stress_endsfree.py and tools/stress_affine2p.py at a fixed seed and round count under every launch-shape switch,
and a deterministic grid of edge shapes (int16 offset limit, tier boundaries, clamp-edge spans, crossover gap lengths,
ties in repeats, a short pair among long ones).  Every pair: score == the exact DP, CIGAR valid at that cost, CIGAR == the CPU model's
bytes.  A case that claims a tier shows it: the launch shape of its first pass (WFAGPU_VERBOSE) is checked."""
import os
import re
import subprocess
import sys
from multiprocessing import Pool

import numpy as np
import pytest

from affine2p_ref import cost_ok
from endsfree_ref import mutate, rand_seq, span_cost_ok, window_pairs
from newpath_cases import indel_pair
from newpath_sweep import gpu_align, reference

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ROUNDS, SEED = 4, 20261020

VARIANTS = {
    "base": {},
    "force_large": {"WFAGPU_FORCE_LARGE": "1"},
    "warp_kernel_on": {"WFAGPU_WARP_KERNEL": "1"},
    "warp_kernel_off": {"WFAGPU_WARP_KERNEL": "0"},
    "stages_1": {"WFAGPU_STAGES": "1"},
    "stages_2": {"WFAGPU_STAGES": "2"},
    "threads_64": {"WFAGPU_THREADS": "64"},
    "two_workers": {"WFAGPU_DEVICES": "0,0", "NEWPATH_BATCH": "16"},
    "host_cigar": {"WFAGPU_HOST_CIGAR": "1"},
}
EF_ONLY = {"no_bound": {"WFAGPU_NO_BOUND": "1"}, "force_bound": {"WFAGPU_FORCE_BOUND": "1"}}
SWEEPS = [("stress_endsfree.py", v) for v in sorted({**VARIANTS, **EF_ONLY})] + \
         [("stress_affine2p.py", v) for v in sorted(VARIANTS)]


@pytest.fixture(scope="module")
def ref_cache(tmp_path_factory):
    # the CPU references of a round depend on its seed only: the first variant computes them, the others reuse them
    return str(tmp_path_factory.mktemp("newpath_refs"))


@pytest.mark.parametrize("tool,variant", SWEEPS)
def test_short_sweep(ref_cache, tool, variant):
    env = dict(os.environ, NEWPATH_REF_CACHE=ref_cache, **{**VARIANTS, **EF_ONLY}[variant])
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "tools", tool), str(ROUNDS), str(SEED)], env=env,
                        capture_output=True, text=True, timeout=900)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]
    assert "rounds=%d " % ROUNDS in pr.stdout and "mismatches=0" in pr.stdout, pr.stdout[-3000:]


# ---- deterministic edge grid ----------------------------------------------------------------------------------------

def _check(lib, kind, pairs, pen, span=None, budget=400):
    """Align with CIGAR and check every pair against the DP, the validator and the model.  -> the GPU scores."""
    ap = pen if kind == "ap" else None
    scores, cigars, failed = gpu_align(pairs, pen, True, budget, len(pairs), span=span, affine2p=ap)
    assert failed == 0
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        order = sorted(range(len(pairs)), key=lambda i: -len(pairs[i][0]) - len(pairs[i][1]))
        got = pool.map(reference, [(kind, pairs[i][0], pairs[i][1], pen, span) for i in order], chunksize=1)
    refs = dict(zip(order, got))
    for i, (p, t) in enumerate(pairs):
        s, fin, ms, mc = refs[i]
        where = (pen, span, i, len(p), len(t))
        assert fin and ms == s, where + ("model", ms, s)
        assert scores[i] == s, where + (scores[i], s)
        ok = span_cost_ok(lib, p, t, *pen, span, s, cigars[i]) if kind == "ef" else cost_ok(lib, p, t, pen, s, cigars[i])
        assert ok, where + (cigars[i][:80],)
        assert cigars[i] == mc, where + (cigars[i][:80], mc[:80])
    return scores


def _first_pass(capfd, kind, pairs, pen, span=None, budget=400):
    """-> (n_cap, group threads, groups per CTA, tier) of the first wavefront pass of one score-only call."""
    os.environ["WFAGPU_VERBOSE"] = "1"
    try:
        capfd.readouterr()
        gpu_align(pairs, pen, False, budget, len(pairs), span=span, affine2p=pen if kind == "ap" else None)
        err = capfd.readouterr().err
    finally:
        del os.environ["WFAGPU_VERBOSE"]
    m = re.search(r"pass: .* n_cap=(\d+) .* group=(\d+) x(\d+) .* tier=(\S+)", err)
    assert m, err[-2000:]
    n_cap, threads, groups, tier = int(m.group(1)), int(m.group(2)), int(m.group(3)), m.group(4)
    return n_cap, threads, groups, ("large" if tier.startswith("global") else ("warp" if threads == 32 else "cta"))


def _boundary(capfd, kind, pen, make, lo, hi, tier_lo):
    """Smallest v in (lo, hi] whose batch make(v) = (pairs, span, budget) leaves `tier_lo` in its first pass."""
    def tier(v):
        pairs, span, budget = make(v)
        return _first_pass(capfd, kind, pairs, pen, span, budget)[3]
    assert tier(lo) == tier_lo and tier(hi) != tier_lo, (lo, hi, tier(lo), tier(hi))
    while hi - lo > 1:
        mid = (lo + hi) // 2
        if tier(mid) == tier_lo:
            lo = mid
        else:
            hi = mid
    return hi


def _both_sides(lib, capfd, kind, pen, make, lo, hi, tier_lo, tier_hi):
    """Find the switch, then show the tier of each side's first pass and check its results (pairs that outgrow that
    pass are re-dispatched, the results are checked all the same)."""
    v = _boundary(capfd, kind, pen, make, lo, hi, tier_lo)
    for w, tier in ((v - 1, tier_lo), (v, tier_hi)):
        pairs, span, budget = make(w)
        assert _first_pass(capfd, kind, pairs, pen, span, budget)[3] == tier, (w, tier)
        _check(lib, kind, pairs, pen, span, budget)
    return v


@pytest.mark.parametrize("n", [32767, 32768])
def test_int16_offset_limit(lib, n):
    # offsets reach the int16 limit on the shared-memory tier (32767) and go to the large tier one base later; the last
    # bases of the text sit in a gap, so an I cell there is one past the limit
    rng = np.random.default_rng(n)
    t = rand_seq(rng, n)
    core = mutate(rng, t[:n - 40], 0.002)
    pairs = [(t, t), (t[:n - 30], t), (t[:20000] + t[20040:], t), (core[:n], t), (t, t[:n - 25])]
    for span in ((0, 0, 150, 150), (5, 5, 0, 0)):
        _check(lib, "ef", pairs, (2, 3, 1), span, budget=2000)
    for pen in ((4, 4, 2, 24, 1), (12, 2, 2, 6, 1)):
        _check(lib, "ap", pairs, pen, budget=2000)


def test_spans_at_the_clamp_edges(lib):
    rng = np.random.default_rng(0xC1A)
    pl, tl = 300, 360
    pairs = []
    for err in (0.0, 0.05, 0.2):
        t = rand_seq(rng, tl)
        pairs.append((mutate(rng, t[30:330], err)[:pl].ljust(pl, "A"), t))
    pairs += [(rand_seq(rng, pl), rand_seq(rng, tl)), ("A" * pl, "C" * tl)]
    edges = []
    for side in range(4):
        full = pl if side < 2 else tl
        for v in (full - 1, full, full + 1):
            s = [0, 0, 0, 0]
            s[side] = v
            edges.append(tuple(s))
    for pen in ((2, 3, 1), (9, 1, 1), (2, 24, 9)):
        for span in edges:
            _check(lib, "ef", pairs, pen, span)
        # the whole pattern free together with the whole text at one end: nothing to align
        for span in ((pl, pl, tl, tl), (pl, 0, 0, tl), (0, pl, tl, 0), (10 ** 6,) * 4):
            assert _check(lib, "ef", pairs, pen, span) == [0] * len(pairs), span


@pytest.mark.parametrize("pen", [(4, 4, 2, 24, 1), (4, 6, 4, 20, 2), (3, 2, 3, 12, 1), (19, 39, 3, 81, 1),
                                 (4, 24, 1, 4, 2), (4, 20, 2, 6, 4)])
def test_gaps_at_the_crossover_length(lib, pen):
    x, o1, e1, o2, e2 = pen
    c = (o2 - o1) // (e1 - e2)
    rng = np.random.default_rng(sum(pen))
    pairs = [indel_pair(rng, length, err, L) for L in (c - 1, c, c + 1) for length in (150, 1000)
             for err in (0.0, 0.0, 0.02)]
    _check(lib, "ap", pairs, pen)


def _repeat_pairs(rng, n, length, max_gap):
    """Texts of tandem repeats and homopolymers, patterns with a few indels of 1 .. max_gap bases inside them: many
    gap placements and many pieces reach the same cell at the same score, so every tie-break of the traceback decides
    the CIGAR text."""
    out = []
    for _ in range(n):
        t = ""
        while len(t) < length:
            t += rand_seq(rng, int(rng.integers(1, 4))) * int(rng.integers(3, 30))
        t = t[:length]
        p = t
        for _ in range(int(rng.integers(2, 7))):
            L, at = int(rng.integers(1, max_gap + 1)), int(rng.integers(0, max(1, len(p))))
            p = p[:at] + p[at:at + L] + p[at:] if rng.random() < 0.5 else p[:at] + p[at + L:]
        out.append((mutate(rng, p, 0.01), t))
    return out


@pytest.mark.parametrize("pen", [(4, 24, 1, 4, 2), (4, 4, 2, 24, 1), (5, 1, 5, 0, 3), (5, 0, 3, 1, 5), (3, 12, 1, 2, 3),
                                 (4, 20, 2, 6, 4), (2, 3, 1, 3, 1)])
def test_ties_in_repeats(lib, pen):
    x, o1, e1, o2, e2 = pen
    c = (o2 - o1) // (e1 - e2) if e1 != e2 else 8
    rng = np.random.default_rng(sum(pen) + 7)
    _check(lib, "ap", _repeat_pairs(rng, 16, 300, max(4, c + 3)) + _repeat_pairs(rng, 6, 1500, max(4, c + 3)), pen)


@pytest.mark.parametrize("pen", [(4, 6, 4, 20, 2), (6, 6, 4, 9, 2), (2, 6, 1, 0, 2), (4, 20, 2, 6, 4)])
def test_equal_gaps_of_both_pieces(lib, pen):
    # short repeat pairs under pieces with a common factor: now and then a piece-1 gap and a piece-2 gap of different
    # lengths reach the same cell at the same score, and only M's "D1 before D2" (or "I1 before I2") picks the CIGAR
    # (about one pair in a hundred; these seeds hold such pairs for every set)
    rng = np.random.default_rng(sum(pen) + 11)
    _check(lib, "ap", _repeat_pairs(rng, 150, 60, 12) + _repeat_pairs(rng, 30, 300, 12), pen)


def test_ends_free_ties_in_repeats(lib):
    rng = np.random.default_rng(0x7E5)
    pairs = _repeat_pairs(rng, 16, 300, 6)
    for pen in ((2, 3, 1), (4, 6, 2), (9, 1, 1)):
        for span in ((0, 0, 20, 20), (20, 20, 0, 0), (0, 15, 15, 0), (7, 0, 0, 7)):
            _check(lib, "ef", pairs, pen, span)


def test_short_pair_among_long_pairs_under_a_wide_span(lib):
    # the batch's start row is 2000 diagonals wide: the 30-base pair computes (NULL) cells out to it
    pairs = window_pairs(0x5A5A, [(6, 5000, 300, 0.03)])
    rng = np.random.default_rng(30)
    t = rand_seq(rng, 30)
    pairs[3:3] = [(mutate(rng, t, 0.1), t), (t, rand_seq(rng, 12) + t + rand_seq(rng, 9))]
    for span in ((0, 0, 2000, 2000), (2000, 2000, 0, 0), (2000, 0, 0, 2000)):
        _check(lib, "ef", pairs, (2, 3, 1), span, budget=2000)


def _window_batch(rng, core, flank, err, n=6):
    pairs = []
    for _ in range(n):
        c = rand_seq(rng, core)
        pairs.append((mutate(rng, c, err), rand_seq(rng, flank) + c + rand_seq(rng, flank)))
    return pairs


def test_warp_tier_boundary(lib, capfd):
    # 1024-base texts: the start row's width W decides warp per pair or CTA per pair; both sides of the switch, then one
    # text base more (max_len 1025) leaves the warp tier at the same W
    rng = np.random.default_rng(0x3A4)
    pairs = _window_batch(rng, 824, 100, 0.004)
    assert max(len(t) for _, t in pairs) == 1024 and max(len(p) for p, _ in pairs) <= 1024
    pen = (2, 3, 1)
    w = _both_sides(lib, capfd, "ef", pen, lambda v: (pairs, (0, 0, v, v), 40), 1, 1000, "warp", "cta")
    longer = pairs + [(pairs[0][0], pairs[0][1] + "A")]
    assert _first_pass(capfd, "ef", longer, pen, (0, 0, w - 1, w - 1), 40)[3] == "cta"
    _check(lib, "ef", longer, pen, (0, 0, w - 1, w - 1), 40)
    # 2-piece: the budget decides
    gpairs = [(mutate(rng, t, 0.004)[:1024], t) for _, t in pairs]
    _both_sides(lib, capfd, "ap", (4, 4, 2, 24, 1), lambda v: (gpairs, None, v), 1, 2000, "warp", "cta")


def test_shared_memory_tier_boundary(lib, capfd):
    # rings that just fit one CTA's shared memory, and one step wider: the large tier with rings in global memory
    rng = np.random.default_rng(0x5BE)
    pairs = _window_batch(rng, 1500, 14000, 0.01, n=3)
    _both_sides(lib, capfd, "ef", (2, 3, 1), lambda v: (pairs, (0, 0, v, v), 400), 1, 14000, "cta", "large")
    # 2-piece with a deep piece-2 ring: the budget decides
    gpairs = [indel_pair(rng, 3000, 0.002, L) for L in (20, 60)]
    _both_sides(lib, capfd, "ap", (4, 4, 2, 120, 1), lambda v: (gpairs, None, v), 1, 20000, "cta", "large")
