"""Seeded cases for the randomised checks of the ends-free and gap-affine 2-piece paths: penalty draws (named regimes
plus random ones), pair shapes, ends-free spans, budgets and batch sizes.  Everything comes from one integer seed, so a
round is reproduced from its seed alone (tools/stress_endsfree.py, tools/stress_affine2p.py,
tests/test_newpath_models_random.py).

Every drawn pair's optimal score stays far below the 60 000-step cap: unrelated pairs (reversed, all-mismatch, random)
are at most 600 bases and mutated pairs have at most 15 % error, so a round may assert that no pair failed."""
import numpy as np

from endsfree_ref import mutate, rand_seq, window_pairs

# every single-piece set of tests/test_endsfree_model.py, plus a mismatch that sets the ring depth and o = 0 with e = 2
EF_REGIMES = [(2, 3, 1), (1, 0, 1), (2, 24, 9), (4, 6, 2), (5, 3, 2), (3, 1, 4), (2, 10, 5), (6, 4, 2), (9, 1, 1),
              (12, 0, 2)]
# every set of tests/test_affine2p_host.py::PENALTIES, a dominated piece 2 (o2 >= o1, e2 >= e1), equal extensions with
# different opens, the mismatch deepest, a very deep piece-2 ring; then each of them with its pieces swapped
_AP = [(4, 4, 2, 24, 1), (19, 39, 3, 81, 1), (2, 3, 1, 3, 1), (4, 6, 4, 20, 2), (2, 0, 2, 6, 1), (4, 24, 1, 4, 2),
       (1, 0, 1, 5, 1), (3, 2, 3, 12, 1), (5, 1, 5, 0, 3),
       (2, 3, 1, 5, 2), (3, 2, 2, 10, 2), (12, 2, 2, 6, 1), (4, 4, 2, 120, 1)]
AP_REGIMES = _AP + [(x, o2, e2, o1, e1) for x, o1, e1, o2, e2 in _AP if (o1, e1) != (o2, e2)]
BUDGETS = list(range(1, 21)) + [100, 400, 2000]
# packed-word edges (8 bases per 16-bit word, 16 per 32-bit word) and the warp tier's max_len of 1024
EDGE_LENS = [7, 8, 9, 15, 16, 17, 31, 32, 33, 1024, 1025]
BUCKETS = [(0, 40), (40, 400), (400, 1500), (1500, 3000)]
BIG = 10 ** 6


def crossover(pen):
    """The gap length L* = (o2 - o1) / (e1 - e2) where the cheaper piece flips, or None (parallel pieces, or L* < 1)."""
    x, o1, e1, o2, e2 = pen
    if e1 == e2 or (o2 - o1) * (e1 - e2) <= 0:
        return None
    return (o2 - o1) / (e1 - e2)


def dominated(pen):
    x, o1, e1, o2, e2 = pen
    return o2 >= o1 and e2 >= e1


def ef_penalty(rng):
    if rng.random() < 0.5:
        return EF_REGIMES[int(rng.integers(len(EF_REGIMES)))]
    return int(rng.integers(1, 13)), int(rng.integers(0, 31)), int(rng.integers(1, 9))


def ap_penalty(rng):
    if rng.random() < 0.5:
        return AP_REGIMES[int(rng.integers(len(AP_REGIMES)))]
    return (int(rng.integers(1, 13)), int(rng.integers(0, 31)), int(rng.integers(1, 9)), int(rng.integers(0, 91)),
            int(rng.integers(1, 9)))


def _length(rng):
    if rng.random() < 0.25:
        return EDGE_LENS[int(rng.integers(len(EDGE_LENS)))]
    lo, hi = BUCKETS[int(rng.integers(len(BUCKETS)))]
    return int(rng.integers(max(lo, 1), hi + 1))


def indel_pair(rng, length, err, L):
    """The text mutated at `err` with one insertion or deletion (a coin flip) of L bases at a random place."""
    t = rand_seq(rng, length)
    p = mutate(rng, t, err)
    at = int(rng.integers(0, max(1, len(p) - L)))
    if rng.random() < 0.5:
        return p[:at] + rand_seq(rng, L) + p[at:], t
    return p[:at] + p[at + L:], t


def pairs(rng, pen=None, scale=1.0):
    """One round's pairs: flanked windows and dovetails, one long indel (at L* - 1, L*, L* + 1 when `pen` is a 2-piece
    set with a crossover), and the structured shapes: empty and one-base sequences, homopolymers, identical, reversed,
    all-mismatch and tie pairs, 'N' at an end or inside."""
    out = []
    for _ in range(int(rng.integers(1, 3))):
        L = _length(rng)
        n = max(1, min(24, int(scale * 6000 // max(L, 60))))
        flank = int(rng.integers(0, max(2, L // 4)))
        out += window_pairs(int(rng.integers(1 << 31)), [(n, L, flank, float(rng.choice([0.0, 0.02, 0.05, 0.15])))])
    Ls = [int(rng.integers(1, 300))]
    if pen is not None and len(pen) == 5 and crossover(pen) is not None:
        c = crossover(pen)
        Ls = sorted({int(c) - 1, int(c), int(np.ceil(c)), int(np.ceil(c)) + 1})
    for L in Ls:
        if L >= 1:
            out.append(indel_pair(rng, int(rng.integers(L + 20, L + 800)), float(rng.choice([0.0, 0.03])), L))
    base = rand_seq(rng, int(rng.integers(1, 600)))
    h = int(rng.integers(1, 300))
    out += [("", ""), ("", base[:int(rng.integers(1, 40))]), (base[:int(rng.integers(1, 40))], ""), ("A", "C"), ("G", "G"),
            (base, base), (base, base[::-1]), ("A" * h, "A" * int(rng.integers(1, 300))),
            ("AC", "ACAC"), ("ACAC", "AC"), ("ACGT" * int(rng.integers(1, 8)), "ACGT" * int(rng.integers(1, 12)))]
    m = int(rng.integers(1, 300))
    out.append(("A" * m, "C" * int(rng.integers(max(1, m - 5), m + 6))))           # all mismatch
    for _ in range(2):
        p, t = out[int(rng.integers(len(out)))]
        out.append(_put_n(rng, p, t))
    return out


def _put_n(rng, p, t):
    """'N' at the first base, the last base or somewhere inside one of the two sequences (the byte-compare kernel)."""
    if not p and not t:
        return p, t
    on_p = bool(p) and (not t or rng.random() < 0.5)
    s = p if on_p else t
    where = int(rng.integers(3))
    i = 0 if where == 0 else (len(s) - 1 if where == 1 else int(rng.integers(len(s))))
    s = s[:i] + "N" + s[i + 1:]
    return (s, t) if on_p else (p, s)


def span(rng, pairs_):
    """Each side is 0, a random value, the length (or one less) of a pair's pattern or text, or 10**6 (fully free)."""
    p, t = pairs_[int(rng.integers(len(pairs_)))]
    pl, tl = len(p), len(t)

    def side():
        return [0, int(rng.integers(0, 200)), pl, max(0, pl - 1), tl, max(0, tl - 1), BIG][int(rng.integers(7))]

    return side(), side(), side(), side()


def budget(rng):
    return BUDGETS[int(rng.integers(len(BUDGETS)))]


def batch_size(rng, n):
    return [n, max(1, n // 3), 97][int(rng.integers(3))]


def ef_round(seed, scale=1.0):
    """-> dict(pen, span, pairs, budget, batch, cigar) of one ends-free round."""
    rng = np.random.default_rng(seed)
    pen = ef_penalty(rng)
    ps = pairs(rng, None, scale)
    return dict(pen=pen, span=span(rng, ps), pairs=ps, budget=budget(rng), batch=batch_size(rng, len(ps)),
                cigar=bool(rng.random() < 0.85))


def ap_round(seed, scale=1.0):
    """-> dict(pen, pairs, budget, batch, cigar) of one 2-piece round."""
    rng = np.random.default_rng(seed)
    pen = ap_penalty(rng)
    ps = pairs(rng, pen, scale)
    return dict(pen=pen, pairs=ps, budget=budget(rng), batch=batch_size(rng, len(ps)), cigar=bool(rng.random() < 0.85))
