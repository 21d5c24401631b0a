"""Ends-free (semi-global) ground truth for the tests: an exact gap-affine DP with free leading / trailing bases, the
pairs the tests align (flank + mutated core + flank), and the library's CIGAR helpers through ctypes.

span = (pattern_begin_free, pattern_end_free, text_begin_free, text_end_free), WFA2-lib's order; clamped per pair."""
import ctypes as C

import numpy as np

import wfagpu


def clamp(span, plen, tlen):
    pb, pe, tb, te = span
    return min(pb, plen), min(pe, plen), min(tb, tlen), min(te, tlen)


def gotoh_span(p, t, x, o, e, span):
    """Exact ends-free gap-affine score (byte equality): the first row (j <= tb) and the first column (i <= pb) start at
    0, the answer is the minimum over the last row (j >= tlen - te) and the last column (i >= plen - pe).  One DP row
    at a time, the recurrence of tests/golden/make_cpu_wfa_scores.py::gotoh."""
    P, T = np.frombuffer(p.encode(), np.uint8), np.frombuffer(t.encode(), np.uint8)
    m, n = len(P), len(T)
    pb, pe, tb, te = clamp(span, m, n)
    big = np.int64(1) << 40
    j = np.arange(n + 1, dtype=np.int64)
    H = np.where(j <= tb, 0, o + e * (j - tb)).astype(np.int64)
    D = np.full(n + 1, big, np.int64)
    best = int(H[n]) if m - pe <= 0 else int(big)
    for i in range(1, m + 1):
        D = np.minimum(H + (o + e), D + e)
        Hn = np.empty_like(H)
        Hn[0] = 0 if i <= pb else o + e * (i - pb)
        if n:
            Hn[1:] = np.minimum(H[:-1] + np.where(T == P[i - 1], 0, x), D[1:])
            run = np.minimum.accumulate(Hn - e * j)
            Hn[1:] = np.minimum(Hn[1:], run[:-1] + o + e * j[1:])
        H = Hn
        if i >= m - pe:
            best = min(best, int(H[n]))
    return min(best, int(H[n - te:].min()))


def gotoh_span_cells(p, t, x, o, e, span):
    """The same quantity cell by cell with three explicit matrices (small pairs only): an independent statement."""
    m, n = len(p), len(t)
    pb, pe, tb, te = clamp(span, m, n)
    INF = 1 << 40
    M = [[INF] * (n + 1) for _ in range(m + 1)]
    I = [[INF] * (n + 1) for _ in range(m + 1)]   # gap in the pattern: consumes text
    D = [[INF] * (n + 1) for _ in range(m + 1)]   # gap in the text: consumes pattern
    for i in range(m + 1):
        for jj in range(n + 1):
            if (i == 0 and jj <= tb) or (jj == 0 and i <= pb):
                M[i][jj] = 0
                continue
            if jj:
                I[i][jj] = min(min(M[i][jj - 1], D[i][jj - 1]) + o + e, I[i][jj - 1] + e)
            if i:
                D[i][jj] = min(min(M[i - 1][jj], I[i - 1][jj]) + o + e, D[i - 1][jj] + e)
            if i and jj:
                M[i][jj] = min(M[i - 1][jj - 1], I[i - 1][jj - 1], D[i - 1][jj - 1]) + (0 if p[i - 1] == t[jj - 1] else x)
    best = lambda i, jj: min(M[i][jj], I[i][jj], D[i][jj])
    return min([best(m, jj) for jj in range(n - te, n + 1)] + [best(i, n) for i in range(m - pe, m + 1)])


def mutate(rng, s, err):
    out = []
    i = 0
    while i < len(s):
        r = rng.random()
        if r < err / 3:
            out.append("ACGT"[rng.integers(4)])          # substitution (may keep the base)
        elif r < 2 * err / 3:
            pass                                           # deletion
        elif r < err:
            out.append(s[i])
            out.append("ACGT"[rng.integers(4)])          # insertion
        else:
            out.append(s[i])
        i += 1
    return "".join(out)


def rand_seq(rng, n):
    return "".join("ACGT"[c] for c in rng.integers(0, 4, n))


def window_pairs(seed, specs):
    """specs: (n, core length, flank, error).  Three shapes in turn: a read inside a flanked window of the text, a
    flanked read against its core, and a dovetail (pattern suffix overlaps text prefix).  -> [(pattern, text)]"""
    rng = np.random.default_rng(seed)
    pairs = []
    for n, core, flank, err in specs:
        for i in range(n):
            c = rand_seq(rng, core)
            shape = i % 3
            if shape == 0:
                pairs.append((mutate(rng, c, err), rand_seq(rng, flank) + c + rand_seq(rng, flank)))
            elif shape == 1:
                pairs.append((rand_seq(rng, flank) + c + rand_seq(rng, flank), mutate(rng, c, err)))
            else:
                pairs.append((rand_seq(rng, flank) + c, mutate(rng, c, err) + rand_seq(rng, flank)))
    return pairs


def span_cost_ok(lib, p, t, x, o, e, span, score, cigar):
    """wfagpu_check_result_span: `cigar` aligns p with t and costs `score` under `span`."""
    sp = wfagpu.Span(*span)
    return bool(lib.wfagpu_check_result_span(p.encode(), len(p), t.encode(), len(t), wfagpu.AffinePenalties(x, o, e),
                                             C.byref(sp), score, cigar.encode()))


def ops_to_cigar_span(lib, p, t, k_begin, ops_oldest_first):
    """wfagpu_ops_to_cigar_span on a list of 2-bit ops given oldest first (the library stores them newest first)."""
    n = len(ops_oldest_first)
    words = (C.c_uint32 * max(1, (n + 15) // 16))()
    for idx, op in enumerate(ops_oldest_first):
        jn = n - 1 - idx
        words[jn >> 4] |= op << (2 * (jn & 15))
    cg = wfagpu.Cigar()
    assert lib.wfagpu_ops_to_cigar_span(p.encode(), len(p), t.encode(), len(t), k_begin, words, n, C.byref(cg))
    out = C.string_at(cg.buffer).decode() if cg.buffer else ""
    C.CDLL(None).free(C.c_void_p(cg.buffer))
    return out
