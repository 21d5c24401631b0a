"""Gap-affine 2-piece ground truth for the tests: an exact DP under WFA2-lib's affine2p model (a gap of L bases costs
min(o1 + e1 L, o2 + e2 L), a mismatch x), the pairs the tests align (reads with one long indel), and the library's
2-piece helpers through ctypes.

pen = (x, o1, e1, o2, e2)."""
import ctypes as C

import numpy as np

import wfagpu
from endsfree_ref import mutate, rand_seq


def gotoh2p(p, t, x, o1, e1, o2, e2):
    """Exact global 2-piece score (byte equality), one DP row at a time: per piece a vertical gap matrix, and the
    horizontal gaps of a row by the `minimum.accumulate` trick once per piece (two gaps in a row are never cheaper
    than one gap over both, so a horizontal gap may start from the row before its own horizontal update)."""
    P, T = np.frombuffer(p.encode(), np.uint8), np.frombuffer(t.encode(), np.uint8)
    m, n = len(P), len(T)
    big = np.int64(1) << 40
    pieces = ((o1, e1), (o2, e2))
    j = np.arange(n + 1, dtype=np.int64)

    def gap(L):
        return np.minimum(o1 + e1 * L, o2 + e2 * L)

    H = np.where(j == 0, 0, gap(j)).astype(np.int64)
    Ds = [np.full(n + 1, big, np.int64) for _ in pieces]
    for i in range(1, m + 1):
        Ds = [np.minimum(H + (o + e), Dk + e) for (o, e), Dk in zip(pieces, Ds)]
        Hn = np.minimum(Ds[0], Ds[1])
        Hn[0] = gap(i)
        if n:
            Hn[1:] = np.minimum(Hn[1:], H[:-1] + np.where(T == P[i - 1], 0, x))
            Hh = Hn.copy()
            for o, e in pieces:
                run = np.minimum.accumulate(Hn - e * j)
                Hh[1:] = np.minimum(Hh[1:], run[:-1] + o + e * j[1:])
            Hn = Hh
        H = Hn
    return int(H[n])


def gotoh2p_cells(p, t, x, o1, e1, o2, e2):
    """The same score cell by cell with five explicit matrices (small pairs only): an independent statement."""
    m, n = len(p), len(t)
    INF = 1 << 40
    M = [[INF] * (n + 1) for _ in range(m + 1)]
    Is = [[[INF] * (n + 1) for _ in range(m + 1)] for _ in range(2)]   # gaps in the pattern: consume text
    Ds = [[[INF] * (n + 1) for _ in range(m + 1)] for _ in range(2)]   # gaps in the text: consume pattern
    pieces = ((o1, e1), (o2, e2))
    M[0][0] = 0
    for i in range(m + 1):
        for jj in range(n + 1):
            if i == 0 and jj == 0:
                continue
            best = INF
            for q, (o, e) in enumerate(pieces):
                if jj:
                    Is[q][i][jj] = min(M[i][jj - 1] + o + e, Is[q][i][jj - 1] + e)
                if i:
                    Ds[q][i][jj] = min(M[i - 1][jj] + o + e, Ds[q][i - 1][jj] + e)
                best = min(best, Is[q][i][jj], Ds[q][i][jj])
            if i and jj:
                best = min(best, M[i - 1][jj - 1] + (0 if p[i - 1] == t[jj - 1] else x))
            M[i][jj] = best
    return M[m][n]


def indel_pairs(seed, specs):
    """specs: (n, length, error, indel_lo, indel_hi).  The pattern is the text mutated at `error` (`mutate`) with one
    insertion or deletion of indel_lo .. indel_hi bases (alternating) at a random position.  -> [(pattern, text)]"""
    rng = np.random.default_rng(seed)
    pairs = []
    for n, length, err, lo, hi in specs:
        for i in range(n):
            t = rand_seq(rng, length)
            p = mutate(rng, t, err)
            L = int(rng.integers(lo, hi + 1))
            at = int(rng.integers(0, max(1, len(p) - L)))
            if i % 2 == 0:
                p = p[:at] + rand_seq(rng, L) + p[at:]
            else:
                p = p[:at] + p[at + L:]
            pairs.append((p, t))
    return pairs


def affine2p(pen):
    return wfagpu.Affine2p(*pen)


def cost_ok(lib, p, t, pen, score, cigar):
    """wfagpu_check_result_affine2p: `cigar` aligns p with t and costs `score` under the 2-piece penalties."""
    q = affine2p(pen)
    return bool(lib.wfagpu_check_result_affine2p(p.encode(), len(p), t.encode(), len(t), C.byref(q), score,
                                                 cigar.encode()))


def step_table(lib, pen, max_steps, max_dist):
    """wfagpu_build_step_table_affine2p -> (d_end, [(row_off, n, kind)], arena units)."""
    tab = (wfagpu.Step * (max_dist + 1))()
    units = C.c_uint64()
    d_end = lib.wfagpu_build_step_table_affine2p(*pen, max_steps, max_dist, tab, C.byref(units))
    return d_end, [(tab[d].row_off, tab[d].n, tab[d].kind) for d in range(max(d_end, 0))], units.value
