"""CPU model of the ends-free wavefront kernel (wfa_exact_kernel<..., EF = true> + its decision-byte traceback +
cigar_text_kernel<true>), one pair at a time, vectorised per score with numpy.

It keeps the kernel's data layout and hygiene so that a wrong read shows up as a wrong result:
  * rings of depth A (M) and e + 1 (I, D), rows of width 2C + 1 around k = 0; every cell the kernel does not write for
    a score holds POISON (the kernel never clears its rings: stale values of earlier scores or pairs);
  * the prologue NULLs [-W - 2G, W + 2G] of every row, the start row is the extend of (max(0, -k), max(0, k)) on
    [-pb, tb] within the pruning window of score 0;
  * per score: the window of diagonals within (Dmax - d) / e of the target range [kt - te, kt + pe], clamped to the
    widened half width n(d) = W + min(#MDI steps, (d - o) / e); G guard cells of NULL on both sides (M-only scores:
    NULL I / D over [lo - G, hi + G]); an all-NULL step writes NULL over the clamped full range;
  * the recurrence, extend and decision bits of the kernel (I / D: extend beats open; M: D beats X beats I);
  * the end test on the written M cells: offset == min(tlen, plen + k) on a target diagonal, lowest k of the first
    finishing score;
  * the traceback from (dist, k_end) over the decision bits down to score 0 on k_begin.
The model's CIGAR comes from its own decoder (`decode`), written from the rules of the format, not from the library.

span = (pattern_begin_free, pattern_end_free, text_begin_free, text_end_free), clamped per pair."""
import ctypes as C

import numpy as np

from endsfree_ref import clamp

NULL = -32000
POISON = 12345
KIND_NULL, KIND_M, KIND_MDI = 0, 1, 2
OP_INS, OP_SUB, OP_DEL = 1, 2, 3


def steps(oracle, x, o, e, max_steps, W):
    """(n, kind) per score: the oracle's step table (km_build_steps) with every half width widened by W."""
    from oracle import KmStep
    max_dist = max_steps * (max(x, o + e) + 2) + 16
    tab = (KmStep * (max_dist + 1))()
    words = C.c_uint64()
    d_end = oracle.L.km_build_steps(x, o, e, max_steps, max_dist, tab, C.byref(words))
    n = np.array([tab[d].n + W for d in range(d_end)], np.int64)
    kind = np.array([tab[d].kind for d in range(d_end)], np.int64)
    return n, kind


class _Seqs:
    def __init__(self, p, t):
        self.plen, self.tlen = len(p), len(t)
        # distinct pads: a run never continues past the end of either sequence
        self.P = np.frombuffer(p.encode() + b"\xfe" * 40, np.uint8)
        self.T = np.frombuffer(t.encode() + b"\xff" * 40, np.uint8)

    def extend(self, k, off):
        """Vectorised extend: off + common prefix of P[off - k ..] and T[off ..]; NULL outside the sequences."""
        k, off = np.asarray(k, np.int64), np.asarray(off, np.int64).copy()
        v = off - k
        rem = np.minimum(self.plen - v, self.tlen - off)
        out = np.where(rem < 0, NULL, off)
        act = np.nonzero(rem > 0)[0]
        run = np.zeros(len(act), np.int64)
        j = np.arange(32)
        while len(act):
            vi = (v[act] + run)[:, None] + j
            hi_ = (off[act] + run)[:, None] + j
            eq = self.P[np.minimum(vi, len(self.P) - 1)] == self.T[np.minimum(hi_, len(self.T) - 1)]
            first = np.where(eq.all(axis=1), 32, np.argmin(eq, axis=1))
            run += first
            cont = (first == 32) & (run < rem[act])
            out[act] = off[act] + np.minimum(run, rem[act])
            act, run = act[cont], run[cont]
        return out


def prune(n, tlo, thi, q):
    lo, hi = max(-n, tlo - q), min(n, thi + q)
    if lo <= hi:
        return True, lo, hi
    return False, -n, n


def align(oracle, p, t, x, o, e, span, max_steps=4000, dmax=-1, cigar=True):
    """-> dict(finished, distance, k_begin, k_end, ops (oldest first), cigar)."""
    s = _Seqs(p, t)
    plen, tlen = s.plen, s.tlen
    pb, pe, tb, te = clamp(span, plen, tlen)
    W = max(pb, tb)
    ns, kinds = steps(oracle, x, o, e, max_steps, W)
    d_end = len(ns)
    A, E1 = max(o + e, x) + 1, e + 1
    G = A
    Cc = int(ns.max()) + 2 * G + 2
    width = 2 * Cc + 1
    Mr = np.full((A, width), POISON, np.int64)
    Ir = np.full((E1, width), POISON, np.int64)
    Dr = np.full((E1, width), POISON, np.int64)
    pro = slice(Cc - 2 * G - W, Cc + 2 * G + W + 1)
    Mr[:, pro] = NULL
    Ir[:, pro] = NULL
    Dr[:, pro] = NULL
    kt = tlen - plen
    klo, khi = kt - te, kt + pe
    Dmax = d_end - 1 if dmax < 0 else min(dmax, d_end - 1)
    decs = {}

    def ix(lo, hi):
        return slice(Cc + lo, Cc + hi + 1)

    def lowest_finish(row, lo, hi):
        a, b = max(lo, klo), min(hi, khi)
        if a > b:
            return None
        ks = np.arange(a, b + 1)
        hit = np.nonzero(row[ix(a, b)] == np.minimum(tlen, plen + ks))[0]
        return int(ks[hit[0]]) if len(hit) else None

    fin, dist, k_end = False, 0, None
    live0, lo0, hi0 = prune(int(ns[0]), klo, khi, Dmax // e)
    if live0:
        slo, shi = max(-pb, lo0), min(tb, hi0)
        if slo <= shi:
            ks = np.arange(slo, shi + 1)
            Mr[0, ix(slo, shi)] = s.extend(ks, np.maximum(0, ks))
            k_end = lowest_finish(Mr[0], slo, shi)
            fin = k_end is not None
    d = 0
    if not fin:
        for d in range(1, Dmax + 1):
            n, kind = int(ns[d]), int(kinds[d])
            live, lo, hi = prune(n, klo, khi, (Dmax - d) // e)
            Mc, Ic, Dc = Mr[d % A], Ir[d % E1], Dr[d % E1]
            Mc[:] = POISON
            Ic[:] = POISON
            Dc[:] = POISON
            if kind == KIND_NULL or not live:
                Mc[ix(lo - G, hi + G)] = NULL
                Ic[ix(lo - G, hi + G)] = NULL
                Dc[ix(lo - G, hi + G)] = NULL
                continue
            Mx = Mr[(d - x) % A]
            ks = np.arange(lo, hi + 1)
            if kind == KIND_M:
                Ic[ix(lo - G, hi + G)] = NULL
                Dc[ix(lo - G, hi + G)] = NULL
                Mc[ix(lo - G, lo - 1)] = NULL
                Mc[ix(hi + 1, hi + G)] = NULL
                m = Mx[ix(lo, hi)] + 1
                ok = m >= 0
                m[ok] = s.extend(ks[ok], m[ok])
                Mc[ix(lo, hi)] = m
            else:
                for R in (Mc, Ic, Dc):
                    R[ix(lo - G, lo - 1)] = NULL
                    R[ix(hi + 1, hi + G)] = NULL
                Mo, Ie, De = Mr[(d - o - e) % A], Ir[(d - e) % E1], Dr[(d - e) % E1]
                io, ie = Mo[ix(lo - 1, hi - 1)] + 1, Ie[ix(lo - 1, hi - 1)] + 1
                dopen, dext = Mo[ix(lo + 1, hi + 1)], De[ix(lo + 1, hi + 1)]
                X = Mx[ix(lo, hi)] + 1
                I, D = np.maximum(io, ie), np.maximum(dopen, dext)
                M = np.maximum(np.maximum(X, D), I)
                dec = ((ie >= io).astype(np.int64) | ((dext >= dopen).astype(np.int64) << 1) |
                       (((D >= X) | (I > X)).astype(np.int64) << 2) | (((D >= I) | (X >= I)).astype(np.int64) << 3))
                ok = M >= 0
                M[ok] = s.extend(ks[ok], M[ok])
                Ic[ix(lo, hi)], Dc[ix(lo, hi)], Mc[ix(lo, hi)] = I, D, M
                decs[d] = (lo, dec)
            k_end = lowest_finish(Mc, lo, hi)
            if k_end is not None:
                fin, dist = True, d
                break
    if not fin:
        return dict(finished=False, distance=0, k_begin=None, k_end=None, ops=None, cigar=None)
    ops, cd, ck, comp = [], dist, k_end, 0
    oe = o + e
    while not (comp == 0 and cd == 0):
        kind = int(kinds[cd])
        if comp == 0:
            op = OP_SUB
            if kind == KIND_M:
                cd -= x
            else:
                mop = (_dec(decs, cd, ck) >> 2) & 3
                if mop == OP_SUB:
                    cd -= x
                elif mop == OP_INS:
                    comp = 1
                else:
                    comp = 2
        else:
            assert kind == KIND_MDI, "gap walk on a score without gaps"
            dec = _dec(decs, cd, ck)
            if comp == 1:
                op = OP_INS
                ck -= 1
                if dec & 1:
                    cd -= e
                else:
                    cd -= oe
                    comp = 0
            else:
                op = OP_DEL
                ck += 1
                if dec & 2:
                    cd -= e
                else:
                    cd -= oe
                    comp = 0
        ops.append(op)
        assert cd >= 0, "traceback below score 0"
    ops.reverse()
    cg = decode(p, t, ck, ops) if cigar else None
    return dict(finished=True, distance=dist, k_begin=ck, k_end=k_end, ops=ops, cigar=cg)


def _dec(decs, d, k):
    assert d in decs, "traceback reads a score that wrote no decisions"
    lo, dec = decs[d]
    assert 0 <= k - lo < len(dec), "traceback leaves the window of its score"
    return int(dec[k - lo])


def decode(p, t, k_begin, ops):
    """CIGAR text of an ends-free path (ops oldest first): a leading I (k_begin > 0, text) or D run of |k_begin|, the
    path from (max(0, -k_begin), max(0, k_begin)) -- match runs re-derived on the sequences between ops, X inside a gap
    is its closing delimiter and prints nothing, equal ops merge unless a delimiter or a match run separates them --
    and a trailing I / D run to the end of both sequences.  A free run and a gap run of the same letter next to it
    (no match run between them) print as one run."""
    runs = []                                # [letter, length, is_gap_run_closed_by_delimiter]

    def put(letter, n):
        if n:
            runs.append([letter, n])

    def match(v, h):
        m = 0
        while v + m < len(p) and h + m < len(t) and p[v + m] == t[h + m]:
            m += 1
        return m

    k, off = k_begin, max(0, k_begin)
    lead = "I" if k_begin > 0 else "D"
    pending = [lead, abs(k_begin)]           # run being accumulated
    in_gap = False
    last_closed = None                       # gap run closed by the last op's delimiter, not printed yet
    for idx, op in enumerate(ops):
        letter = "?IXD"[op]
        closing = in_gap and op == OP_SUB
        if not closing and pending[1] and pending[0] != letter:
            put(*pending)
            pending = [letter, 0]
        if not in_gap:
            m = match(off - k, off)
            if m:
                put(*pending)
                pending = [letter, 0]
                put("M", m)
                off += m
        if op == OP_DEL:
            in_gap = True
            k -= 1
            pending = [letter, pending[1] + 1] if pending[0] == letter else [letter, 1]
        elif op == OP_INS:
            in_gap = True
            k += 1
            off += 1
            pending = [letter, pending[1] + 1] if pending[0] == letter else [letter, 1]
        else:
            if in_gap:
                in_gap = False
                if idx != len(ops) - 1:
                    put(*pending)                # the delimiter ends the gap run
                    pending = ["?", 0]
            else:
                off += 1
                pending = ["X", pending[1] + 1] if pending[0] == "X" else ["X", 1]
    m = 0 if in_gap else match(off - k, off)
    if m:
        put(*pending)
        pending = ["?", 0]
        put("M", m)
        off += m
    tail_i, tail_d = len(t) - off, len(p) - (off - k)
    tail = ("I", tail_i) if tail_i else ("D", tail_d)
    if tail[1]:
        if pending[1] and pending[0] == tail[0]:
            pending[1] += tail[1]
        else:
            put(*pending)
            pending = list(tail)
    put(*pending)
    return "".join("%d%s" % (n, letter) for letter, n in runs)
