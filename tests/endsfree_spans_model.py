"""CPU model of the ends-free kernel for one pair of a batch with per-pair spans (DESIGN.md §9, "Per-pair spans"): the
step table is widened by the batch's widest start row W_b (at least the pair's own W = max(pb, tb)), the prologue is the
pair's own [-W - 2G, W + 2G], and every window is clamped to the pair's own reach [-pb - r(d), tb + r(d)],
r(d) = n(d) - W_b.  `trim` = (low, high) narrows that clamp by as many diagonals (a deliberately wrong kernel).

It is the forward pass of tests/endsfree_model.py (rings with every cell a score does not write poisoned, start row,
range pruning, guard cells, recurrence, decision bits, lowest-k end rule) with the clamp, plus the origin rows of
tests/endsfree_origin_model.py (no prologue, no NULL stores, unwritten origin cells poisoned), and the decision-byte
traceback and CIGAR decoder of tests/endsfree_model.py.  With W_b = W and no trim the clamp never cuts a cell that can be
non-NULL, so the results must equal those two models'."""
import numpy as np

from endsfree_model import KIND_M, KIND_NULL, NULL, OP_DEL, OP_INS, OP_SUB, POISON, _dec, _Seqs, decode, steps
from endsfree_origin_model import OPOISON
from endsfree_ref import clamp


def reach_window(n, tlo, thi, q, dp, dt):
    """prune_window_range of the kernel: the diagonals within q of [tlo, thi] inside the own reach [dp - n, n - dt]; an
    all-NULL step NULLs that reach."""
    lo, hi = max(dp - n, tlo - q), min(n - dt, thi + q)
    if lo <= hi:
        return True, lo, hi
    return False, dp - n, n - dt


def align(oracle, p, t, x, o, e, span, batch_w, trim=(0, 0), max_steps=4000, dmax=-1, cigar=True):
    """-> dict(finished, distance, k_begin, k_end, k_origin, ops (oldest first), cigar)."""
    s = _Seqs(p, t)
    plen, tlen = s.plen, s.tlen
    pb, pe, tb, te = clamp(span, plen, tlen)
    W = max(pb, tb)
    Wb = max(batch_w, W)
    dp, dt = Wb - pb + trim[0], Wb - tb + trim[1]
    ns, kinds = steps(oracle, x, o, e, max_steps, Wb)
    d_end = len(ns)
    A, E1 = max(o + e, x) + 1, e + 1
    G = A
    Cc = int(ns.max()) + 2 * G + 2
    width = 2 * Cc + 1
    Mr = np.full((A, width), POISON, np.int64)
    Ir = np.full((E1, width), POISON, np.int64)
    Dr = np.full((E1, width), POISON, np.int64)
    pro = slice(Cc - 2 * G - W, Cc + 2 * G + W + 1)          # the pair's own prologue, not the batch's
    Mr[:, pro] = NULL
    Ir[:, pro] = NULL
    Dr[:, pro] = NULL
    Om = np.full((A, width), OPOISON, np.int64)
    Oi = np.full((E1, width), OPOISON, np.int64)
    Od = np.full((E1, width), OPOISON, np.int64)
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

    fin, dist, k_end, k_origin = False, 0, None, None
    live0, lo0, hi0 = reach_window(int(ns[0]), klo, khi, Dmax // e, dp, dt)
    if live0 and lo0 <= hi0:
        ks = np.arange(lo0, hi0 + 1)
        Mr[0, ix(lo0, hi0)] = s.extend(ks, np.maximum(0, ks))
        Om[0, ix(lo0, hi0)] = ks
        k_end = lowest_finish(Mr[0], lo0, hi0)
        if k_end is not None:
            fin, k_origin = True, int(Om[0][Cc + k_end])
    if not fin:
        for d in range(1, Dmax + 1):
            n, kind = int(ns[d]), int(kinds[d])
            live, lo, hi = reach_window(n, klo, khi, (Dmax - d) // e, dp, dt)
            Mc, Ic, Dc = Mr[d % A], Ir[d % E1], Dr[d % E1]
            Omc, Oic, Odc = Om[d % A], Oi[d % E1], Od[d % E1]
            for R in (Mc, Ic, Dc):
                R[:] = POISON
            for R in (Omc, Oic, Odc):
                R[:] = OPOISON
            if kind == KIND_NULL or not live:
                for R in (Mc, Ic, Dc):
                    R[ix(lo - G, hi + G)] = NULL
                continue
            Mx, OMx = Mr[(d - x) % A], Om[(d - x) % A]
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
                Omc[ix(lo, hi)] = OMx[ix(lo, hi)]
            else:
                for R in (Mc, Ic, Dc):
                    R[ix(lo - G, lo - 1)] = NULL
                    R[ix(hi + 1, hi + G)] = NULL
                Mo, Ie, De = Mr[(d - o - e) % A], Ir[(d - e) % E1], Dr[(d - e) % E1]
                OMo, OIe, ODe = Om[(d - o - e) % A], Oi[(d - e) % E1], Od[(d - e) % E1]
                io, ie = Mo[ix(lo - 1, hi - 1)] + 1, Ie[ix(lo - 1, hi - 1)] + 1
                dopen, dext = Mo[ix(lo + 1, hi + 1)], De[ix(lo + 1, hi + 1)]
                X = Mx[ix(lo, hi)] + 1
                I, D = np.maximum(io, ie), np.maximum(dopen, dext)
                M = np.maximum(np.maximum(X, D), I)
                bI, bD = ie >= io, dext >= dopen
                bM0, bM1 = (D >= X) | (I > X), (D >= I) | (X >= I)
                dec = (bI.astype(np.int64) | (bD.astype(np.int64) << 1) | (bM0.astype(np.int64) << 2) |
                       (bM1.astype(np.int64) << 3))
                oI = np.where(bI, OIe[ix(lo - 1, hi - 1)], OMo[ix(lo - 1, hi - 1)])
                oD = np.where(bD, ODe[ix(lo + 1, hi + 1)], OMo[ix(lo + 1, hi + 1)])
                oM = np.where(bM1, np.where(bM0, oD, OMx[ix(lo, hi)]), oI)
                ok = M >= 0
                M[ok] = s.extend(ks[ok], M[ok])
                Ic[ix(lo, hi)], Dc[ix(lo, hi)], Mc[ix(lo, hi)] = I, D, M
                Oic[ix(lo, hi)], Odc[ix(lo, hi)], Omc[ix(lo, hi)] = oI, oD, oM
                decs[d] = (lo, dec)
            k_end = lowest_finish(Mc, lo, hi)
            if k_end is not None:
                fin, dist, k_origin = True, d, int(Omc[Cc + k_end])
                break
    if not fin:
        return dict(finished=False, distance=0, k_begin=None, k_end=None, k_origin=None, ops=None, cigar=None)
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
                else:
                    comp = 1 if mop == OP_INS else 2
        else:
            dec = _dec(decs, cd, ck)
            op = OP_INS if comp == 1 else OP_DEL
            ck += -1 if comp == 1 else 1
            if dec & comp:                           # bit 0: I extends, bit 1: D extends
                cd -= e
            else:
                cd -= oe
                comp = 0
        ops.append(op)
        assert cd >= 0, "traceback below score 0"
    ops.reverse()
    return dict(finished=True, distance=dist, k_begin=ck, k_end=k_end, k_origin=k_origin, ops=ops,
                cigar=decode(p, t, ck, ops) if cigar else None)
