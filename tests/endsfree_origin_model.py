"""CPU model of the score-only ends-free kernel with origin rows (wfa_exact_kernel<..., EF = true, BT = false,
ORG = true>), one pair at a time, vectorised per score with numpy.

The forward pass is the one of tests/endsfree_model.py (same rings, prologue, start row, range pruning, guard cells,
recurrence and lowest-k end rule, built from its helpers), plus the kernel's origin rows: every written M, I and D cell
also stores the score-0 diagonal its path started on, taken from the winner the decision bits of the CIGAR kernel
record (I / D: extend beats open; M: D > X > I; an M-only step copies M[d - x][k]; extend keeps it).  Origin rows have
no prologue and no NULL stores, so every origin cell a score does not write -- pruned, guard, NULL-step and prologue
cells included -- holds OPOISON; a read of one on the optimal path shows up as a wrong k_origin.  There is no
traceback: the origin of the finishing cell is the model's k_begin, which tests/test_endsfree_origin_model.py compares
with the traceback of tests/endsfree_model.py."""
import numpy as np

from endsfree_model import KIND_M, KIND_NULL, NULL, POISON, _Seqs, prune, steps
from endsfree_ref import clamp

OPOISON = 7654321                            # an origin cell the kernel never writes: no diagonal of any pair


def align(oracle, p, t, x, o, e, span, max_steps=4000, dmax=-1):
    """-> dict(finished, distance, k_end, k_origin)."""
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
    Om = np.full((A, width), OPOISON, np.int64)      # origin rows: no prologue
    Oi = np.full((E1, width), OPOISON, np.int64)
    Od = np.full((E1, width), OPOISON, np.int64)
    kt = tlen - plen
    klo, khi = kt - te, kt + pe
    Dmax = d_end - 1 if dmax < 0 else min(dmax, d_end - 1)

    def ix(lo, hi):
        return slice(Cc + lo, Cc + hi + 1)

    def lowest_finish(row, lo, hi):
        a, b = max(lo, klo), min(hi, khi)
        if a > b:
            return None
        ks = np.arange(a, b + 1)
        hit = np.nonzero(row[ix(a, b)] == np.minimum(tlen, plen + ks))[0]
        return int(ks[hit[0]]) if len(hit) else None

    live0, lo0, hi0 = prune(int(ns[0]), klo, khi, Dmax // e)
    if live0:
        slo, shi = max(-pb, lo0), min(tb, hi0)
        if slo <= shi:
            ks = np.arange(slo, shi + 1)
            Mr[0, ix(slo, shi)] = s.extend(ks, np.maximum(0, ks))
            Om[0, ix(slo, shi)] = ks
            k_end = lowest_finish(Mr[0], slo, shi)
            if k_end is not None:
                return dict(finished=True, distance=0, k_end=k_end, k_origin=int(Om[0][Cc + k_end]))
    for d in range(1, Dmax + 1):
        n, kind = int(ns[d]), int(kinds[d])
        live, lo, hi = prune(n, klo, khi, (Dmax - d) // e)
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
            # the winners the decision bits record: I / D extend beats open; M: D (bM0 & bM1) > X (bM1) > I
            oI = np.where(ie >= io, OIe[ix(lo - 1, hi - 1)], OMo[ix(lo - 1, hi - 1)])
            oD = np.where(dext >= dopen, ODe[ix(lo + 1, hi + 1)], OMo[ix(lo + 1, hi + 1)])
            bM0, bM1 = (D >= X) | (I > X), (D >= I) | (X >= I)
            oM = np.where(bM1, np.where(bM0, oD, OMx[ix(lo, hi)]), oI)
            ok = M >= 0
            M[ok] = s.extend(ks[ok], M[ok])
            Ic[ix(lo, hi)], Dc[ix(lo, hi)], Mc[ix(lo, hi)] = I, D, M
            Oic[ix(lo, hi)], Odc[ix(lo, hi)], Omc[ix(lo, hi)] = oI, oD, oM
        k_end = lowest_finish(Mc, lo, hi)
        if k_end is not None:
            return dict(finished=True, distance=d, k_end=k_end, k_origin=int(Omc[Cc + k_end]))
    return dict(finished=False, distance=0, k_end=None, k_origin=None)
