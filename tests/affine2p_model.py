"""CPU model of the gap-affine 2-piece wavefront kernel (wfa_exact_kernel<..., P2 = true> + its decision-byte
traceback), one pair at a time, vectorised per score with numpy.

It keeps the kernel's data layout and hygiene so that a wrong read shows up as a wrong result:
  * rings of depth A = max(x, o1 + e1, o2 + e2) + 1 (M), e1 + 1 (I1, D1) and e2 + 1 (I2, D2), rows of width 2C + 1
    around k = 0; every cell the kernel does not write for a score holds POISON (the kernel never clears its rings);
  * the prologue NULLs [-2G, 2G] of every row (G = A), score 0 is the extend of (0, 0) on k = 0;
  * per score: the window of diagonals within (Dmax - d) / min(e1, e2) of kt, clamped to the half width of the step
    table (`steps`, a restatement of wfagpu_build_step_table_affine2p); G guard cells of NULL on both sides (M-only
    scores: NULL I1 / D1 / I2 / D2 over [lo - G, hi + G]); an all-NULL step writes NULL over the clamped full range;
  * the recurrence, extend and decision byte of the kernel: bit0 I1 extends, bit1 D1, bit2 I2, bit3 D2 (extend beats
    open), bits 5:4 the op of M's source (1 I, 2 X, 3 D), bit6 the source is piece 2 (M: D1 > D2 > X > I1 > I2);
  * the end test M[kt] == tlen, and the five-component traceback from (dist, kt) to score 0.
The CIGAR comes from endsfree_model.decode with k_begin = 0 (a global path).

pen = (x, o1, e1, o2, e2)."""
import numpy as np

from endsfree_model import KIND_M, KIND_MDI, KIND_NULL, NULL, OP_DEL, OP_INS, OP_SUB, POISON, _Seqs, decode


def steps(x, o1, e1, o2, e2, max_steps, max_dist=None):
    """(n, kind) per score 0 .. d_end - 1: a gap of piece i exists at d when M existed at d - o_i - e_i or that gap at
    d - e_i; a score is an M/I/D step when either gap exists, an M step when only M[d - x] does.  The half width is
    min(#M/I/D steps, max((d - o1) / e1, (d - o2) / e2)), at least 0.  The budget: M/I/D steps stop once the step count
    (which starts at 1 for score 0) reaches max_steps - 1."""
    if max_dist is None:
        max_dist = max_steps * (max(x, o1 + e1, o2 + e2) + 1) + 16
    has_m, g1, g2 = [True], [False], [False]
    ns, kinds = [0], [KIND_M]
    n = mdi = 0
    nsteps = 1
    for d in range(1, max_dist):
        if nsteps >= max_steps - 1 or n >= 65535 or mdi >= 65535:
            break
        a = d - o1 - e1 >= 0 and (has_m[d - o1 - e1] or g1[d - e1])
        b = d - o2 - e2 >= 0 and (has_m[d - o2 - e2] or g2[d - e2])
        g1.append(a)
        g2.append(b)
        if a or b:
            kind = KIND_MDI
            mdi += 1
            nsteps += 1
            reach = max(int((d - o1) / e1), int((d - o2) / e2))      # C division: towards zero
            n = max(0, min(mdi, reach))
        elif d - x >= 0 and has_m[d - x]:
            kind = KIND_M
        else:
            kind = KIND_NULL
        has_m.append(kind != KIND_NULL)
        ns.append(n)
        kinds.append(kind)
    return np.array(ns, np.int64), np.array(kinds, np.int64)


def prune(n, kt, q):
    lo, hi = max(-n, kt - q), min(n, kt + q)
    if lo <= hi:
        return True, lo, hi
    return False, -n, n


def align(p, t, x, o1, e1, o2, e2, max_steps=4000, dmax=-1, cigar=True):
    """-> dict(finished, distance, ops (oldest first), cigar)."""
    s = _Seqs(p, t)
    plen, tlen = s.plen, s.tlen
    ns, kinds = steps(x, o1, e1, o2, e2, max_steps)
    d_end = len(ns)
    A, E1, E2 = max(x, o1 + e1, o2 + e2) + 1, e1 + 1, e2 + 1
    G = A
    ep = min(e1, e2)
    Cc = int(ns.max()) + 2 * G + 2
    width = 2 * Cc + 1
    Mr = np.full((A, width), POISON, np.int64)
    I1r, D1r = np.full((E1, width), POISON, np.int64), np.full((E1, width), POISON, np.int64)
    I2r, D2r = np.full((E2, width), POISON, np.int64), np.full((E2, width), POISON, np.int64)
    pro = slice(Cc - 2 * G, Cc + 2 * G + 1)
    for R in (Mr, I1r, D1r, I2r, D2r):
        R[:, pro] = NULL
    kt = tlen - plen
    Dmax = d_end - 1 if dmax < 0 else min(dmax, d_end - 1)
    decs = {}

    def ix(lo, hi):
        return slice(Cc + lo, Cc + hi + 1)

    Mr[0, Cc] = s.extend([0], [0])[0]
    fin, dist = kt == 0 and Mr[0, Cc] == tlen, 0
    if not fin:
        for d in range(1, Dmax + 1):
            n, kind = int(ns[d]), int(kinds[d])
            live, lo, hi = prune(n, kt, (Dmax - d) // ep)
            cur = (Mr[d % A], I1r[d % E1], D1r[d % E1], I2r[d % E2], D2r[d % E2])
            for R in cur:
                R[:] = POISON
            Mc, I1c, D1c, I2c, D2c = cur
            if kind == KIND_NULL or not live:
                for R in cur:
                    R[ix(lo - G, hi + G)] = NULL
                continue
            Mx = Mr[(d - x) % A]
            ks = np.arange(lo, hi + 1)
            if kind == KIND_M:
                for R in cur[1:]:
                    R[ix(lo - G, hi + G)] = NULL
                Mc[ix(lo - G, lo - 1)] = NULL
                Mc[ix(hi + 1, hi + G)] = NULL
                m = Mx[ix(lo, hi)] + 1
                ok = m >= 0
                m[ok] = s.extend(ks[ok], m[ok])
                Mc[ix(lo, hi)] = m
            else:
                for R in cur:
                    R[ix(lo - G, lo - 1)] = NULL
                    R[ix(hi + 1, hi + G)] = NULL
                # piece 2 (or 1) may not exist yet: M[d - o - e] is then a row no score has written, NULL from the
                # prologue as long as the window stays within [-2G, 2G]
                Mo1, Mo2 = Mr[(d - o1 - e1) % A], Mr[(d - o2 - e2) % A]
                I1e, D1e, I2e, D2e = I1r[(d - e1) % E1], D1r[(d - e1) % E1], I2r[(d - e2) % E2], D2r[(d - e2) % E2]
                io1, ie1 = Mo1[ix(lo - 1, hi - 1)] + 1, I1e[ix(lo - 1, hi - 1)] + 1
                io2, ie2 = Mo2[ix(lo - 1, hi - 1)] + 1, I2e[ix(lo - 1, hi - 1)] + 1
                do1, de1 = Mo1[ix(lo + 1, hi + 1)], D1e[ix(lo + 1, hi + 1)]
                do2, de2 = Mo2[ix(lo + 1, hi + 1)], D2e[ix(lo + 1, hi + 1)]
                X = Mx[ix(lo, hi)] + 1
                I1, D1, I2, D2 = np.maximum(io1, ie1), np.maximum(do1, de1), np.maximum(io2, ie2), np.maximum(do2, de2)
                I, D = np.maximum(I1, I2), np.maximum(D1, D2)
                M = np.maximum(np.maximum(X, D), I)
                src = np.where((D >= X) & (D >= I), np.where(D1 >= D2, 0x30, 0x70),
                               np.where(X >= I, 0x20, np.where(I1 >= I2, 0x10, 0x50)))
                dec = ((ie1 >= io1).astype(np.int64) | ((de1 >= do1).astype(np.int64) << 1) |
                       ((ie2 >= io2).astype(np.int64) << 2) | ((de2 >= do2).astype(np.int64) << 3) | src)
                ok = M >= 0
                M[ok] = s.extend(ks[ok], M[ok])
                I1c[ix(lo, hi)], D1c[ix(lo, hi)], I2c[ix(lo, hi)], D2c[ix(lo, hi)] = I1, D1, I2, D2
                Mc[ix(lo, hi)] = M
                decs[d] = (lo, dec)
            if lo <= kt <= hi and Mc[Cc + kt] == tlen:
                fin, dist = True, d
                break
    if not fin:
        return dict(finished=False, distance=0, ops=None, cigar=None)
    ops, cd, ck, comp = [], dist, kt, 0
    ext = {1: e1, 2: e1, 3: e2, 4: e2}
    opn = {1: o1 + e1, 2: o1 + e1, 3: o2 + e2, 4: o2 + e2}
    while not (comp == 0 and cd == 0):
        kind = int(kinds[cd])
        if comp == 0:
            op = OP_SUB
            if kind == KIND_M:
                cd -= x
            else:
                dec = _dec(decs, cd, ck)
                mop = (dec >> 4) & 3
                if mop == OP_SUB:
                    cd -= x
                elif mop == OP_INS:
                    comp = 3 if dec & 64 else 1
                else:
                    comp = 4 if dec & 64 else 2
        else:
            assert kind == KIND_MDI, "gap walk on a score without gaps"
            dec = _dec(decs, cd, ck)
            ins = comp in (1, 3)
            op = OP_INS if ins else OP_DEL
            ck += -1 if ins else 1
            if dec & (1 << (comp - 1)):
                cd -= ext[comp]
            else:
                cd -= opn[comp]
                comp = 0
        ops.append(op)
        assert cd >= 0, "traceback below score 0"
    assert ck == 0, "traceback does not end on diagonal 0"
    ops.reverse()
    return dict(finished=True, distance=dist, ops=ops, cigar=decode(p, t, 0, ops) if cigar else None)


def _dec(decs, d, k):
    assert d in decs, "traceback reads a score that wrote no decisions"
    lo, dec = decs[d]
    assert 0 <= k - lo < len(dec), "traceback leaves the window of its score"
    return int(dec[k - lo])
