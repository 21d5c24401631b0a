"""Pairs for the byte-compare kernels (pairs the packer flags: an 'N' in either sequence, or any aligned 4-byte group
whose bytes all differ from 'N' in no common bit, such as "YTGC") and their relabelled twins.

The byte-compare kernels, the packed kernels and the oracle compare bases only for equality, so a result (score, CIGAR
text, whether the band finishes) does not change when the bytes of a pair are relabelled one to one.  A flagged pair
that uses at most four distinct bytes therefore has a twin over ACGT -- the same pair with its bytes mapped one to one
onto A, C, G, T -- that the packer does not flag, and the byte-compare result of the pair must equal the packed result
and the oracle's result of its twin.  Pairs with five or more distinct bytes have no twin (None).

Every generator is seeded and returns (pairs, twins)."""
import random

ACGT = "ACGT"


def packer_flags(seq):
    """The pack kernel's flag for one sequence: an aligned group of four bytes (NUL past the end) that is not all NUL and
    whose (byte ^ 'N') values AND to zero.  The oracle's orc_has_N also flags every sequence of 32768 bases or more (the
    reference's int16 offsets); the pack kernel does not, such sequences take the large tier."""
    b = seq.encode() if isinstance(seq, str) else seq
    for g in range(0, len(b) + 4 - len(b) % 4, 4):
        grp = (b[g:g + 4] + b"\0\0\0\0")[:4]
        if any(grp) and (grp[0] ^ 0x4E) & (grp[1] ^ 0x4E) & (grp[2] ^ 0x4E) & (grp[3] ^ 0x4E) == 0:
            return True
    return False


def pair_flagged(p, t):
    return packer_flags(p) or packer_flags(t)


def twin(rng, p, t):
    """(p, t) with its distinct bytes mapped one to one onto a random choice of A, C, G, T; None for five or more bytes."""
    used = sorted(set(p + t))
    if len(used) > 4:
        return None
    m = dict(zip(used, rng.sample(ACGT, 4)))
    return "".join(m[c] for c in p), "".join(m[c] for c in t)


def _seq(rng, alpha, n, weights=None):
    return "".join(rng.choices(alpha, weights=weights, k=n))


def _mutate(rng, s, err, alpha):
    """Substitutions, deletions and insertions at rate `err` in total, new bases drawn from `alpha`."""
    out = []
    for c in s:
        r = rng.random()
        if r < err / 3:
            out.append(rng.choice(alpha))
        elif r < 2 * err / 3:
            continue
        elif r < err:
            out.append(c)
            out.append(rng.choice(alpha))
        else:
            out.append(c)
    return "".join(out)


# four-byte alphabets with an N in them (N dense: uniform; N sparse: weight 1 in 60)
N_ALPHABETS = ["ACGN", "NCGT", "ANGT", "ACNT"]


def _n_weights(alpha, sparse):
    return [1 if c == "N" else 20 for c in alpha] if sparse else None


def _finish(rng, pairs):
    return pairs, [twin(rng, p, t) for p, t in pairs]


def mutated_reads(seed, n, length, err_lo, err_hi):
    """Reads over a four-byte alphabet with an N (dense or sparse N), mutated against their text."""
    rng = random.Random(seed)
    pairs = []
    for i in range(n):
        alpha = N_ALPHABETS[i % len(N_ALPHABETS)]
        t = _seq(rng, alpha, length, _n_weights(alpha, i % 2 == 1))
        p = _mutate(rng, t, rng.uniform(err_lo, err_hi), alpha)
        if not pair_flagged(p, t):                    # sparse N: make sure the pair has one
            at = rng.randrange(len(t))
            t = t[:at] + "N" + t[at + 1:]
        pairs.append((p, t) if i % 3 else (t, p))
    return _finish(rng, pairs)


def n_homopolymers(seed, n, flank, run_max):
    """An N run between two ACG flanks, of a different length on each side: where the gap goes in the run ties."""
    rng = random.Random(seed)
    pairs = []
    for i in range(n):
        a, b = _seq(rng, "ACG", rng.randint(0, flank)), _seq(rng, "ACG", rng.randint(0, flank))
        k = rng.randint(1, run_max)
        d = rng.randint(1, max(1, k // 3 + 2))
        p, t = a + "N" * k + b, _mutate(rng, a, 0.03, "ACG") + "N" * (k + d) + b
        pairs.append((p, t) if i % 2 else (t, p))
    return _finish(rng, pairs)


def n_tandem_repeats(seed, n, copies_max):
    """Tandem repeats of a short N-rich unit with a different copy number on each side (ties between gap placements)."""
    rng = random.Random(seed)
    units = ["NA", "NNC", "NAG", "NNNT", "GNN", "ANCN", "NG"]
    pairs = []
    for i in range(n):
        u = units[i % len(units)]
        c = rng.randint(4, copies_max)
        d = rng.randint(1, 4)
        a, b = _seq(rng, "ACG" if "T" not in u else "ACT", rng.randint(0, 30)), _seq(rng, "ACG" if "T" not in u else "ACT", 20)
        p, t = a + u * c + b, a + u * (c + d) + b
        if i % 3 == 2:
            t = _mutate(rng, t, 0.03, sorted(set(u + a + b)))
        pairs.append((p, t) if i % 2 else (t, p))
    return _finish(rng, pairs)


def all_n():
    """All-N against all-N: score 0 for equal lengths, one gap otherwise (lengths around the 4-byte groups)."""
    rng = random.Random(0xA11)
    lens = [1, 2, 3, 4, 5, 7, 8, 9, 31, 32, 33, 150]
    pairs = [("N" * k, "N" * k) for k in lens] + [("N" * 40, "N" * 47), ("N" * 9, "N" * 4), ("N" * 3, "N" * 64)]
    return _finish(rng, pairs)


def n_positions():
    """A single N at the first and last base and at every position of a 4-byte group, the final partial group too, in
    the pattern or in the text (the other sequence over ACG, equal or with one substitution)."""
    rng = random.Random(0x905)
    pairs = []
    for length in (8, 9, 10, 11, 150, 151, 153):
        for pos in sorted({0, 1, 2, 3, length - 4, length - 3, length - 2, length - 1}):
            base = _seq(rng, "ACG", length)
            withn = base[:pos] + "N" + base[pos + 1:]
            other = base if pos % 2 else _mutate(rng, base, 0.1, "ACG")
            pairs.append((withn, other) if (pos + length) % 2 else (other, withn))
    return _finish(rng, pairs)


def tiny():
    """"N" against "N", "" against "N", and one-base pairs."""
    rng = random.Random(0x717)
    pairs = [("N", "N"), ("", "N"), ("N", ""), ("N", "A"), ("C", "N"), ("N", "NN"), ("NN", "N"), ("N", "ACG"), ("GAT", "N")]
    return _finish(rng, pairs)


def one_sided_gaps(seed, n, length, gap_lo, gap_hi):
    """A long insertion or deletion in one sequence of an N-bearing pair."""
    rng = random.Random(seed)
    pairs = []
    for i in range(n):
        alpha = N_ALPHABETS[i % len(N_ALPHABETS)]
        s = _seq(rng, alpha, length, _n_weights(alpha, True))
        at = rng.randint(0, length)
        g = _seq(rng, alpha, rng.randint(gap_lo, gap_hi), _n_weights(alpha, i % 2 == 1))
        if not pair_flagged(s, s):
            s = "N" + s[1:]
        pairs.append((s, s[:at] + g + s[at:]) if i % 2 else (s[:at] + g + s[at:], s))
    return _finish(rng, pairs)


def ytgc(seed, n, length):
    """Flagged pairs without any N: sequences over Y, T, G, C in which some aligned group holds Y, T and G or C."""
    rng = random.Random(seed)
    pairs = []
    for i in range(n):
        t = _seq(rng, "YTGC", length)
        if not packer_flags(t):
            g = 4 * rng.randrange(len(t) // 4)
            t = t[:g] + "YTGC" + t[g + 4:]
        p = _mutate(rng, t, 0.06, "YTGC")
        pairs.append((p, t) if i % 2 else (t, p))
    return _finish(rng, pairs)


def five_symbol(seed, n, length):
    """ACGT reads with a few Ns: five distinct bytes, no twin."""
    rng = random.Random(seed)
    pairs = []
    for _ in range(n):
        t = _seq(rng, ACGT, length)
        p = _mutate(rng, t, 0.05, ACGT)
        p, t = list(p), list(t)
        for s in (p, t):
            for _ in range(rng.randint(1, 4)):
                s[rng.randrange(len(s))] = "N"
        pairs.append(("".join(p), "".join(t)))
    return _finish(rng, pairs)


def long_pair():
    """One pair of 33 kbp with Ns (beyond the int16 offsets: the large tier) and its twin."""
    rng = random.Random(0x10A6)
    t = _seq(rng, "ACGN", 33000, _n_weights("ACGN", True))
    return _finish(rng, [(_mutate(rng, t, 0.01, "ACGN"), t)])


def _join(*parts):
    pairs, twins = [], []
    for p, t in parts:
        pairs += p
        twins += t
    return pairs, twins


def short_group():
    """Pairs of at most 1024 bases (the warp tier can take them)."""
    return _join(mutated_reads(0xB150, 32, 150, 0.01, 0.08), n_homopolymers(0xB151, 10, 40, 30), n_tandem_repeats(0xB152, 8, 20),
                 all_n(), n_positions(), tiny(), one_sided_gaps(0xB153, 4, 150, 40, 120), ytgc(0xB154, 6, 150),
                 five_symbol(0xB155, 4, 150))


def mid_group():
    """1 kbp and 3-5 kbp reads, long N runs and repeats, long one-sided gaps (CTA tier).  Gaps of 20-200 bases in 800 bp
    make the adaptive band re-centre on diagonals that tie for the smallest distance to the target."""
    rng = random.Random(0xB1C0)
    reads = [mutated_reads(0xB1C1, 16, 1000, 0.02, 0.10)]
    reads += [mutated_reads(0xB1C2 + i, 1, rng.randint(3000, 5000), 0.01, 0.06) for i in range(4)]
    return _join(*reads, n_homopolymers(0xB1C8, 6, 500, 200), n_tandem_repeats(0xB1C9, 6, 120),
                 one_sided_gaps(0xB1CA, 4, 1200, 200, 600), one_sided_gaps(0xB1D0, 8, 800, 20, 200), ytgc(0xB1CB, 2, 1500),
                 five_symbol(0xB1CC, 3, 1000))


def cli_group():
    """Short pairs with both sequences non-empty (the .seq file format has no empty sequence lines)."""
    pairs, twins = short_group()
    keep = [i for i, (p, t) in enumerate(pairs) if p and t]
    return [pairs[i] for i in keep], [twins[i] for i in keep]


GROUPS = {"short": short_group, "mid": mid_group, "long": long_pair, "cli": cli_group}


def batch(group):
    """Originals and twins of a group alternating in one batch -> (pairs, kinds); kinds[i] is "orig", "twin" or "five"
    (an original without a twin); the twin of an original at i sits at i + 1."""
    pairs, twins = GROUPS[group]()
    out, kinds = [], []
    for pt, tw in zip(pairs, twins):
        out.append(pt)
        kinds.append("orig" if tw else "five")
        if tw:
            out.append(tw)
            kinds.append("twin")
    return out, kinds
