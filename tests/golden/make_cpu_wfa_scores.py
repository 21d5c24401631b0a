#!/usr/bin/env python3
"""Writes cpu_wfa_scores.json: the exact gap-affine scores of the GPU tests' workloads, computed on the CPU.

The GPU tests check every score of these workloads against an exact CPU aligner.  Storing the scores keeps
the tests self-contained.  Pairs of A/C/G/T up to 32767 bases are scored by the oracle (oracle/, the
restatement of the reference aligner that tests/test_oracle_ref.py pins to the reference's CPU WFA).
Pairs with other bytes, or longer than the oracle's int16 offsets allow, are scored by `gotoh` below
(byte equality, as the reference's CPU WFA compares them); the script checks `gotoh` against the oracle first.
Workloads of up to 2000 pairs are stored score by score, larger ones as a sample plus a SHA-256 of the
whole list (little-endian int32).  Needs the built library and oracle (`python __graft_entry__.py`).

usage: make_cpu_wfa_scores.py [workload ...]    (default: all; others are kept from the existing file)
"""
import hashlib
import json
import os
import sys
from multiprocessing import Pool

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
for d in ("oracle", os.path.join("wfa-gpu_b200", "python"), "tests"):
    sys.path.insert(0, os.path.join(ROOT, d))
OUT = os.path.join(HERE, "cpu_wfa_scores.json")

# name -> (synth_aligner specs, seed, penalties); "non_acgt" is util.non_acgt_pairs()
WORKLOADS = {
    "config1": ([(10000, 150, 0.02, 0.02)], 0xB2000001, (2, 3, 1)),
    "config2": ([(1000000, 150, 0.05, 0.05)], 0xB2000002, (2, 3, 1)),
    "config3": ([(100000, 1000, 0.10, 0.10)], 0xB2000003, (2, 3, 1)),
    "headline": ([(8192, 10000, 0.05, 0.05)], 0xB2000004, (2, 3, 1)),
    "non_acgt": (None, None, (2, 3, 1)),
    "longer_than_32767": ([(4, 50000, 0.15, 0.15), (4, 40000, 0.03, 0.03)], 0xB2004000, (2, 3, 1)),
    "config5_64": ([(64, 50000, 0.15, 0.15)], 0xB2000005, (2, 3, 1)),
}
for _pen in ((4, 6, 2), (3, 1, 4), (2, 10, 5), (5, 3, 2)):
    WORKLOADS["long_reads_%d_%d_%d" % _pen] = ([(1536, 5000, 0.02, 0.08)], 0xB2000040 + _pen[2], _pen)
FULL_LIST_MAX = 2000
SAMPLE = 500


def gotoh(p, t, x, o, e):
    """Exact gap-affine score (mismatch x, gap of length L costs o + L * e), one DP row at a time."""
    pb, tb = np.frombuffer(p.encode(), np.uint8), np.frombuffer(t.encode(), np.uint8)
    n = len(tb)
    if len(pb) == 0 or n == 0:
        return o + e * (len(pb) + n) if len(pb) + n else 0
    big = np.int64(1) << 40
    j = np.arange(n + 1, dtype=np.int64)
    H = o + e * j
    H[0] = 0
    D = np.full(n + 1, big, np.int64)
    for i in range(1, len(pb) + 1):
        D = np.minimum(H + (o + e), D + e)                                      # gap in the text (down)
        Hn = np.empty_like(H)
        Hn[0] = o + e * i
        Hn[1:] = np.minimum(H[:-1] + np.where(tb == pb[i - 1], 0, x), D[1:])
        # gap in the pattern (right): I[j] = min_{k < j} Hn[k] + o + e (j - k)
        run = np.minimum.accumulate(Hn - e * j)
        Hn[1:] = np.minimum(Hn[1:], run[:-1] + o + e * j[1:])
        H = Hn
    return int(H[n])


_cache = {}


def _pairs(name):
    if name not in _cache:
        import util
        specs, seed, _ = WORKLOADS[name]
        if specs is None:
            _cache[name] = util.non_acgt_pairs()[0]
        else:
            a = util.synth_aligner(specs, seed)
            _cache[name] = a
    return _cache[name]


def _score_range(job):
    name, lo, hi = job
    from oracle import Oracle
    orc = Oracle()
    x, o, e = WORKLOADS[name][2]
    src = _pairs(name)
    out = []
    for i in range(lo, hi):
        p, t = src[i] if isinstance(src, list) else src.pair(i)
        if max(len(p), len(t)) <= 32767 and not (set(p) | set(t)) - set("ACGT"):
            r = orc.align(p, t, x, o, e, 100000, cigar=False)
            assert r["finished"], (name, i)
            out.append(r["distance"])
        else:
            out.append(gotoh(p, t, x, o, e))
    return out


def self_check():
    import util
    from oracle import Oracle
    orc = Oracle()
    a = util.synth_aligner([(6, 300, 0.05, 0.15), (3, 1200, 0.02, 0.10)], 0xB20C0DE)
    for pen in ((2, 3, 1), (4, 6, 2), (3, 1, 4), (2, 10, 5)):
        for i in range(a.num_pairs):
            p, t = a.pair(i)
            assert gotoh(p, t, *pen) == orc.align(p, t, *pen, 100000, cigar=False)["distance"], (pen, i)
    for p, t in (("", "ACGT"), ("ACG", ""), ("", ""), ("ACGT", "ACGT"), ("A", "C")):
        assert gotoh(p, t, 2, 3, 1) == orc.align(p, t, 2, 3, 1, 1000, cigar=False)["distance"], (p, t)


def main(names):
    self_check()
    data = {}
    if os.path.exists(OUT):
        with open(OUT) as f:
            data = json.load(f)
    with Pool(os.cpu_count()) as pool:
        for name in names:
            src = _pairs(name)
            n = len(src) if isinstance(src, list) else src.num_pairs
            step = max(1, min(2000, n // (4 * os.cpu_count())))
            jobs = [(name, lo, min(n, lo + step)) for lo in range(0, n, step)]
            scores = [s for part in pool.map(_score_range, jobs, chunksize=1) for s in part]
            _cache.pop(name, None)
            if n <= FULL_LIST_MAX:
                data[name] = {"n": n, "penalties": list(WORKLOADS[name][2]), "scores": scores}
            else:
                k = n // SAMPLE
                data[name] = {"n": n, "penalties": list(WORKLOADS[name][2]), "every": k, "sample": scores[::k],
                              "sha256": hashlib.sha256(np.asarray(scores, dtype="<i4").tobytes()).hexdigest()}
            print(name, n, "pairs, max score", max(scores), flush=True)
    with open(OUT, "w") as f:
        json.dump({k: data[k] for k in sorted(data)}, f, separators=(",", ":"))
        f.write("\n")


if __name__ == "__main__":
    main(sys.argv[1:] or list(WORKLOADS))
