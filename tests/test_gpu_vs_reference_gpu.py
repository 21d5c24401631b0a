"""Bit-exact CIGAR parity against the reference's own GPU path: the unmodified
reference (built for sm_100 into oracle/_ref/gpu) and our library run on the same
synthetic pairs on the same B200; scores and CIGAR text must be identical, and the
oracle (restatement) must agree with both -- this is what pins the oracle's CIGARs.
Where the reference binary is not built, every pair is compared with the oracle's
restatement of the reference GPU path instead."""
import pytest

import refgpu
from util import synth_aligner

pytestmark = pytest.mark.gpu


def reference_gpu(oracle, pairs, pen, max_error, band=None, window=None):
    """[(score, CIGAR)] of the reference GPU path: its binary where built, else the oracle's restatement of it."""
    if refgpu.available():
        return refgpu.run(pairs, pen, max_error, cigar=True, band=band, threads=window)[0]
    out = []
    for p, t in pairs:
        r = oracle.align(p, t, *pen, max_error, band=band or -1, window=window or 0)
        assert r["finished"]            # the specs give budgets the reference's GPU kernels finish with
        out.append((r["distance"], r["cigar"]))
    return out


def ours(specs, pen, max_error, seed):
    a = synth_aligner(specs, seed)
    assert a.initialize_parameters(*pen)
    a.options.compute_cigar = True
    a.options.max_error = max_error
    a.align()
    return a


@pytest.mark.parametrize("specs,pen,max_error", [
    ([(3000, 150, 0.02, 0.02)], (2, 3, 1), 50),          # config 1 shape
    ([(600, 1000, 0.10, 0.10)], (2, 3, 1), 700),          # config 3 shape (budget large enough: no CPU fallback in the reference)
    ([(48, 10000, 0.01, 0.05)], (2, 3, 1), 3000),         # config 4 shape
    ([(300, 400, 0.08, 0.08)], (5, 3, 2), 600),
    ([(300, 400, 0.08, 0.08)], (4, 6, 2), 900),
])
def test_cigars_identical_to_reference_gpu(oracle, specs, pen, max_error):
    a = ours(specs, pen, max_error, 0xB2001000)
    pairs = [a.pair(i) for i in range(a.num_pairs)]
    ref = reference_gpu(oracle, pairs, pen, max_error)
    assert len(ref) == len(pairs)
    diff = [(i, a.error(i), ref[i][0]) for i in range(len(pairs)) if a.error(i) != ref[i][0]]
    assert diff == []
    diff = [(i, a.cigar(i)[:60], ref[i][1][:60]) for i in range(len(pairs)) if a.cigar(i) != ref[i][1]]
    assert diff == []
    # and the CPU restatement says the same on a sample
    step = max(1, len(pairs) // 40)
    for i in range(0, len(pairs), step):
        r = oracle.align(*pairs[i], *pen, max_error)
        assert (r["distance"], r["cigar"]) == ref[i]


@pytest.mark.parametrize("specs,pen,max_error,band,window", [
    ([(48, 10000, 0.01, 0.05)], (2, 3, 1), 3000, 25, 512),     # config 4: -e 3000 -x -B auto -t 512
    ([(400, 1000, 0.10, 0.10)], (2, 3, 1), 800, 25, 128),
    ([(400, 1000, 0.10, 0.10)], (2, 3, 1), 800, 10, 64),
])
def test_banded_identical_to_reference_gpu(oracle, specs, pen, max_error, band, window):
    a = synth_aligner(specs, 0xB2002000)
    assert a.initialize_parameters(*pen)
    a.options.compute_cigar = True
    a.options.max_error = max_error
    a.options.band = band
    a.options.threads_per_block = window
    a.align()
    pairs = [a.pair(i) for i in range(a.num_pairs)]
    ref = reference_gpu(oracle, pairs, pen, max_error, band=band, window=window)
    diff = [(i, a.error(i), ref[i][0]) for i in range(len(pairs)) if (a.error(i), a.cigar(i)) != ref[i]]
    assert diff == []
