"""Large tier: wavefront rings in global memory with int32 offsets (wavefronts wider than an
SM's shared memory, sequences >= 32768 bases -- BASELINE config 5's shape, which the reference
GPU path cannot run at all: lib/wfa_types.h:28-32)."""
import os
import subprocess
import sys

import pytest

from util import cpu_wfa_scores, synth_aligner

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_forced_large_tier_is_bit_exact_vs_oracle():
    env = dict(os.environ, WFAGPU_FORCE_LARGE="1")
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "large_tier_check.py")], env=env,
                        capture_output=True, text=True, timeout=1200)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]


def test_wide_wavefront_falls_into_large_tier(oracle):
    # 10 kbp at 30 % error: score ~ 7000 -> rings of ~14000 diagonals do not fit 227 KB
    a = synth_aligner([(6, 10000, 0.30, 0.30)], 0xB2003000)
    assert a.initialize_parameters(2, 3, 1)
    a.options.compute_cigar = True
    a.options.max_error = 9000
    a.align()
    for i in range(a.num_pairs):
        p, t = a.pair(i)
        r = oracle.align(p, t, 2, 3, 1, 9000)
        assert r["finished"]
        assert (a.error(i), a.cigar(i)) == (r["distance"], r["cigar"])


def test_sequences_longer_than_32767(oracle):
    # config 5 shape (50 kbp Nanopore-like, 15 % error), initial budget deliberately too small so
    # that every pair is re-dispatched on the GPU; parity = CPU WFA score + valid CIGAR of that score
    a = synth_aligner([(4, 50000, 0.15, 0.15), (4, 40000, 0.03, 0.03)], 0xB2004000)
    assert a.initialize_parameters(2, 3, 1)
    a.options.compute_cigar = True
    a.options.max_error = 2000
    a.align()
    pairs = [a.pair(i) for i in range(a.num_pairs)]
    errs = cpu_wfa_scores("longer_than_32767")["scores"]
    assert len(errs) == len(pairs)
    for i, (p, t) in enumerate(pairs):
        assert a.error(i) == errs[i]
        assert oracle.cigar_score(p, t, a.cigar(i), 2, 3, 1) == errs[i]
    assert a.run_stats()["redispatched"] >= a.num_pairs


def test_config5_shape_on_64_pairs_matches_cpu_wfa(oracle):
    # BASELINE config 5 (50 kbp, 15 %, CIGAR, first budget 8000 below every score: every pair is re-dispatched on the GPU
    # with a bound-guided budget) on 64 pairs: every score == the stored exact score of the CPU WFA, every CIGAR an alignment of
    # exactly that cost; the re-dispatched pass runs wfa_quadg_kernel (int32 rings in L2)
    a = synth_aligner([(64, 50000, 0.15, 0.15)], 0xB2000005)
    assert a.initialize_parameters(2, 3, 1)
    a.options.compute_cigar = True
    a.options.max_error = 8000
    a.align()
    st = a.run_stats()
    assert st["redispatched"] == 64 and st["failed_pairs"] == 0
    pairs = [a.pair(i) for i in range(a.num_pairs)]
    errs = cpu_wfa_scores("config5_64")["scores"]
    assert a.errors() == errs
    for i, (p, t) in enumerate(pairs):
        assert oracle.cigar_score(p, t, a.cigar(i), 2, 3, 1) == errs[i]
