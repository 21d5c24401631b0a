"""GPU parity: the CUDA path through the public C API vs the oracle (bit-exact
scores and CIGAR text).  Needs a B200; run with -m gpu."""
import os

import pytest

import wfagpu
from util import assert_cpu_wfa_scores, check_against_oracle, cpu_wfa_scores, non_acgt_pairs, synth_aligner

pytestmark = pytest.mark.gpu


def run(specs, pen, cigar, max_error=None, batch=None, seed=0xB2000000):
    a = synth_aligner(specs, seed)
    assert a.initialize_parameters(*pen)
    a.options.compute_cigar = cigar
    if max_error is not None:
        a.options.max_error = max_error
    if batch is not None:
        a.set_batch_size(batch)
    a.align()
    return a


@pytest.mark.parametrize("cigar", [False, True])
def test_short_reads_150bp(oracle, cigar):
    # BASELINE config 1 shape: 150 bp, 2 % error, x=2,o=3,e=1 (and 5 % for config 2)
    a = run([(2000, 150, 0.02, 0.02), (2000, 150, 0.05, 0.05)], (2, 3, 1), cigar)
    assert check_against_oracle(oracle, a, 2, 3, 1, a.options.max_error, cigar) == []


@pytest.mark.parametrize("cigar", [False, True])
def test_1kbp_10pct_with_redispatch(oracle, cigar):
    # config 3 shape: default budget 300 leaves ~5 % of the pairs over budget -> GPU re-dispatch
    a = run([(400, 1000, 0.10, 0.10)], (2, 3, 1), cigar)
    assert a.options.max_error == 300
    assert check_against_oracle(oracle, a, 2, 3, 1, 300, cigar) == []


def test_10kbp_cigar(oracle):
    # headline shape: 10 kbp, 5 % error, -e 3000, CIGAR
    a = run([(64, 10000, 0.05, 0.05)], (2, 3, 1), True, max_error=3000)
    assert check_against_oracle(oracle, a, 2, 3, 1, 3000, True) == []


@pytest.mark.parametrize("pen", [(1, 2, 1), (3, 1, 4), (5, 3, 2), (4, 6, 2), (2, 10, 5), (3, 5, 2)])
def test_penalty_sets(oracle, pen):
    a = run([(200, 150, 0.05, 0.05), (60, 700, 0.08, 0.08), (100, 30, 0.3, 0.3)], pen, True, max_error=400)
    assert check_against_oracle(oracle, a, *pen, 400, True) == []


def test_multi_batch_matches_single_batch(oracle):
    a = run([(1000, 200, 0.04, 0.04)], (2, 3, 1), True, batch=1000)
    b = run([(1000, 200, 0.04, 0.04)], (2, 3, 1), True, batch=130)
    assert a.errors() == b.errors()
    assert a.cigars() == b.cigars()


def test_edge_cases(oracle):
    a = wfagpu.Aligner()
    cases = [("ACGT", "ACGT"), ("A", "A"), ("A", "C"), ("", "ACGT"), ("ACGT", ""), ("", ""),
             ("ACGTACGTACGT", "ACGT"), ("ACGT", "ACGTACGTACGTTTTT"), ("AAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAAA", "A"),
             ("ACGTNACGT", "ACGTNACGT"), ("ACGTNACGT", "ACGTACGT"), ("acgtacgt", "ACGTACGT"),
             ("ACGTRYACGT", "ACGTRYACGT")]
    for p, t in cases:
        assert a.add_sequences(p, t)
    assert a.initialize_parameters(2, 3, 1)
    a.options.compute_cigar = True
    a.align()
    for i, (p, t) in enumerate(cases):
        if oracle.has_N(p) or oracle.has_N(t):
            # the reference sends these to CPU WFA (byte equality): check score + CIGAR validity
            sc = oracle.cigar_score(p, t, a.cigar(i), 2, 3, 1)
            assert sc == a.error(i), (p, t, a.cigar(i))
            continue
        r = oracle.align(p, t, 2, 3, 1, 200)
        assert r["finished"]
        assert (a.error(i), a.cigar(i)) == (r["distance"], r["cigar"]), (p, t)


def run_banded(specs, pen, cigar, band, window, max_error, seed=0xB2000000):
    a = synth_aligner(specs, seed)
    assert a.initialize_parameters(*pen)
    a.options.compute_cigar = cigar
    a.options.max_error = max_error
    a.options.band = band
    a.options.threads_per_block = window
    a.align()
    return a


@pytest.mark.parametrize("cigar", [False, True])
@pytest.mark.parametrize("specs,pen,band,window,max_error", [
    ([(24, 10000, 0.01, 0.05)], (2, 3, 1), 25, 512, 3000),      # config 4: -B auto -t 512
    ([(300, 1000, 0.10, 0.10)], (2, 3, 1), 25, 128, 800),       # narrow band: recall < 100 %
    ([(300, 1000, 0.10, 0.10)], (2, 3, 1), 10, 64, 800),
    ([(200, 700, 0.08, 0.08)], (5, 3, 2), 25, 96, 1200),
    ([(200, 700, 0.08, 0.08)], (4, 6, 2), 50, 128, 1500),       # gcd > 1: null steps, stale ring slots
])
def test_banded_equals_oracle(oracle, cigar, specs, pen, band, window, max_error):
    a = run_banded(specs, pen, cigar, band, window, max_error)
    bad = []
    n_subopt = 0
    for i in range(a.num_pairs):
        p, t = a.pair(i)
        r = oracle.align(p, t, *pen, max_error, band=band, window=window, cigar=cigar)
        assert r["finished"]
        if a.error(i) != r["distance"] or (cigar and a.cigar(i) != r["cigar"]):
            bad.append((i, a.error(i), r["distance"]))
        if cigar:
            # the heuristic may be sub-optimal, but the CIGAR must describe a real alignment of that score
            assert oracle.cigar_score(p, t, a.cigar(i), *pen) == a.error(i)
        exact = oracle.align(p, t, *pen, max_error, cigar=False)
        n_subopt += exact["distance"] != a.error(i)
    assert bad == []
    assert n_subopt <= a.num_pairs // 2


def test_multi_gpu_sharding_matches_single_gpu(lib):
    import ctypes as C
    n = C.c_int(0)
    lib.get_num_cuda_devices(C.byref(n))
    if n.value < 2:
        pytest.skip("needs >= 2 GPUs (gpurun --gpus 2)")
    specs = [(3000, 300, 0.05, 0.05), (200, 3000, 0.05, 0.05)]
    wfagpu.set_devices("0")
    a = run(specs, (2, 3, 1), True, max_error=600, batch=400)
    wfagpu.set_devices("all")
    b = run(specs, (2, 3, 1), True, max_error=600, batch=400)
    st = b.run_stats()
    wfagpu.set_devices("0")
    assert st["devices"] >= 2
    assert a.errors() == b.errors()
    assert a.cigars() == b.cigars()


def test_host_and_device_cigar_text_agree(oracle, monkeypatch):
    specs = [(500, 150, 0.05, 0.05), (100, 1500, 0.08, 0.08), (8, 10000, 0.05, 0.05)]
    a = run(specs, (2, 3, 1), True, max_error=3000)                 # text printed by cigar_text_kernel
    launches_dev = a.run_stats()["launches"]
    monkeypatch.setenv("WFAGPU_HOST_CIGAR", "1")
    b = run(specs, (2, 3, 1), True, max_error=3000)                 # text printed by wfagpu_ops_to_cigar
    launches_host = b.run_stats()["launches"]
    monkeypatch.delenv("WFAGPU_HOST_CIGAR")
    assert a.errors() == b.errors()
    assert a.cigars() == b.cigars()
    assert launches_dev > launches_host


@pytest.mark.parametrize("variant", [{"WFAGPU_FORCE_BOUND": "1"}, {"WFAGPU_NO_BOUND": "1"}, {"WFAGPU_NO_CKPT": "1"},
                                     {"WFAGPU_FORCE_BOUND": "1", "WFAGPU_CK_PERIOD": "7"},
                                     {"WFAGPU_FORCE_BOUND": "1", "WFAGPU_CK_PERIOD": "31"},
                                     {"WFAGPU_FORCE_BOUND": "1", "WFAGPU_NO_HINT": "1"},
                                     {"WFAGPU_FORCE_BOUND": "1", "WFAGPU_ARENA_MB": "8"},
                                     {"WFAGPU_FORCE_BOUND": "1", "WFAGPU_NO_PREBOUND": "1"}, {"WFAGPU_FORCE_BOUND": "1", "WFAGPU_NO_SKIP_OPEN": "1"},
                                     {"WFAGPU_FORCE_BOUND": "1", "WFAGPU_NO_BOUND_ORDER": "1"},
                                     {"WFAGPU_QUAD_MIN": "1"}, {"WFAGPU_QUAD_MIN": "1", "WFAGPU_FORCE_BOUND": "1", "WFAGPU_CK_PERIOD": "31"},
                                     {"WFAGPU_QUAD_MIN": "1", "WFAGPU_QUAD_PAIRS": "1"},
                                     {"WFAGPU_QUAD_MIN": "1", "WFAGPU_QUAD_PAIRS": "1", "WFAGPU_FORCE_BOUND": "1", "WFAGPU_CK_PERIOD": "7"},
                                     {"WFAGPU_NO_QUAD": "1"}, {"WFAGPU_NO_BAND_TB": "1"}, {"WFAGPU_FORCE_LARGE": "1"}, {"WFAGPU_FORCE_LARGE": "1", "WFAGPU_NO_QUAD": "1"}])
def test_kernel_variants_are_bit_exact(variant):
    # per-pair score bounds on/off, bounds before or inside the pass, queue in bound or length order, unbounded pairs skipping
    # the first pass or not, ring snapshots vs decision bytes, snapshot periods, four diagonals per thread (forced for
    # every ring width with WFAGPU_QUAD_MIN=1) vs one, one or two scores per barrier interval, the large tier: one result
    import subprocess, sys as _sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    pr = subprocess.run([_sys.executable, os.path.join(root, "tests", "variant_check.py")], env=dict(os.environ, **variant),
                        capture_output=True, text=True, timeout=1500)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]


@pytest.mark.parametrize("pen,length,err,max_error", [((2, 250, 3), 400, 0.05, 2000), ((2, 250, 3), 3000, 0.03, 40), ((3, 120, 2), 2500, 0.04, 3000)])
def test_penalties_whose_rings_do_not_fit_the_bound_kernel(oracle, pen, length, err, max_error):
    # o + e = 253: the bound kernel's per-warp rings (A + 2 (e + 1) rows of 128 bytes, 8 warps) exceed the shared memory of an SM.
    # No score bounds then: launch-bound pruning only, and over-budget pairs double their budget until they finish.
    a = synth_aligner([(24, length, err, err)], 0xB2007700)
    assert a.initialize_parameters(*pen)
    a.options.compute_cigar = True
    a.options.max_error = max_error
    assert a.align()
    assert a.run_stats()["failed_pairs"] == 0
    for i in range(a.num_pairs):
        p, t = a.pair(i)
        r = oracle.align(p, t, *pen, 60000)
        assert (a.error(i), a.cigar(i)) == (r["distance"], r["cigar"])


def test_headline_batch_at_full_size(oracle):
    # BASELINE's headline configuration at bench.py's full size (8192 x 10 kbp, 5 %, -e 3000, CIGAR),
    # checked through properties that do not need the oracle on every pair:
    #   * every score equals the stored exact score of the CPU WFA (all pairs),
    #   * every CIGAR is an alignment of its two sequences whose gap-affine cost is that score,
    #   * a second call (provisioned from the first one's scores: per-pair bounds, tighter rings,
    #     another CTA per SM) returns byte-identical results,
    #   * a sample equals the oracle's CIGAR text byte for byte.
    a = run([(8192, 10000, 0.05, 0.05)], (2, 3, 1), True, max_error=3000, batch=4096, seed=0xB2000004)
    errs, cigs = a.errors(), a.cigars()
    pairs = [a.pair(i) for i in range(a.num_pairs)]
    assert_cpu_wfa_scores("headline", errs)
    for (p, t), s, c in zip(pairs, errs, cigs):
        assert oracle.cigar_score(p, t, c, 2, 3, 1) == s
    a.reset_results()
    a.align()
    assert a.errors() == errs and a.cigars() == cigs
    for i in range(0, a.num_pairs, 683):
        r = oracle.align(pairs[i][0], pairs[i][1], 2, 3, 1, 3000)
        assert (errs[i], cigs[i]) == (r["distance"], r["cigar"])


@pytest.mark.parametrize("pen", [(4, 6, 2), (3, 1, 4), (2, 10, 5), (5, 3, 2)])
def test_long_reads_with_gap_extension_above_one(oracle, pen):
    # e > 1 exercises the quotient of the score-bound pruning ((Dmax - d) / e), the reachability bound
    # and the snapshot geometry at sizes where bounds, hints and re-provisioning are all active:
    # scores vs the stored exact scores of the CPU WFA, CIGARs must be alignments of exactly that cost,
    # and a sample must equal the oracle's CIGAR text.
    a = run([(1536, 5000, 0.02, 0.08)], pen, True, max_error=6000, batch=512, seed=0xB2000040 + pen[2])
    errs, cigs = a.errors(), a.cigars()
    pairs = [a.pair(i) for i in range(a.num_pairs)]
    assert_cpu_wfa_scores("long_reads_%d_%d_%d" % pen, errs)
    for (p, t), s, c in zip(pairs, errs, cigs):
        assert oracle.cigar_score(p, t, c, *pen) == s
    for i in range(0, a.num_pairs, 191):
        r = oracle.align(pairs[i][0], pairs[i][1], *pen, 6000)
        assert (errs[i], cigs[i]) == (r["distance"], r["cigar"])


def test_banded_pairs_over_budget_are_finished_by_the_exact_kernels(oracle):
    # The reference hands pairs the banded kernel did not finish to the CPU WFA; here they are
    # re-dispatched on the GPU through the exact kernels (a band that lost the alignment does not find
    # it again with a larger budget).  Pairs the banded pass finishes keep the heuristic's result.
    pen, band, window, budget = (2, 3, 1), 10, 64, 120
    a = run_banded([(200, 1000, 0.02, 0.12)], pen, True, band, window, budget)
    n_exact = 0
    for i in range(a.num_pairs):
        p, t = a.pair(i)
        r = oracle.align(p, t, *pen, budget, band=band, window=window, cigar=True)
        if not r["finished"]:
            r = oracle.align(p, t, *pen, 8000, cigar=True)       # exact
            n_exact += 1
        assert r["finished"]
        assert (a.error(i), a.cigar(i)) == (r["distance"], r["cigar"])
    assert 10 < n_exact < a.num_pairs
    assert a.run_stats()["redispatched"] == n_exact


def test_non_acgt_pairs_match_cpu_wfa_scores(oracle):
    # Pairs the packer flags (an 'N' in either sequence, sequence_packing_kernel.cu:54-76) go through the
    # byte-compare kernels, as the reference sends them to its CPU WFA: same byte-equality semantics, so
    # the same optimal score; the CIGAR must be an alignment of that cost.  (Other non-ACGT bytes are not
    # flagged by the reference and are 2-bit encoded as (c & 6) >> 1 on its GPU path -- and here.)
    # Mixed with clean pairs in one batch, small budget so that some flagged pairs are also re-dispatched.
    pairs, dirty = non_acgt_pairs()
    b = wfagpu.Aligner()
    for p, t in pairs:
        assert b.add_sequences(p, t)
    assert b.initialize_parameters(2, 3, 1)
    b.options.compute_cigar = True
    b.options.max_error = 150
    b.align()
    bp = [b.pair(i) for i in range(b.num_pairs)]
    assert bp == pairs
    ref = cpu_wfa_scores("non_acgt")["scores"]
    assert b.errors() == ref
    for i, (p, t) in enumerate(bp):
        assert oracle.cigar_score(p, t, b.cigar(i), 2, 3, 1) == ref[i]
    # every flagged pair is routed to the byte-compare kernels exactly once, re-dispatched or not
    flagged = [i for i, (p, t) in enumerate(bp) if oracle.has_N(p) or oracle.has_N(t)]
    assert flagged and set(flagged) <= set(dirty)
    assert b.run_stats()["ascii_pairs"] == len(flagged)
