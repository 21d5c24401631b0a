"""Ends-free alignment on the GPU: every score equals the exact ends-free DP, every CIGAR equals the CPU model of the
kernel path (tests/endsfree_model.py) byte for byte and aligns both full sequences at a span cost equal to its score,
and the kernel variants, the host decoder and two workers per GPU print the same bytes."""
import ctypes as C
import json
import os
import re
import subprocess
import sys
from multiprocessing import Pool

import numpy as np
import pytest

import wfagpu
from endsfree_check import CONFIGS, batch, key, run
from endsfree_ref import gotoh_span, rand_seq, mutate, span_cost_ok
import endsfree_model

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _dp(args):
    return gotoh_span(*args)


def _run_check(tmp_path, name, env):
    out = tmp_path / (name + ".json")
    e = dict(os.environ)
    e.update(env)
    subprocess.run([sys.executable, os.path.join(HERE, "endsfree_check.py"), str(out)], check=True, env=e, timeout=900)
    return json.loads(out.read_text())


@pytest.fixture(scope="module")
def base(tmp_path_factory):
    return _run_check(tmp_path_factory.mktemp("ef"), "base", {})


@pytest.fixture(scope="module")
def dp_scores():
    pairs = batch()
    jobs = [(p, t) + pen + (span,) for pen, span, cigar in CONFIGS for p, t in pairs]
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        flat = pool.map(_dp, jobs, chunksize=4)
    out, i = {}, 0
    for pen, span, cigar in CONFIGS:
        out[key(pen, span, cigar)] = flat[i:i + len(pairs)]
        i += len(pairs)
    return out


def test_scores_equal_the_dp(base, dp_scores):
    for k, want in dp_scores.items():
        got = base[k]["scores"]
        bad = [(i, g, w) for i, (g, w) in enumerate(zip(got, want)) if g != w]
        assert not bad, (k, bad[:5])


def test_cigars_cover_both_sequences_at_the_score(base, lib):
    pairs = batch()
    for pen, span, cigar in CONFIGS:
        if not cigar:
            continue
        r = base[key(pen, span, cigar)]
        for i, (p, t) in enumerate(pairs):
            assert span_cost_ok(lib, p, t, *pen, span, r["scores"][i], r["cigars"][i]), (pen, span, i, r["cigars"][i][:80])


def _model(args):
    from oracle import Oracle
    p, t, pen, span = args
    m = endsfree_model.align(Oracle(), p, t, *pen, span, max_steps=20000)     # 5 kbp pairs at (2,24,9) score ~6000
    return m["distance"], m["cigar"]


def test_cigars_equal_the_model(base):
    pairs = batch()
    cfgs = [(pen, span) for pen, span, cigar in CONFIGS if cigar]
    jobs = [(p, t, pen, span) for pen, span in cfgs for p, t in pairs]
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        flat = pool.map(_model, jobs, chunksize=2)
    for c, (pen, span) in enumerate(cfgs):
        r = base[key(pen, span, True)]
        want = flat[c * len(pairs):(c + 1) * len(pairs)]
        bad = [(i, r["cigars"][i][:60], w[1][:60]) for i, w in enumerate(want) if (r["scores"][i], r["cigars"][i]) != w]
        assert not bad, (pen, span, bad[:4])


def test_score_only_equals_the_cigar_runs(base):
    for span in ((0, 0, 20, 20), (3, 7, 11, 2)):
        assert base[key((2, 3, 1), span, False)]["scores"] == base[key((2, 3, 1), span, True)]["scores"]


# (ends-free batches always take the decision-byte traceback: the snapshot switches select nothing for them)
VARIANTS = {
    "force_large": {"WFAGPU_FORCE_LARGE": "1"},
    "warp_kernel": {"WFAGPU_WARP_KERNEL": "1"},
    "no_bound": {"WFAGPU_NO_BOUND": "1"},
    "force_bound": {"WFAGPU_FORCE_BOUND": "1"},
    "redispatch": {"EF_MAX_ERROR": "20"},
    "host_cigar": {"WFAGPU_HOST_CIGAR": "1"},
    "two_workers": {"WFAGPU_DEVICES": "0,0", "EF_BATCH": "16"},
}


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_variants_print_the_same_bytes(base, tmp_path, name):
    got = _run_check(tmp_path, name, VARIANTS[name])
    for k in base:
        assert got[k] == base[k], (name, k)


def test_pair_longer_than_32767():
    rng = np.random.default_rng(0xEF32)
    core = rand_seq(rng, 33000)
    p, t = mutate(rng, core, 0.01), rand_seq(rng, 200) + core + rand_seq(rng, 150)
    span = (0, 0, 200, 200)
    r = run([(p, t)], (2, 3, 1), span, True, max_error=2000)
    assert r["scores"][0] == gotoh_span(p, t, 2, 3, 1, span)
    assert span_cost_ok(wfagpu.load(), p, t, 2, 3, 1, span, r["scores"][0], r["cigars"][0])
    assert (r["scores"][0], r["cigars"][0]) == _model((p, t, (2, 3, 1), span))


def test_check_correctness_recomputes_under_the_span():
    pairs = batch()
    a = wfagpu.Aligner()
    for p, t in pairs:
        a.add_sequences(p, t)
    a.initialize_parameters(2, 3, 1)
    a.options.max_error = 400
    sp = wfagpu.Span(0, 30, 25, 0)
    a.L.wfagpu_launch_alignments_span(a.s.sequences_buffer, a.s.sequences_buffer_len, a.s.sequences_metadata,
                                      a.s.results, a.s.alignment_options, True, True, C.byref(sp))
    st = a.run_stats()
    assert st["checked"] == len(pairs) and st["incorrect"] == 0, st
    assert a.L.wfagpu_last_launch_ok()


def test_zero_span_is_global_alignment():
    pairs = batch()
    g = run(pairs, (2, 3, 1), None, True)
    z = run(pairs, (2, 3, 1), (0, 0, 0, 0), True)
    assert g == z


@pytest.mark.parametrize("span,band", [((0, 0, 20, 20), 10), ((0, -1, 0, 0), 0)])
def test_band_or_negative_values_fail_cleanly(span, band):
    a = wfagpu.Aligner()
    for p, t in batch()[:8]:
        a.add_sequences(p, t)
    a.initialize_parameters(2, 3, 1)
    a.options.compute_cigar = True
    a.options.band = band
    with pytest.raises(RuntimeError):
        a.align(ends_free=span)
    assert a.errors() == [0] * 8 and not any(a.cigars())


def test_cli_ends_free(tmp_path):
    pairs = batch()[:33] + batch()[-6:-1]
    seq = tmp_path / "ef.seq"
    seq.write_text("".join(f">{p}\n<{t}\n" for p, t in pairs))
    binary = os.path.join(os.path.dirname(HERE), "bin", "wfa.affine.gpu")
    outs = []
    for extra in ([], ["-S", "10"]):
        out = tmp_path / ("out%d.txt" % len(outs))
        pr = subprocess.run([binary, "-i", str(seq), "-F", "0,30,25,0", "-x", "-c", "-e", "400", "-o", str(out)] + extra,
                            capture_output=True, text=True, timeout=600)
        assert pr.returncode == 0, pr.stderr[-3000:]
        counts = re.findall(r"Incorrect=(\d+)", pr.stderr)
        assert counts and set(counts) == {"0"}, pr.stderr[-3000:]
        outs.append(out.read_text())
    assert outs[0] == outs[1]
    rows = [l.split("\t") for l in outs[0].splitlines()]
    assert [-int(r[0]) for r in rows] == [gotoh_span(p, t, 2, 3, 1, (0, 30, 25, 0)) for p, t in pairs]
    pr = subprocess.run([binary, "-i", str(seq), "-F", "0,30,25,0", "-B", "auto"], capture_output=True, text=True, timeout=600)
    assert pr.returncode != 0 and "cannot be combined" in pr.stderr
