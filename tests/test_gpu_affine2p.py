"""Gap-affine 2-piece alignment on the GPU: every score equals the exact 2-piece DP, every CIGAR equals the CPU model
of the kernel path (tests/affine2p_model.py) byte for byte and costs its score, identical pieces print the bytes of
the single-piece path, and the kernel variants, the host decoder and two workers per GPU print the same bytes."""
import ctypes as C
import json
import os
import re
import subprocess
import sys
from multiprocessing import Pool

import numpy as np
import pytest

import affine2p_model
import wfagpu
from affine2p_check import CONFIGS, batch, key, run
from affine2p_ref import cost_ok, gotoh2p, indel_pairs
from endsfree_ref import mutate, rand_seq

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _run_check(tmp_path, name, env):
    out = tmp_path / (name + ".json")
    e = dict(os.environ)
    e.update(env)
    subprocess.run([sys.executable, os.path.join(HERE, "affine2p_check.py"), str(out)], check=True, env=e, timeout=900)
    return json.loads(out.read_text())


@pytest.fixture(scope="module")
def base(tmp_path_factory):
    return _run_check(tmp_path_factory.mktemp("ap"), "base", {})


def _dp(args):
    return gotoh2p(*args)


def _model(args):
    p, t, pen = args
    m = affine2p_model.align(p, t, *pen, max_steps=20000)
    return m["distance"], m["cigar"]


def test_scores_equal_the_dp(base):
    pairs = batch()
    pens = sorted({pen for pen, _ in CONFIGS})
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        flat = pool.map(_dp, [(p, t) + pen for pen in pens for p, t in pairs], chunksize=2)
    for c, pen in enumerate(pens):
        want = flat[c * len(pairs):(c + 1) * len(pairs)]
        for cigar in (True, False):
            if (pen, cigar) in CONFIGS:
                got = base[key(pen, cigar)]["scores"]
                bad = [(i, g, w) for i, (g, w) in enumerate(zip(got, want)) if g != w]
                assert not bad, (pen, cigar, bad[:5])


def test_cigars_equal_the_model_and_cost_the_score(base, lib):
    pairs = batch()
    pens = [pen for pen, cigar in CONFIGS if cigar]
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        flat = pool.map(_model, [(p, t, pen) for pen in pens for p, t in pairs], chunksize=2)
    for c, pen in enumerate(pens):
        r = base[key(pen, True)]
        want = flat[c * len(pairs):(c + 1) * len(pairs)]
        bad = [(i, r["cigars"][i][:60], w[1][:60]) for i, w in enumerate(want) if (r["scores"][i], r["cigars"][i]) != w]
        assert not bad, (pen, bad[:4])
        for i, (p, t) in enumerate(pairs):
            assert cost_ok(lib, p, t, pen, r["scores"][i], r["cigars"][i]), (pen, i, r["cigars"][i][:80])


def test_score_only_equals_the_cigar_runs(base):
    for pen in ((4, 4, 2, 24, 1), (2, 3, 1, 3, 1)):
        assert base[key(pen, False)]["scores"] == base[key(pen, True)]["scores"]


@pytest.mark.parametrize("pen", [(2, 3, 1, 3, 1), (4, 6, 2, 6, 2)])
def test_identical_pieces_print_the_single_piece_bytes(pen):
    # the plain call runs the headline kernels (four diagonals per thread, ring snapshots); the 2-piece call the
    # one-diagonal-per-thread kernels with decision bytes
    pairs = batch()
    assert run(pairs, pen, True) == run(pairs, pen, True, single=True)
    assert run(pairs, pen, False) == run(pairs, pen, False, single=True)


VARIANTS = {
    "force_large": {"WFAGPU_FORCE_LARGE": "1"},
    "warp_kernel": {"WFAGPU_WARP_KERNEL": "1"},
    "redispatch": {"AP_MAX_ERROR": "20"},
    "host_cigar": {"WFAGPU_HOST_CIGAR": "1"},
    "two_workers": {"WFAGPU_DEVICES": "0,0", "AP_BATCH": "16"},
}


@pytest.mark.parametrize("name", sorted(VARIANTS))
def test_variants_print_the_same_bytes(base, tmp_path, name):
    got = _run_check(tmp_path, name, VARIANTS[name])
    for k in base:
        assert got[k] == base[k], (name, k)


def test_pair_longer_than_32767(lib):
    rng = np.random.default_rng(0xA232)
    t = rand_seq(rng, 33000)
    p = mutate(rng, t, 0.01)
    p = p[:20000] + p[20400:]
    pen = (4, 4, 2, 24, 1)
    r = run([(p, t)], pen, True, max_error=2000)
    assert r["scores"][0] == gotoh2p(p, t, *pen)
    assert cost_ok(lib, p, t, pen, r["scores"][0], r["cigars"][0])


def test_check_correctness_validates_every_pair():
    pairs = batch()
    a = wfagpu.Aligner()
    for p, t in pairs:
        a.add_sequences(p, t)
    a.initialize_parameters(2, 3, 1)
    a.options.max_error = 600
    q = wfagpu.Affine2p(4, 4, 2, 24, 1)
    a.L.wfagpu_launch_alignments_affine2p(a.s.sequences_buffer, a.s.sequences_buffer_len, a.s.sequences_metadata,
                                          a.s.results, a.s.alignment_options, True, True, C.byref(q))
    st = a.run_stats()
    assert st["checked"] == len(pairs) and st["incorrect"] == 0, st
    assert a.L.wfagpu_last_launch_ok()


@pytest.mark.parametrize("case", ["band", "span", "negative", "e2_zero"])
def test_rejected_combinations_fail_cleanly(case):
    a = wfagpu.Aligner()
    for p, t in batch()[:8]:
        a.add_sequences(p, t)
    a.initialize_parameters(2, 3, 1)
    a.options.compute_cigar = True
    pen, span = (4, 4, 2, 24, 1), None
    if case == "band":
        a.options.band = 10
    elif case == "span":
        span = (0, 0, 20, 20)
    elif case == "negative":
        pen = (4, 4, 2, -24, 1)
    else:
        pen = (4, 4, 2, 24, 0)
    with pytest.raises((RuntimeError, ValueError)):
        a.align(ends_free=span, affine2p=pen)
    assert a.errors() == [0] * 8 and not any(a.cigars())
    # the C entry point rejects the span combination as well (the device layer returns -3 before anything is aligned)
    if case == "span":
        L = a.L
        d = L.wfagpu_device_open(0)
        assert d
        plan = wfagpu.Plan(4, 4, 2, 100, 0, 0, 1, 0, 0, 24, 1)
        sp = wfagpu.Span(0, 0, 20, 20)
        assert L.wfagpu_device_align_span(d, 0, 0, C.byref(plan), 0, C.byref(sp)) == -3
        L.wfagpu_device_release(d)


def test_cli_affine2p(tmp_path):
    pairs = batch()[:33] + batch()[-6:-1]
    seq = tmp_path / "ap.seq"
    seq.write_text("".join(f">{p}\n<{t}\n" for p, t in pairs))
    binary = os.path.join(os.path.dirname(HERE), "bin", "wfa.affine.gpu")
    outs = []
    for extra in ([], ["-S", "10"]):
        out = tmp_path / ("out%d.txt" % len(outs))
        pr = subprocess.run([binary, "-i", str(seq), "-G", "4,4,2,24,1", "-x", "-c", "-e", "600", "-o", str(out)] + extra,
                            capture_output=True, text=True, timeout=600)
        assert pr.returncode == 0, pr.stderr[-3000:]
        counts = re.findall(r"Incorrect=(\d+)", pr.stderr)
        assert counts and set(counts) == {"0"}, pr.stderr[-3000:]
        assert "O2=24, E2=1" in pr.stderr
        outs.append(out.read_text())
    assert outs[0] == outs[1]
    rows = [l.split("\t") for l in outs[0].splitlines()]
    assert [-int(r[0]) for r in rows] == [gotoh2p(p, t, 4, 4, 2, 24, 1) for p, t in pairs]
    for extra in (["-B", "auto"], ["-F", "0,0,5,5"], ["-g", "2,3,1"]):
        pr = subprocess.run([binary, "-i", str(seq), "-G", "4,4,2,24,1"] + extra, capture_output=True, text=True, timeout=600)
        assert pr.returncode != 0 and "cannot be combined" in pr.stderr, (extra, pr.stderr[-500:])
