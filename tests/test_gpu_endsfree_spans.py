"""Per-pair ends-free spans on the GPU (wfagpu_align_spans, Aligner.align(ends_free=[...]), the CLI's -E): every pair of
a mixed-span batch equals that pair aligned alone through wfagpu_align_span with its span -- score, CIGAR text and
coordinates, score-only and with CIGAR -- and the ends-free DP, and its CIGAR passes wfagpu_check_result_span.  n equal
spans reproduce the batch-span call and all-zero spans wfagpu_align byte for byte.  Every kernel variant, re-dispatch,
two workers per GPU with chunks that cut the span array mid-way, and check_correctness agree."""
import json
import os
import subprocess
import sys
from multiprocessing import Pool

import pytest

from endsfree_ref import gotoh_span, span_cost_ok
from endsfree_spans_check import jobs

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "bin", "wfa.affine.gpu")

VARIANTS = {
    "force_large": {"WFAGPU_FORCE_LARGE": "1"},
    "warp_kernel_on": {"WFAGPU_WARP_KERNEL": "1"},
    "warp_kernel_off": {"WFAGPU_WARP_KERNEL": "0"},
    "stages_1": {"WFAGPU_STAGES": "1"},
    "threads_64": {"WFAGPU_THREADS": "64"},
    "host_cigar": {"WFAGPU_HOST_CIGAR": "1"},
    "redispatch": {"EF_MAX_ERROR": "5"},
    "two_workers": {"WFAGPU_DEVICES": "0,0", "EF_BATCH": "7"},
}


def _run_check(tmp_path, name, env, alone=False):
    out = tmp_path / (name + ".json")
    subprocess.run([sys.executable, os.path.join(HERE, "endsfree_spans_check.py"), str(out)] + (["alone"] if alone else []),
                   check=True, env=dict(os.environ, **env), timeout=1800)
    return json.loads(out.read_text())


@pytest.fixture(scope="module")
def base(tmp_path_factory):
    return _run_check(tmp_path_factory.mktemp("spans"), "base", {}, alone=True)


@pytest.mark.gpu
def test_every_pair_equals_the_pair_aligned_alone(base):
    for name, r in base.items():
        for mode in ("cigar", "score"):
            for key in r["alone"][mode]:
                assert r[mode][key] == r["alone"][mode][key], (name, mode, key)
        assert r["plain"]["cigars"] == r["cigar"]["cigars"] and r["plain"]["scores"] == r["cigar"]["scores"], name


def _dp(job):
    p, t, pen, span = job
    return gotoh_span(p, t, *pen, span)


@pytest.mark.gpu
def test_scores_equal_the_dp_and_cigars_cost_the_score(base, lib):
    todo = [(name, i, (p, t, pen, sp)) for name, (pairs, pen, spans, _, _, _) in jobs().items()
            if name != "long" for i, ((p, t), sp) in enumerate(zip(pairs, spans))]
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        got = pool.map(_dp, [j for _, _, j in todo], chunksize=4)
    for (name, i, (p, t, pen, sp)), s in zip(todo, got):
        assert base[name]["cigar"]["scores"][i] == s, (name, i, sp)
        assert span_cost_ok(lib, p, t, *pen, sp, s, base[name]["cigar"]["cigars"][i]), (name, i, sp)


@pytest.mark.gpu
def test_equal_spans_and_zero_spans_reproduce_the_single_span_calls(base):
    for name in ("uniform", "zeros"):
        for mode in ("cigar", "score"):
            assert base[name][mode] == base[name]["ref"][mode], (name, mode)
    # zero-span pairs inside an ends-free batch get their global alignment
    z = [i for i, sp in enumerate(jobs()["mixed"][2]) if sp == (0, 0, 0, 0)]
    assert z and all(base["mixed"]["cigar"]["coords"][i][0] == 0 for i in z)
    for i in z:
        assert base["mixed"]["cigar"]["cigars"][i] == base["mixed"]["alone"]["cigar"]["cigars"][i]


@pytest.mark.gpu
def test_check_correctness(base):
    for name, (pairs, _, _, _, _, _) in jobs().items():
        for checked, incorrect, failed in base[name]["check"]:
            assert (checked, incorrect, failed) == (len(pairs), 0, 0), name


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_variants_give_the_same_results(base, tmp_path, variant):
    got = _run_check(tmp_path, variant, VARIANTS[variant])
    for name in base:
        for mode in ("cigar", "score", "plain"):
            assert got[name][mode] == base[name][mode], (variant, name, mode)
        assert got[name]["check"] == base[name]["check"], (variant, name)


def _seq_file(path, pairs):
    path.write_text("".join(">%s\n<%s\n" % (p, t) for p, t in pairs))


def _span_file(path, spans, extra=""):
    path.write_text("".join("%d,%d,%d,%d\n" % tuple(sp) for sp in spans) + extra)


def _cli(args):
    return subprocess.run([BIN] + args, capture_output=True, text=True, timeout=600)


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [[], ["-x"], ["-S", "7"], ["-x", "-S", "7", "-O"], ["-x", "-c"], ["-P", "-S", "5"]])
def test_cli_ends_free_file(base, tmp_path, extra):
    pairs, pen, spans, _, _, _ = jobs()["mixed"]
    seq, sf, out = tmp_path / "in.seq", tmp_path / "spans.txt", tmp_path / "out.txt"
    _seq_file(seq, pairs)
    _span_file(sf, spans)
    pr = _cli(["-i", str(seq), "-E", str(sf), "-g", ",".join(map(str, pen)), "-o", str(out)] + extra)
    assert pr.returncode == 0, pr.stderr[-2000:]
    lines = [ln.split("\t") for ln in out.read_text().splitlines()]
    assert len(lines) == len(pairs)
    for i, cols in enumerate(lines):
        assert -int(cols[0]) == base["mixed"]["cigar"]["scores"][i], (extra, i)
        if "-x" in extra:
            assert cols[1] == base["mixed"]["cigar"]["cigars"][i], (extra, i)
        if "-P" in extra:
            assert [int(v) for v in cols[2:6]] == base["mixed"]["score"]["coords"][i], (extra, i)
        if "-O" in extra:
            assert cols[2:] == list(pairs[i]), (extra, i)
    if "-c" in extra:
        assert "Incorrect=0" in pr.stderr and "Incorrect=1" not in pr.stderr, pr.stderr[-2000:]


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["short", "long", "malformed", "negative", "with_F", "with_B", "with_G", "n_short",
                                  "stream_short"])
def test_cli_ends_free_file_errors(tmp_path, case):
    pairs = jobs()["mixed"][0][:10]
    spans = [(1, 2, 3, 4)] * 10
    seq, sf = tmp_path / "in.seq", tmp_path / "spans.txt"
    _seq_file(seq, pairs)
    args = ["-i", str(seq), "-E", str(sf)]
    if case in ("short", "stream_short"):
        _span_file(sf, spans[:9])
        args += ["-S", "4"] if case == "stream_short" else []
    elif case == "long":
        _span_file(sf, spans + [(0, 0, 0, 0)])
    elif case == "malformed":
        _span_file(sf, spans[:4], "1,2,3\n" + "1,2,3,4\n" * 5)
    elif case == "negative":
        _span_file(sf, spans[:4], "1,2,-3,4\n" + "1,2,3,4\n" * 5)
    elif case == "n_short":
        _span_file(sf, spans)
        args += ["-n", "6"]                   # six pairs read, ten lines
    else:
        _span_file(sf, spans)
        args += {"with_F": ["-F", "1,1,1,1"], "with_B": ["-B", "10"], "with_G": ["-G", "4,4,2,24,1"]}[case]
    pr = _cli(args)
    assert pr.returncode != 0 and "ERROR" in pr.stderr, (case, pr.stderr[-2000:])
