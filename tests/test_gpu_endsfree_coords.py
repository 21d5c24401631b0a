"""Where each ends-free alignment lies (wfagpu_coords_t, Aligner.align(coords=True), the CLI's -P) on the GPU: the
score-only coordinates (origin rows) equal the CIGAR-mode coordinates (traceback) and the CPU model's (k_begin, k_end);
scores and CIGAR text equal the plain ends-free call; and the global DP of the aligned sub-pair equals the ends-free
score, an independent check that the interval is optimal.  Every kernel variant, re-dispatch and two workers per GPU
give the same coordinates."""
import json
import os
import subprocess
import sys
from multiprocessing import Pool

import pytest

import endsfree_model
import wfagpu
from endsfree_coords_check import jobs
from endsfree_ref import clamp, gotoh_span

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "bin", "wfa.affine.gpu")

VARIANTS = {
    "force_large": {"WFAGPU_FORCE_LARGE": "1"},
    "warp_kernel_on": {"WFAGPU_WARP_KERNEL": "1"},
    "warp_kernel_off": {"WFAGPU_WARP_KERNEL": "0"},
    "stages_1": {"WFAGPU_STAGES": "1"},
    "threads_64": {"WFAGPU_THREADS": "64"},
    "redispatch": {"EF_MAX_ERROR": "5"},
    "two_workers": {"WFAGPU_DEVICES": "0,0", "EF_BATCH": "16"},
}


def coords_of(k_begin, k_end, plen, tlen):
    te = min(tlen, plen + k_end)
    return (max(0, -k_begin), te - k_end, max(0, k_begin), te)


def _run_check(tmp_path, name, env):
    out = tmp_path / (name + ".json")
    subprocess.run([sys.executable, os.path.join(HERE, "endsfree_coords_check.py"), str(out)], check=True,
                   env=dict(os.environ, **env), timeout=1800)
    return json.loads(out.read_text())


@pytest.fixture(scope="module")
def base(tmp_path_factory):
    return _run_check(tmp_path_factory.mktemp("coords"), "base", {})


def _spanned():
    for name, (pairs, pen, span, _, _) in jobs().items():
        if span is not None:
            yield name, pairs, pen, span


_oracle = None


def _model_begin_end(job):
    global _oracle
    from oracle import Oracle
    if _oracle is None:
        _oracle = Oracle()
    p, t, pen, span, score = job
    m = endsfree_model.align(_oracle, p, t, *pen, span, max_steps=score + 8, cigar=False)
    return m["finished"], m["k_begin"], m["k_end"]


def _subpair_dp(job):
    p, t, pen, c = job
    pb, pe, tb, te = c
    return gotoh_span(p[pb:pe], t[tb:te], *pen, (0, 0, 0, 0))


@pytest.mark.gpu
def test_score_only_coords_equal_cigar_coords_and_the_plain_call(base):
    for name, r in base.items():
        assert r["score"]["coords"] == r["cigar"]["coords"], name
        assert r["score"]["scores"] == r["plain"]["scores"] == r["cigar"]["scores"], name
        assert r["cigar"]["cigars"] == r["plain"]["cigars"], name


@pytest.mark.gpu
def test_coords_equal_the_model(base):
    todo = [(name, i, (p, t, pen, span, base[name]["score"]["scores"][i]))
            for name, pairs, pen, span in _spanned() for i, (p, t) in enumerate(pairs)]
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        got = pool.map(_model_begin_end, [j for _, _, j in todo], chunksize=2)
    for (name, i, (p, t, pen, span, _)), (fin, kb, ke) in zip(todo, got):
        assert fin, (name, i)
        assert tuple(base[name]["score"]["coords"][i]) == coords_of(kb, ke, len(p), len(t)), (name, i, kb, ke)


@pytest.mark.gpu
def test_global_dp_of_the_aligned_part_equals_the_score(base):
    todo = [(name, i, (p, t, pen, tuple(base[name]["score"]["coords"][i])))
            for name, pairs, pen, span in _spanned() for i, (p, t) in enumerate(pairs)]
    with Pool(min(32, os.cpu_count() or 1)) as pool:
        got = pool.map(_subpair_dp, [j for _, _, j in todo], chunksize=1)
    for (name, i, (p, t, pen, c)), dp in zip(todo, got):
        pb, pe, tb, te = c
        assert 0 <= pb <= pe <= len(p) and 0 <= tb <= te <= len(t), (name, i, c)
        # the unaligned ends are free: within the span, and on one sequence at each end
        spb, spe, stb, ste = clamp(jobs()[name][2], len(p), len(t))
        assert pb <= spb and tb <= stb and len(p) - pe <= spe and len(t) - te <= ste, (name, i, c)
        assert min(pb, tb) == 0 and min(len(p) - pe, len(t) - te) == 0, (name, i, c)
        assert dp == base[name]["score"]["scores"][i], (name, i, c, dp)


@pytest.mark.gpu
def test_global_calls_cover_both_sequences(base):
    for name, (pairs, pen, span, _, _) in jobs().items():
        if span is None:
            want = [[0, len(p), 0, len(t)] for p, t in pairs]
            assert base[name]["score"]["coords"] == want and base[name]["cigar"]["coords"] == want, name


@pytest.mark.gpu
def test_score_zero_and_fully_free_text(base):
    # the read sits inside the text at score 0: the interval is the read's copy in the text
    r = base["edge|0,0,1000000,1000000"]
    edges = jobs()["edge|0,0,1000000,1000000"][0]
    i = next(j for j, (p, t) in enumerate(edges) if len(t) == 260 and t[30:230] == p)
    assert r["score"]["scores"][i] == 0 and r["score"]["coords"][i] == [0, 200, 30, 230]


@pytest.mark.gpu
@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_variants_give_the_same_coords(base, tmp_path, variant):
    got = _run_check(tmp_path, variant, VARIANTS[variant])
    for name in base:
        for mode in ("score", "cigar"):
            assert got[name][mode]["coords"] == base[name][mode]["coords"], (variant, name, mode)
            assert got[name][mode]["scores"] == base[name][mode]["scores"], (variant, name, mode)
        assert got[name]["cigar"]["cigars"] == base[name]["cigar"]["cigars"], (variant, name)


def _seq_file(path, pairs):
    path.write_text("".join(">%s\n<%s\n" % (p, t) for p, t in pairs))


@pytest.mark.gpu
@pytest.mark.parametrize("extra", [[], ["-x"], ["-S", "7"], ["-x", "-S", "7", "-O"]])
def test_cli_print_coords(base, tmp_path, extra):
    name = "edge|0,199,259,0"
    pairs, pen, span, _, _ = jobs()[name]
    seq, out = tmp_path / "in.seq", tmp_path / "out.txt"
    _seq_file(seq, pairs)
    for f, key in ((["-F", ",".join(map(str, span))], name), ([], "edge|global")):
        args = [BIN, "-i", str(seq), "-g", ",".join(map(str, pen)), "-P", "-o", str(out)] + f + extra
        if not f:
            args[args.index("-g") + 1] = "4,6,2"
        pr = subprocess.run(args, capture_output=True, text=True, timeout=600)
        assert pr.returncode == 0, pr.stderr[-2000:]
        lines = [ln.split("\t") for ln in out.read_text().splitlines()]
        assert len(lines) == len(pairs)
        for i, cols in enumerate(lines):
            assert -int(cols[0]) == base[key]["score"]["scores"][i], (f, extra, i)
            assert [int(v) for v in cols[2:6]] == base[key]["score"]["coords"][i], (f, extra, i, cols)
            if "-x" in extra:
                assert cols[1] == base[key]["cigar"]["cigars"][i]
            if "-O" in extra:
                assert cols[6:] == list(pairs[i]), (f, extra, i)
            else:
                assert len(cols) == 6


@pytest.mark.gpu
def test_cli_print_coords_with_affine2p_is_an_error(tmp_path):
    seq = tmp_path / "in.seq"
    _seq_file(seq, [("ACGT", "ACGT")])
    pr = subprocess.run([BIN, "-i", str(seq), "-G", "4,4,2,24,1", "-P"], capture_output=True, text=True, timeout=600)
    assert pr.returncode != 0 and "cannot be combined" in pr.stderr, pr.stderr[-2000:]


def test_coords_with_affine2p_raise_before_aligning():
    a = wfagpu.Aligner()
    assert a.add_sequences("ACGT", "ACGA")
    with pytest.raises(ValueError, match="cannot be combined"):
        a.align(affine2p=(4, 4, 2, 24, 1), coords=True)
    with pytest.raises(RuntimeError):
        a.coords()
