"""The byte-compare kernels (pairs the packer flags: ASCII extend, ASCII traceback and decision bytes, the banded byte-compare
kernel, the byte-compare re-dispatch, the -c re-score) pinned to the oracle through relabelled twins: every flagged pair
with at most four distinct bytes is aligned in the same batch as its twin over ACGT, which takes the packed kernels.
Byte equality on the pair is base equality on the twin, so the pair's score and CIGAR text must equal its twin's, and
the twin's must equal the oracle's (banded: the oracle's banded result at the first budget, the exact result for pairs
the band does not finish).  Pairs with five distinct bytes: score == the byte-equality DP, CIGAR of that cost.  Under
-B, flagged pairs take the band as their twins do (the reference scores them exactly on its CPU).  Every kernel
variant, two workers per GPU with chunks that separate a pair from its twin, check_correctness and the CLI agree; the
tiers the file claims to cover show up in the launch lines of the byte-compare passes."""
import json
import os
import re
import subprocess
import sys
from functools import lru_cache

import pytest

import byte_compare_cases as bc
from byte_compare_check import BIG, CHECKED, PENS, VARIANT_JOBS, jobs
from endsfree_ref import gotoh_span

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BIN = os.path.join(ROOT, "bin", "wfa.affine.gpu")

VARIANTS = {
    "no_ckpt": {"WFAGPU_NO_CKPT": "1"},
    "ck_period_7": {"WFAGPU_CK_PERIOD": "7"},
    "ck_period_31": {"WFAGPU_CK_PERIOD": "31"},
    "arena_8mb": {"WFAGPU_ARENA_MB": "8"},
    "force_large": {"WFAGPU_FORCE_LARGE": "1"},
    "warp_kernel_off": {"WFAGPU_WARP_KERNEL": "0"},
    "warp_kernel_on": {"WFAGPU_WARP_KERNEL": "1"},
    "stages_1": {"WFAGPU_STAGES": "1"},
    "threads_64": {"WFAGPU_THREADS": "64"},
    "host_cigar": {"WFAGPU_HOST_CIGAR": "1"},
    "two_workers": {"WFAGPU_DEVICES": "0,0", "BC_BATCH": "7"},
    "no_quad": {"WFAGPU_NO_QUAD": "1"},
}


def _run_check(tmp_path, name, env, variant=False):
    out = tmp_path / (name + ".json")
    pr = subprocess.run([sys.executable, os.path.join(HERE, "byte_compare_check.py"), str(out)] + (["variant"] if variant else []),
                        env=dict(os.environ, **env), capture_output=True, text=True, timeout=1800)
    assert pr.returncode == 0, pr.stdout[-3000:] + pr.stderr[-3000:]
    return json.loads(out.read_text())


@pytest.fixture(scope="module")
def base(tmp_path_factory):
    return _run_check(tmp_path_factory.mktemp("bytecmp"), "base", {})


@lru_cache(maxsize=None)
def _batch(group):
    return bc.batch(group)


def _results(base, name):
    group, pen, cigar, budget, band, window = jobs()[name]
    pairs, kinds = _batch(group)
    r = base[name]
    cigars = r["cigars"] or [None] * len(pairs)
    return pairs, kinds, r["scores"], cigars, (group, pen, cigar, budget, band, window)


def test_every_flagged_pair_equals_its_twin(base):
    for name in jobs():
        pairs, kinds, scores, cigars, _ = _results(base, name)
        for i, k in enumerate(kinds):
            if k == "orig":
                assert (scores[i], cigars[i]) == (scores[i + 1], cigars[i + 1]), (name, i, pairs[i][0][:40], pairs[i][1][:40])


@lru_cache(maxsize=None)
def _expected(oracle, p, t, pen, cigar, budget, band, window):
    """The oracle's result of the twin: banded at the first budget, exact if the band does not finish it."""
    r = oracle.align(p, t, *pen, budget, band=band, window=window, cigar=cigar) if band else \
        oracle.align(p, t, *pen, budget, cigar=cigar)
    in_band = bool(band) and r["finished"]
    if not r["finished"]:
        r = oracle.align(p, t, *pen, BIG, cigar=cigar)
        assert r["finished"]
    return r["distance"], r["cigar"] if cigar else None, in_band


def test_twins_equal_the_oracle(base, oracle):
    band_finished = band_left = 0
    for name in jobs():
        pairs, kinds, scores, cigars, (group, pen, cigar, budget, band, window) = _results(base, name)
        if group == "long":
            continue                       # the oracle flags sequences of 32768 bases and more
        for i, k in enumerate(kinds):
            if k != "twin":
                continue
            dist, cg, in_band = _expected(oracle, *pairs[i], pen, cigar, budget, band, window)
            assert (scores[i], cigars[i]) == (dist, cg), (name, i, pairs[i][0][:40], pairs[i][1][:40])
            if band:
                band_finished += in_band
                band_left += not in_band
    # the band finishes some flagged pairs and leaves others to the exact kernels
    assert band_finished > 50 and band_left > 50, (band_finished, band_left)


@lru_cache(maxsize=None)
def _dp(p, t, pen):
    return gotoh_span(p, t, *pen, (0, 0, 0, 0))


def test_five_symbol_pairs_equal_the_dp_and_long_cigars_cost_their_score(base, oracle):
    n = 0
    for name in jobs():
        pairs, kinds, scores, cigars, (group, pen, cigar, budget, band, window) = _results(base, name)
        for i, k in enumerate(kinds):
            p, t = pairs[i]
            if k == "five" or group == "long":
                if cigar:
                    assert oracle.cigar_score(p, t, cigars[i], *pen) == scores[i], (name, i)
                if group == "long":
                    continue
                if band:
                    assert scores[i] >= _dp(p, t, pen), (name, i)
                else:
                    assert scores[i] == _dp(p, t, pen), (name, i)
                    n += 1
    assert n >= 7 * 2 * 2 * len(PENS)                # 4 short and 3 mid five-symbol pairs in every exact job


def test_ascii_pairs_equal_the_flagged_pairs_and_none_fail(base):
    for name in jobs():
        pairs, _, _, _, _ = _results(base, name)
        st = base[name]["stats"]
        assert st["ascii_pairs"] == sum(bc.pair_flagged(p, t) for p, t in pairs), (name, st)
        assert st["failed_pairs"] == 0, (name, st)
    # with a budget of 20, flagged pairs go through the byte-compare re-dispatch
    assert base["mid|2,3,1|20|cigar"]["stats"]["redispatched"] > 0


def _tier(line):
    m = re.search(r" group=(\d+) .* band=(\d+) tier=(\S+)", line)
    assert m, line
    threads, band, tier = int(m.group(1)), int(m.group(2)), m.group(3)
    return "band" if band else ("warp" if threads == 32 else tier)


def test_byte_compare_passes_reach_every_tier(base):
    seen = {}
    for name in jobs():
        for ln in base[name]["passes"]:
            seen.setdefault(_tier(ln), []).append(name)
    for tier in ("warp", "smem-int16+ckpt", "smem-int16", "global-int32", "band"):
        assert seen.get(tier), (tier, sorted(seen))
    assert any(n.endswith("score") for n in seen["smem-int16"])
    assert any(n.startswith("long") for n in seen["global-int32"])


def test_check_correctness(base):
    for (group, *_), (checked, incorrect, failed) in zip(CHECKED, base["checked"]):
        assert (checked, incorrect, failed) == (len(_batch(group)[0]), 0, 0), group


def _same(got, want):
    return got["scores"] == want["scores"] and got["cigars"] == want["cigars"] and \
        (got["stats"]["ascii_pairs"], got["stats"]["failed_pairs"]) == (want["stats"]["ascii_pairs"], want["stats"]["failed_pairs"])


@pytest.mark.parametrize("variant", sorted(VARIANTS))
def test_variants_give_the_same_results(base, tmp_path, variant):
    # redispatched is not compared: how many pairs outgrow a pass depends on the launch shape
    got = _run_check(tmp_path, variant, VARIANTS[variant], variant=True)
    for name in VARIANT_JOBS:
        assert _same(got[name], base[name]), (variant, name)
    assert got["checked"] == base["checked"], variant
    if variant == "no_ckpt":
        assert any("tier=smem-int16 " in ln for n in VARIANT_JOBS if n.endswith("cigar") for ln in got[n]["passes"])


@pytest.mark.parametrize("band", [False, True])
def test_cli_prints_what_the_api_returns(base, tmp_path, band):
    pairs, _ = _batch("cli")
    seq, out = tmp_path / "in.seq", tmp_path / "out.txt"
    seq.write_text("".join(">%s\n<%s\n" % pt for pt in pairs))
    job = "cli|band" if band else "cli"
    _, pen, _, budget, b, window = jobs()[job]
    args = ["-i", str(seq), "-o", str(out), "-g", ",".join(map(str, pen)), "-e", str(budget), "-x", "-c"]
    if band:
        args += ["-B", str(b), "-t", str(window)]
    pr = subprocess.run([BIN] + args, capture_output=True, text=True, timeout=600)
    assert pr.returncode == 0, pr.stderr[-3000:]
    assert "Incorrect=0" in pr.stderr and not re.search(r"Incorrect=[1-9]", pr.stderr), pr.stderr[-3000:]
    rows = [ln.split("\t") for ln in out.read_text().splitlines()]
    assert [-int(r[0]) for r in rows] == base[job]["scores"]
    assert [r[1] for r in rows] == base[job]["cigars"]
