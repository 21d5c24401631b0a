"""Aligns the byte-compare jobs and writes {job: {...}} as JSON to argv[1]: per pair the score and (with CIGAR) the CIGAR
text, the run's ascii_pairs / redispatched / failed_pairs, and the WFAGPU_VERBOSE "pass:" lines of its byte-compare
passes (ascii=1); under "checked", the check_correctness counts of a mixed exact and a mixed banded batch.  Every batch
holds a group's flagged pairs and their twins alternating (tests/byte_compare_cases.py::batch).  argv[2] == "variant":
only the jobs of VARIANT_JOBS.  Run in a subprocess with WFAGPU_* variables that select a kernel variant; BC_BATCH sets
the batch size (an odd size cuts the batch between a pair and its twin)."""
import json
import os
import re
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "wfa-gpu_b200", "python"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import byte_compare_cases as bc  # noqa: E402
import wfagpu  # noqa: E402

PENS = [(2, 3, 1), (1, 0, 1), (4, 6, 2), (5, 3, 2), (2, 24, 9), (3, 1, 4)]
BIG, SMALL = 20000, 20          # SMALL: most flagged pairs outgrow the first pass and are re-dispatched (doubling budgets)
# (penalties, band, window, budget): small budgets, so that the band leaves some flagged pairs to the exact kernels
BANDS = [((2, 3, 1), 10, 64, 40), ((2, 3, 1), 25, 128, 60), ((4, 6, 2), 25, 512, 120), ((5, 3, 2), 10, 128, 60),
         ((2, 3, 1), 10, 64, 300)]   # a budget that lets the band re-centre many times and still finish most pairs


def jobs():
    """-> {name: (group, penalties, cigar, budget, band, window)}; band 0: exact"""
    out = {}
    for group in ("short", "mid"):
        for pen in PENS:
            for budget in (BIG, SMALL):
                for cigar in (True, False):
                    out["%s|%d,%d,%d|%d|%s" % ((group,) + pen + (budget, "cigar" if cigar else "score"))] = (
                        group, pen, cigar, budget, 0, 0)
        for pen, band, window, budget in BANDS:
            for cigar in (True, False):
                out["%s|%d,%d,%d|B%d/%d|%d|%s" % ((group,) + pen + (band, window, budget, "cigar" if cigar else "score"))] = (
                    group, pen, cigar, budget, band, window)
    for cigar in (True, False):
        out["long|2,3,1|3000|%s" % ("cigar" if cigar else "score")] = ("long", (2, 3, 1), cigar, 3000, 0, 0)
    out["cli"] = ("cli", (2, 3, 1), True, SMALL, 0, 0)
    out["cli|band"] = ("cli", (2, 3, 1), True, 40, 10, 64)
    return out


VARIANT_PENS = ("2,3,1", "2,24,9")
VARIANT_JOBS = [n for n in jobs() if n.split("|")[0] in ("short", "mid") and n.split("|")[1] in VARIANT_PENS]
CHECKED = [("mid", (2, 3, 1), True, SMALL, 0, 0), ("mid", (2, 3, 1), True, 40, 10, 64)]


class StderrLines:
    """The process's stderr (file descriptor 2, where the library prints) of a block, as a list of lines."""

    def __enter__(self):
        sys.stderr.flush()
        self.tmp = tempfile.TemporaryFile(mode="w+b")
        self.saved = os.dup(2)
        os.dup2(self.tmp.fileno(), 2)
        return self

    def __exit__(self, *exc):
        sys.stderr.flush()
        os.dup2(self.saved, 2)
        os.close(self.saved)
        self.tmp.seek(0)
        text = self.tmp.read().decode(errors="replace")
        self.tmp.close()
        sys.stderr.write(text)
        self.lines = text.splitlines()
        return False


def aligner(pairs, pen, cigar, budget, band, window):
    a = wfagpu.Aligner()
    for p, t in pairs:
        assert a.add_sequences(p, t)
    assert a.initialize_parameters(*pen)
    a.options.compute_cigar = cigar
    a.options.max_error = budget
    if band > 0:
        a.options.band = band
        a.options.threads_per_block = window
    bs = int(os.environ.get("BC_BATCH", "0"))
    if bs:
        a.set_batch_size(bs)
    return a


def run(group, pen, cigar, budget, band, window):
    pairs, _ = bc.batch(group)
    a = aligner(pairs, pen, cigar, budget, band, window)
    with StderrLines() as err:
        a.align()
    st = a.run_stats()
    return dict(scores=a.errors(), cigars=a.cigars() if cigar else None,
                stats={k: st[k] for k in ("ascii_pairs", "redispatched", "failed_pairs")},
                passes=[ln for ln in err.lines if "pass:" in ln and re.search(r" ascii=1 ", ln)])


def checked(group, pen, cigar, budget, band, window):
    pairs, _ = bc.batch(group)
    a = aligner(pairs, pen, cigar, budget, band, window)
    got = a.align_checked()
    return [got[0], got[1], a.run_stats()["failed_pairs"]]


if __name__ == "__main__":
    os.environ["WFAGPU_VERBOSE"] = "1"
    names = VARIANT_JOBS if len(sys.argv) > 2 and sys.argv[2] == "variant" else list(jobs())
    todo = jobs()
    res = {name: run(*todo[name]) for name in names}
    res["checked"] = [checked(*j) for j in CHECKED]
    with open(sys.argv[1], "w") as f:
        json.dump(res, f)
