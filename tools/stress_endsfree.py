#!/usr/bin/env python3
"""Randomised ends-free sweep on a GPU box: random penalty sets (named regimes and random draws), spans at the clamp
edges, pair shapes, budgets and batch sizes through `Aligner.align(ends_free=...)`; every pair against the ends-free DP,
the span validator and the CPU model's CIGAR bytes (tests/newpath_sweep.py).
usage: stress_endsfree.py <seconds|rounds> [seed]     (`60s`: 60 seconds, `12`: 12 rounds; WFAGPU_* select variants)"""
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from newpath_sweep import main  # noqa: E402

if __name__ == "__main__":
    sys.exit(main("ef", sys.argv))
