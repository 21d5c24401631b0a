#!/usr/bin/env python3
"""Randomised gap-affine 2-piece sweep on a GPU box: random penalty sets (named regimes, their swapped pieces and random
draws), long indels at the crossover length, pair shapes, budgets and batch sizes through `Aligner.align(affine2p=...)`;
every pair against the 2-piece DP, the 2-piece validator and the CPU model's CIGAR bytes (tests/newpath_sweep.py).
usage: stress_affine2p.py <seconds|rounds> [seed]     (`60s`: 60 seconds, `12`: 12 rounds; WFAGPU_* select variants)"""
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests"))
from newpath_sweep import main  # noqa: E402

if __name__ == "__main__":
    sys.exit(main("ap", sys.argv))
