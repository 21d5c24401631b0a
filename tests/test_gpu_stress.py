"""Short randomised sweep (tools/stress_parity.py): random penalty sets, lengths 1..3000, error rates,
length offsets, batch sizes and budgets, every pair against the oracle.  The long version of the same
script (5 kernel variants x 60-100 s, 632 k pairs, 0 mismatches) is recorded in DESIGN.md section 2."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("env", [{}, {"WFAGPU_FORCE_BOUND": "1"}, {"WFAGPU_QUAD_MIN": "1"},
                                 {"WFAGPU_QUAD_MIN": "1", "WFAGPU_QUAD_PAIRS": "1", "WFAGPU_FORCE_BOUND": "1"},
                                 {"WFAGPU_FORCE_LARGE": "1"}, {"WFAGPU_DEVICES": "0,0"}, {"WFAGPU_STAGES": "1"},
                                 {"WFAGPU_THREADS": "64"}])
def test_randomised_sweep(env):
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "stress_parity.py"), "15", "7"],
                        env=dict(os.environ, **env), capture_output=True, text=True, timeout=600)
    assert pr.returncode == 0, pr.stdout[-2000:] + pr.stderr[-2000:]
    assert "mismatches=0" in pr.stdout


def test_extreme_shapes():
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "extreme_check.py")], capture_output=True, text=True,
                        timeout=900)
    assert pr.returncode == 0, pr.stdout[-2000:] + pr.stderr[-2000:]


def test_randomised_sweep_vs_reference_gpu_binary():
    # needs oracle/_ref/gpu/wfa.affine.gpu (built here from /root/reference, travels with the snapshot)
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "gpu", "wfa.affine.gpu")):
        pytest.skip("reference GPU binary not built")
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "stress_vs_reference_gpu.py"), "20", "5"],
                        capture_output=True, text=True, timeout=900)
    assert pr.returncode == 0, pr.stdout[-2000:] + pr.stderr[-2000:]
    assert "mismatches=0" in pr.stdout
