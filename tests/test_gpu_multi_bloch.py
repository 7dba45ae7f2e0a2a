"""Bloch transfers on 2 GPUs (skipped with fewer): slab rows of P and R on a periodic-x Bloch grid, and the 2-rank V-cycle
against the global reference (tests/bloch_multi_check.py)."""
import os
import subprocess
import sys

import pytest

from test_gpu_multi import _num_gpus

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_bloch_transfers_and_vcycle_on_two_ranks():
    if _num_gpus() < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29540", os.path.join(ROOT, "tests", "bloch_multi_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    for r in range(2):
        assert "RANK %d OK" % r in res.stdout
