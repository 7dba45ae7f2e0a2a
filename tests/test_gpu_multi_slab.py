"""Slab-partitioned assembly on 2 and 4 GPUs (skipped with fewer): each rank assembles only its slab's rows
(tests/slab_assembly_check.py)."""
import os
import subprocess
import sys

import pytest

from test_gpu_multi import _num_gpus

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("world", [2, 4])
def test_slab_assembly_on_several_ranks(world):
    if _num_gpus() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(29520 + world), os.path.join(ROOT, "tests", "slab_assembly_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    for r in range(world):
        assert "RANK %d OK" % r in res.stdout
