"""Multi-GPU parity (needs >= 2 GPUs on the box; skipped otherwise): halo exchange (the peer-memory single launch by default,
NCCL on request) + all-reduce."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _num_gpus():
    try:
        out = subprocess.check_output(["nvidia-smi", "-L"], text=True)
        return sum(1 for line in out.splitlines() if line.startswith("GPU "))
    except Exception:
        return 0


def _run_check(world, port, env=None):
    if _num_gpus() < world:
        pytest.skip("needs %d GPUs" % world)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(world),
           "--master-addr", "127.0.0.1", "--master-port", str(port), os.path.join(ROOT, "tests", "multi_rank_check.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900, env=dict(os.environ, **(env or {})))
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    for r in range(world):
        assert "RANK %d OK" % r in res.stdout


@pytest.mark.parametrize("world", [2, 4])
def test_multi_rank_halo_and_reductions(world):
    _run_check(world, 29500 + world)


def test_multi_rank_nccl_halo():
    """The same checks with every halo exchanged by NCCL, the only alternative to the single launch: without this run the
    symmetric curl-curl cases never take that path on one node."""
    _run_check(2, 29510, {"MXG_HALO": "nccl"})
