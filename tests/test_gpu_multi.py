"""Multi-GPU HP2 (SURVEY.md §8e): point-sharded solve over N ranks == single-GPU solve to
fp64 reduction-order tolerance.  Needs >= 2 GPUs on the box; skipped otherwise."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_two_rank_solve_matches_single(gpu):
    import particlesfm_b200
    n = particlesfm_b200.device_count()
    if n < 2:
        pytest.skip("needs 2 GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2",
           "--master-addr", "127.0.0.1", "--master-port", "29517", os.path.join(ROOT, "tools", "mgpu_check.py")]
    out = subprocess.run(cmd, capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-3000:]
    assert out.stdout.count("MGPU_CHECK PASS") == 2
