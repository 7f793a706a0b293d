"""Real multi-rank NCCL runs of the two-set functions (pairs.cross_pairs / extend_pairs, tl.wasserstein_d_cross /
wasserstein_d_extend): bit-identical to a single-rank solve.  Needs >= 2 GPUs on the box; skipped on one GPU."""
import os
import socket
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs >= 2 GPUs")
@pytest.mark.parametrize("nproc", [2, 4, 8])
def test_nccl_cross_and_extend_match_single_rank(nproc):
    if torch.cuda.device_count() < nproc:
        pytest.skip(f"needs {nproc} GPUs")
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={nproc}",
           "--master-addr", "127.0.0.1", "--master-port", str(_free_port()),
           os.path.join(ROOT, "tests", "multirank_cross_worker.py")]
    res = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, res.stdout[-3000:] + res.stderr[-3000:]
    assert f"MULTIRANK CROSS OK world={nproc}" in res.stdout
