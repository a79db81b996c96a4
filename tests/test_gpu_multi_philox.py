"""GPU, >= 2 devices (-m gpu; skipped on a single-GPU box): the Philox sensor noise on sharded batches.  With every rank
seeded alike, both cameras sharded over two ranks give the rows of the one-GPU sensor image of the whole batch, bit for bit
(tools/check_philox_sharded.py)."""
import socket
import subprocess
import sys

import pytest
import torch

from conftest import REPO

pytestmark = pytest.mark.gpu


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_both_cameras_sharded_reproduce_the_one_gpu_noise():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), str(REPO / "tools" / "check_philox_sharded.py")]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, (res.stdout + res.stderr)[-3000:]
    assert "PHILOX_SHARDED" in res.stdout and "ok=True" in res.stdout
