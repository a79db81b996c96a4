"""GPU, >= 2 devices (-m gpu; skipped on a single-GPU box): the sharded Image_Caption camera with bf16 sensor images reproduces
the one-GPU bf16 result (tools/check_lens_sharded.py --bf16)."""
import socket
import subprocess
import sys

import pytest
import torch

from conftest import REPO

pytestmark = pytest.mark.gpu


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_caption_camera_sharded_bf16_matches_single_gpu():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), str(REPO / "tools" / "check_lens_sharded.py"), "--bf16"]
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, (res.stdout + res.stderr)[-3000:]
    assert "LENS_SHARDED" in res.stdout and "dtype=bfloat16" in res.stdout and "ok=True" in res.stdout
