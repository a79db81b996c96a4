"""GPU, >= 2 devices (-m gpu; skipped on a single-GPU box): uint8 shards on both cameras.  Every rank's sensor images and the
all-reduced parameter gradient from uint8 shards are bit-identical to those from the same shards converted on the GPU
(tools/check_face_sharded_u8.py, tools/check_lens_sharded.py --u8)."""
import socket
import subprocess
import sys

import pytest
import torch

from conftest import REPO

pytestmark = pytest.mark.gpu


def _torchrun(script, *args):
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), str(REPO / "tools" / script), *args]
    return subprocess.run(cmd, capture_output=True, text=True, timeout=900)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("bf16", [False, True])
def test_face_camera_sharded_u8_equals_converted_shards(bf16):
    res = _torchrun("check_face_sharded_u8.py", *(["--bf16"] if bf16 else []))
    assert res.returncode == 0, (res.stdout + res.stderr)[-3000:]
    assert "FACE_SHARDED_U8" in res.stdout and "ok=True" in res.stdout


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_caption_camera_sharded_u8_equals_converted_shards():
    res = _torchrun("check_lens_sharded.py", "--u8")
    assert res.returncode == 0, (res.stdout + res.stderr)[-3000:]
    assert "LENS_SHARDED" in res.stdout and "u8=True" in res.stdout and "ok=True" in res.stdout
