"""TEST INFRASTRUCTURE ONLY - ctypes wrapper around tests/emu/emu_u8.cpp (CPU emulation of the uint8-image variants of the
sensor kernel bodies, next to their fp32 instantiations in the same library)."""
import ctypes
import subprocess
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
SRC = REPO / "tests" / "emu" / "emu_u8.cpp"
OUT = REPO / "tests" / "_build" / "libb200cam_emu_u8.so"
CSRC = REPO / "privacy-preserving-vision_b200" / "csrc"


def build() -> Path:
    deps = [SRC, *CSRC.glob("*.cuh")]
    if OUT.exists() and all(OUT.stat().st_mtime >= d.stat().st_mtime for d in deps):
        return OUT
    OUT.parent.mkdir(parents=True, exist_ok=True)
    subprocess.run(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-o", str(OUT), str(SRC)], check=True)
    return OUT


_lib = None


def lib():
    global _lib
    if _lib is None:
        _lib = ctypes.CDLL(str(build()))
    return _lib


def _p(t):
    if t is None:
        return ctypes.c_void_p(0)
    assert t.is_contiguous()
    return ctypes.c_void_p(t.data_ptr())


def convert_table() -> torch.Tensor:
    """the fp32 value the kernels read for each of the 256 byte values"""
    out = torch.empty(256)
    assert lib().emu8_convert(_p(out)) == 0
    return out


def rows_r2c(x: torch.Tensor, stream: bool, init=False):
    """forward row pass (K1, or K1s with stream=True) of the planes of x [B, 3, N, N], fp32 or uint8 -> (st [planes, N/2+1, N, 2],
    img_max, tie_count) - the last two only with init=True (the reset the sensor forward asks of the row pass)"""
    N = x.shape[-1]
    planes = x.numel() // (N * N)
    x = x.contiguous()
    st = torch.empty(planes, N // 2 + 1, N, 2)
    mx = torch.zeros(planes // 3) if init else None
    cnt = torch.full((planes // 3,), 7, dtype=torch.int32) if init else None
    assert lib().emu8_rows_r2c(N, planes, int(stream), int(x.dtype == torch.uint8), _p(x), _p(st), _p(mx), _p(cnt)) == 0
    return st, mx, cnt


def tie_term(x: torch.Tensor, gpsf: torch.Tensor, tie_count: torch.Tensor, tie_pos: torch.Tensor, coef: torch.Tensor) -> torch.Tensor:
    """the arg-max gather K8 on x [B, 3, N, N] (fp32 or uint8): returns a copy of gpsf [3, N, N] with the term subtracted"""
    B, _, N, _ = x.shape
    out = gpsf.contiguous().clone()
    rc = lib().emu8_tie_term(N, B, int(x.dtype == torch.uint8), _p(x.contiguous()), _p(out), _p(tie_count.contiguous()),
                             _p(tie_pos.contiguous()), _p(coef.contiguous()))
    assert rc == 0
    return out
