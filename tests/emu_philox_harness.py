"""TEST INFRASTRUCTURE ONLY - ctypes wrapper around tests/emu/emu_philox.cpp (CPU emulation of the Philox sensor read-out:
the block function, the materialiser and the normalise body with the Philox epilogue)."""
import ctypes
import subprocess
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent.parent
SRC = REPO / "tests" / "emu" / "emu_philox.cpp"
OUT = REPO / "tests" / "_build" / "libb200cam_emu_philox.so"
CSRC = REPO / "privacy-preserving-vision_b200" / "csrc"
INCLUDE = REPO / "include"


def build() -> Path:
    deps = [SRC, *CSRC.glob("*.cuh"), *INCLUDE.glob("*.h")]
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


def _p(a):
    if a is None:
        return ctypes.c_void_p(0)
    if isinstance(a, np.ndarray):
        assert a.flags.c_contiguous
        return ctypes.c_void_p(a.ctypes.data)
    assert a.is_contiguous()
    return ctypes.c_void_p(a.data_ptr())


def philox(ctr: np.ndarray, key: np.ndarray) -> np.ndarray:
    """Philox4x32-10 of counters ctr [n, 4] under keys key [n, 2] (uint32) -> [n, 4] uint32"""
    ctr = np.ascontiguousarray(ctr, dtype=np.uint32).reshape(-1, 4)
    key = np.ascontiguousarray(key, dtype=np.uint32).reshape(-1, 2)
    out = np.empty_like(ctr)
    assert lib().emup_philox(_p(ctr), _p(key), _p(out), ctypes.c_longlong(ctr.shape[0])) == 0
    return out


def seed_block(key: int, first4: int) -> np.ndarray:
    return np.array([key, first4], dtype=np.uint64)


def noise(key: int, first4: int, count: int) -> torch.Tensor:
    """the materialiser's body: n(e) for e < count"""
    s = seed_block(key, first4)
    out = torch.empty(count, dtype=torch.float32)
    assert lib().emup_noise(_p(s), _p(out), ctypes.c_longlong(count)) == 0
    return out


def normalise(conv, img_max, seed=None, noise=None, noise_scale=0.0, levels=0.0):
    """the normalise body on conv [B,3,N,N] -> (sensor, tie_count, tie_pos), with the Philox epilogue (seed = (key, first4)) or
    the tensor epilogue (noise)"""
    B, _, N, _ = conv.shape
    y = conv.contiguous().clone()
    tc = torch.zeros(B, dtype=torch.int32)
    tp = torch.zeros(B, 8, dtype=torch.int32)
    s = seed_block(*seed) if seed is not None else None
    rc = lib().emup_normalise(N, B, _p(y), _p(img_max.contiguous()), _p(tc), _p(tp), _p(s),
                              _p(noise.contiguous() if noise is not None else None), ctypes.c_float(noise_scale),
                              ctypes.c_float(levels))
    assert rc == 0
    return y, tc, tp
