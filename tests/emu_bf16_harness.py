"""TEST INFRASTRUCTURE ONLY - ctypes wrapper around tests/emu/emu_bf16.cpp (CPU emulation of the bf16 variants of the sensor
kernel bodies, next to their fp32 instantiations in the same library)."""
import ctypes
import subprocess
from pathlib import Path

import torch

REPO = Path(__file__).resolve().parent.parent
SRC = REPO / "tests" / "emu" / "emu_bf16.cpp"
OUT = REPO / "tests" / "_build" / "libb200cam_emu_bf16.so"
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


def _bits(t: torch.Tensor) -> torch.Tensor:
    """a bf16 tensor's storage as int16 bit patterns (what crosses the C ABI as unsigned short)"""
    assert t.dtype == torch.bfloat16
    return t.contiguous().view(torch.int16)


def bf16_round(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> bf16 through the emulator's host rounding rule (compat.cuh bf16_bits_rn)"""
    x = x.contiguous()
    out = torch.empty(x.shape, dtype=torch.int16)
    assert lib().emu16_round(_p(x), _p(out), ctypes.c_longlong(x.numel())) == 0
    return out.view(torch.bfloat16)


def normalise(conv, img_max, out_bf16: bool, noise=None, noise_scale=0.0, levels=0.0):
    """the normalise body on `conv` [B,3,N,N] -> (sensor, tie_count, tie_pos); fp32 (in place on a copy) or bf16"""
    B, _, N, _ = conv.shape
    y = conv.contiguous().clone()
    tc = torch.zeros(B, dtype=torch.int32)
    tp = torch.zeros(B, 8, dtype=torch.int32)
    out = torch.empty(conv.shape, dtype=torch.int16) if out_bf16 else None
    rc = lib().emu16_normalise(N, B, _p(y), _p(img_max.contiguous()), _p(tc), _p(tp), _p(out),
                               _p(noise.contiguous() if noise is not None else None), ctypes.c_float(noise_scale),
                               ctypes.c_float(levels))
    assert rc == 0
    return (out.view(torch.bfloat16) if out_bf16 else y), tc, tp


def rows_r2c(x: torch.Tensor, stream: bool) -> torch.Tensor:
    """forward row pass (K1, or K1s with stream=True) of the planes of x [..., N, N], fp32 or bf16 -> [planes, N/2+1, N, 2]"""
    N = x.shape[-1]
    planes = x.numel() // (N * N)
    bf = x.dtype == torch.bfloat16
    src = _bits(x) if bf else x.contiguous()
    st = torch.empty(planes, N // 2 + 1, N, 2)
    assert lib().emu16_rows_r2c(N, planes, int(stream), int(bf), _p(src), _p(st)) == 0
    return st


def sensor_fwd(img, psf, out_bf16: bool):
    """the generic sensor forward with the row spectra kept -> (sensor fp32 or bf16, img_max, tie_count, tie_pos, otf, spectrum)"""
    B, _, N, _ = img.shape
    conv = torch.empty_like(img)
    sensor16 = torch.empty(img.shape, dtype=torch.int16) if out_bf16 else None
    img_max = torch.empty(B)
    tie_count = torch.zeros(B, dtype=torch.int32)
    tie_pos = torch.zeros(B, 8, dtype=torch.int32)
    otf = torch.empty(3, N // 2 + 1, N, 2)
    spectrum = torch.empty(3 * B, N // 2 + 1, N, 2)
    rc = lib().emu16_sensor_fwd(int(out_bf16), N, B, _p(img.contiguous()), _p(psf.contiguous()), _p(conv), _p(sensor16), _p(img_max),
                                _p(tie_count), _p(tie_pos), _p(otf), _p(spectrum))
    assert rc == 0
    sensor = sensor16.view(torch.bfloat16) if out_bf16 else conv
    return sensor, img_max, tie_count, tie_pos, otf, spectrum


def sensor_bwd(g, img, img_max, tie_count, tie_pos, psf, otf, want_img_grad=False, spectrum=None):
    """the generic sensor backward on the upstream gradient `g`, fp32 or bf16 (no sensor image argument)"""
    B, _, N, _ = img.shape
    bf = g.dtype == torch.bfloat16
    gpsf = torch.empty(3, N, N)
    gimg = torch.empty_like(img) if want_img_grad else None
    rc = lib().emu16_sensor_bwd(int(bf), N, B, _p(_bits(g) if bf else g.contiguous()), _p(img.contiguous()), _p(img_max),
                                _p(tie_count), _p(tie_pos), _p(psf.contiguous()), _p(otf), _p(spectrum), _p(gpsf), _p(gimg))
    assert rc == 0
    return gpsf, gimg
