"""ctypes binding of ``libb200cam.so`` (C ABI in ``include/b200cam.h``).

The library is built in-tree by ``__graft_entry__.build()`` / ``build_library()`` with
``nvcc -gencode arch=compute_100a,code=sm_100a`` - no torch C++ headers, so it is ABI-stable.
There is deliberately no fallback: if the shared object is missing, or a compute entry point
is called without a CUDA device, a ``RuntimeError`` is raised.
"""
from __future__ import annotations

import ctypes
import os
import subprocess
import threading
from pathlib import Path

CSRC = Path(__file__).resolve().parent / "csrc"
LIB_PATH = CSRC / "libb200cam.so"
INCLUDE = Path(__file__).resolve().parent.parent / "include"

NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-lineinfo", "-O3", "-std=c++17",
              "-shared", "-Xcompiler", "-fPIC"]

_lock = threading.Lock()
_lib = None
_inited: set[tuple[int, int]] = set()

_f = ctypes.c_void_p      # device float*
_SIGNATURES = {
    "b200cam_version": (ctypes.c_int, []),
    "b200cam_error_string": (ctypes.c_char_p, [ctypes.c_int]),
    "b200cam_supported": (ctypes.c_int, [ctypes.c_int]),
    "b200cam_launch_count": (ctypes.c_ulonglong, []),
    "b200cam_col_chunks": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "b200cam_device_error": (ctypes.c_int, [ctypes.c_int]),
    "b200cam_init": (ctypes.c_int, [ctypes.c_int]),
    "b200cam_otf_bytes": (ctypes.c_size_t, [ctypes.c_int]),
    "b200cam_psf_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int]),
    "b200cam_sensor_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "b200cam_psf_fwd": (ctypes.c_int, [_f, _f, _f, _f, ctypes.POINTER(ctypes.c_float), _f, _f, _f,
                                       _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_crop_abs_resize_fwd": (ctypes.c_int, [_f, _f, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_crop_abs_resize_bwd": (ctypes.c_int, [_f, _f, _f, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                                   ctypes.c_void_p]),
    "b200cam_zernike_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_longlong]),
    "b200cam_zernike_fwd": (ctypes.c_int, [_f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_longlong, ctypes.c_void_p]),
    "b200cam_zernike_bwd": (ctypes.c_int, [_f, _f, _f, ctypes.c_int, ctypes.c_longlong, ctypes.c_void_p]),
    "b200cam_zernike_fwd_ex": (ctypes.c_int, [_f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_longlong, ctypes.c_void_p,
                                              _f, ctypes.c_int]),
    "b200cam_zernike_bwd_ex": (ctypes.c_int, [_f, _f, _f, ctypes.c_int, ctypes.c_longlong, ctypes.c_void_p, _f, ctypes.c_int]),
    "b200cam_psf_field": (ctypes.c_int, [_f, _f, _f, ctypes.POINTER(ctypes.c_float), _f,
                                         _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int]),
    "b200cam_psf_otf_early": (ctypes.c_int, [_f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_psf_finish": (ctypes.c_int, [_f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_psf_bwd": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, ctypes.POINTER(ctypes.c_float), _f, _f, _f, _f,
                                       _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_comm_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "b200cam_psf_bwd_allreduce": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, ctypes.POINTER(ctypes.c_float), _f, _f, _f, _f,
                                                 _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_void_p,
                                                 ctypes.POINTER(ctypes.c_void_p), ctypes.c_int, ctypes.c_int, ctypes.c_float]),
    "b200cam_spectrum_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "b200cam_sensor_fwd": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f,
                                          _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_sensor_fwd_ex": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f,
                                             _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                             ctypes.c_int, _f, ctypes.c_float, ctypes.c_int]),
    "b200cam_sensor_finish_ex": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, ctypes.c_int,
                                                _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                                ctypes.c_int, _f, ctypes.c_float, ctypes.c_int]),
    # the Philox read-out's noise materialised (seed block: device address of {key, first4})
    "b200cam_sensor_noise": (ctypes.c_int, [ctypes.c_void_p, _f, ctypes.c_longlong, ctypes.c_void_p]),
    "b200cam_sensor_split_supported":(ctypes.c_int, [ctypes.c_int, ctypes.c_int]),
    "b200cam_sensor_rows": (ctypes.c_int, [_f, _f, _f, _f, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_psf_otf": (ctypes.c_int, [_f, _f, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_sensor_finish": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, ctypes.c_int,
                                             _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_conv_fwd": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_void_p]),
    "b200cam_conv_bwd": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                        ctypes.c_void_p]),
    "b200cam_sensor_bwd": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f, _f, _f, _f,
                                          _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_lens_psf_supported": (ctypes.c_int, [ctypes.c_int, ctypes.c_int]),
    "b200cam_lens_psf_padded": (ctypes.c_int, [ctypes.c_int]),
    "b200cam_lens_psf_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "b200cam_lens_psf_fwd": (ctypes.c_int, [_f, _f, _f, ctypes.POINTER(ctypes.c_double), _f, _f, _f, _f, _f, _f, _f, _f,
                                            ctypes.c_int, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_void_p]),
    "b200cam_lens_psf_bwd": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, ctypes.POINTER(ctypes.c_double), _f, _f, _f, _f,
                                            ctypes.c_int, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                            ctypes.c_void_p]),
    "b200cam_lens_sensor_workspace_bytes": (ctypes.c_size_t, [ctypes.c_int, ctypes.c_int]),
    "b200cam_lens_sensor_fwd": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_lens_sensor_fwd_u8": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_lens_normalise": (ctypes.c_int, [_f, _f, _f, ctypes.c_longlong, ctypes.c_void_p]),
    "b200cam_lens_normalise_ex": (ctypes.c_int, [_f, _f, _f, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_int, _f, ctypes.c_float,
                                                 ctypes.c_int]),
    "b200cam_lens_sensor_dot": (ctypes.c_int, [_f, _f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_lens_sensor_bwd": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                               ctypes.c_void_p]),
    # bf16 sensor image out / gradient in (unsigned short* bit patterns: passed as plain device pointers)
    "b200cam_sensor_fwd_bf16": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f, _f,
                                               _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                               ctypes.c_int, _f, ctypes.c_float, ctypes.c_int]),
    "b200cam_sensor_finish_bf16": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f, ctypes.c_int,
                                                  _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                                  ctypes.c_int, _f, ctypes.c_float, ctypes.c_int]),
    "b200cam_sensor_bwd_bf16": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f, _f, _f,
                                               _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_lens_normalise_bf16": (ctypes.c_int, [_f, _f, _f, ctypes.c_longlong, ctypes.c_void_p, ctypes.c_int, _f, ctypes.c_float,
                                                   ctypes.c_int]),
    "b200cam_lens_sensor_dot_bf16": (ctypes.c_int, [_f, _f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_lens_sensor_bwd_bf16": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f, _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int,
                                                    ctypes.c_void_p]),
    # uint8 images in (unsigned char*: passed as plain device pointers)
    "b200cam_sensor_rows_u8": (ctypes.c_int, [_f, _f, _f, _f, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_sensor_fwd_u8": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f,
                                             _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                             ctypes.c_int, _f, ctypes.c_float, ctypes.c_int]),
    "b200cam_sensor_fwd_u8_bf16": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f, _f,
                                                  _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                                  ctypes.c_int, _f, ctypes.c_float, ctypes.c_int]),
    "b200cam_sensor_bwd_u8": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f, _f, _f, _f,
                                             _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
    "b200cam_sensor_bwd_u8_bf16": (ctypes.c_int, [_f, _f, _f, _f, _f, _f, _f, _f, _f, _f,
                                                  _f, ctypes.c_size_t, ctypes.c_int, ctypes.c_int, ctypes.c_void_p]),
}
EXPORTED_SYMBOLS = tuple(_SIGNATURES)


def sources() -> list[Path]:
    return sorted(CSRC.glob("*.cu"))


def build_library(force: bool = False, verbose: bool = False) -> Path:
    """Compile csrc/*.cu into csrc/libb200cam.so for sm_100a (cross-compiles without a GPU)."""
    headers = list(CSRC.glob("*.cuh")) + list(INCLUDE.glob("*.h"))
    if not force and LIB_PATH.exists() and all(LIB_PATH.stat().st_mtime >= d.stat().st_mtime for d in sources() + headers):
        return LIB_PATH                      # (the GPU box gets the built library, not the objects)
    newest_header = max(h.stat().st_mtime for h in headers)
    nvcc = os.environ.get("NVCC", "nvcc")
    objdir = CSRC / "build"
    objdir.mkdir(exist_ok=True)
    # one object per translation unit, compiled side by side; only stale ones are rebuilt (every TU includes the headers)
    jobs, objs = [], []
    for src in sources():
        obj = objdir / (src.stem + ".o")
        objs.append(obj)
        if force or not obj.exists() or obj.stat().st_mtime < max(src.stat().st_mtime, newest_header):
            cmd = [nvcc, *[f for f in NVCC_FLAGS if f != "-shared"], "-c", "-o", str(obj), str(src)]
            if verbose:
                cmd.insert(1, "-Xptxas=-v")
            jobs.append((cmd, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)))
    for cmd, proc in jobs:
        out, err = proc.communicate()
        if proc.returncode != 0:
            raise RuntimeError(f"nvcc failed:\n{' '.join(cmd)}\n{out}\n{err}")
        if verbose:
            print(err)
    if jobs or not LIB_PATH.exists() or any(LIB_PATH.stat().st_mtime < o.stat().st_mtime for o in objs):
        cmd = [nvcc, "-shared", "-o", str(LIB_PATH), *[str(o) for o in objs]]
        res = subprocess.run(cmd, capture_output=True, text=True)
        if res.returncode != 0:
            raise RuntimeError(f"link failed:\n{' '.join(cmd)}\n{res.stdout}\n{res.stderr}")
    return LIB_PATH


def load_library() -> ctypes.CDLL:
    """dlopen the in-tree library and declare the prototypes.  Raises if it has not been built."""
    global _lib
    with _lock:
        if _lib is None:
            if not LIB_PATH.exists():
                raise RuntimeError(
                    f"{LIB_PATH} is missing - run `python -c 'import __graft_entry__ as g; g.build()'` "
                    "(b200cam has no CPU or PyTorch fallback)")
            lib = ctypes.CDLL(str(LIB_PATH))
            for name, (res, args) in _SIGNATURES.items():
                fn = getattr(lib, name)
                fn.restype, fn.argtypes = res, args
            _lib = lib
        return _lib


def check(code: int) -> None:
    if code != 0:
        msg = load_library().b200cam_error_string(code)
        raise RuntimeError(f"b200cam error {code}: {msg.decode() if msg else '?'}")


def ensure_init(N: int, device_index: int) -> None:
    """b200cam_init(N) once per (device, N); allocates, so it must happen outside graph capture."""
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("b200cam needs a CUDA device (sm_100a); there is no CPU path")
    key = (device_index, N)
    if key in _inited:
        return
    lib = load_library()
    with torch.cuda.device(device_index):
        check(lib.b200cam_init(N))
    _inited.add(key)


_DEVERR = {1: "the per-image maximum exchange of the sensor kernel timed out (clusters of one image not co-resident?)",
           2: "the peer-memory all-reduce of dL/dh timed out waiting for another rank (ranks out of step, or a rank died)",
           3: "the grid barrier of a cooperative PSF kernel timed out"}


def raise_on_device_error(device_index: int) -> None:
    """Surface a device-side error word (include/b200cam.h: B200CAM_DEVERR_*) as a RuntimeError and clear it.
    Reading it is one load from mapped host memory: cheap enough to do once per forward / backward."""
    import torch
    lib = load_library()
    with torch.cuda.device(device_index):
        code = lib.b200cam_device_error(1)
    if code:
        raise RuntimeError(f"b200cam device error {code}: {_DEVERR.get(code, 'unknown')}; the results of the step that "
                           "reported it are invalid")


def ptr(t) -> ctypes.c_void_p:
    return ctypes.c_void_p(t.data_ptr()) if t is not None else ctypes.c_void_p(0)
