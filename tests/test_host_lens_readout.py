"""CPU: the read-out entry points of the Image_Caption camera (uint8 images, noise + quantisation epilogue) are exported and
validate their arguments on the host, before anything is enqueued."""
import ctypes

import pytest

from b200cam import _lib

E_BAD_SIZE, E_NULL, E_ALIGN = -1, -2, -5
NOISE, QUANT = 1, 2


@pytest.fixture(scope="module")
def library():
    _lib.build_library()
    return _lib.load_library()


def test_readout_symbols_are_exported(library):
    for name in ("b200cam_lens_sensor_fwd_u8", "b200cam_lens_normalise_ex"):
        assert name in _lib.EXPORTED_SYMBOLS
        assert getattr(library, name) is not None


def test_uint8_forward_rejects_bad_arguments_without_gpu(library):
    null = ctypes.c_void_p(0)
    a = ctypes.c_void_p(1 << 20)                  # 16-byte aligned, never dereferenced: validation fails first
    odd = ctypes.c_void_p((1 << 20) + 1)
    ws = library.b200cam_lens_sensor_workspace_bytes(256, 4)
    fwd = library.b200cam_lens_sensor_fwd_u8
    assert fwd(a, a, a, a, a, a, a, ws, 4, 368, null) == E_BAD_SIZE          # 736 is not a power of two
    assert fwd(a, a, a, a, a, a, a, ws, 0, 256, null) == E_BAD_SIZE
    assert fwd(null, a, a, a, a, a, a, ws, 4, 256, null) == E_NULL
    assert fwd(odd, a, a, a, a, a, a, ws, 4, 256, null) == E_ALIGN
    assert fwd(a, a, odd, a, a, a, a, ws, 4, 256, null) == E_ALIGN
    assert fwd(a, a, a, a, a, a, a, ws - 1, 4, 256, null) == -3              # workspace too small


def test_normalise_ex_rejects_bad_arguments_without_gpu(library):
    null = ctypes.c_void_p(0)
    a = ctypes.c_void_p(1 << 20)
    odd = ctypes.c_void_p((1 << 20) + 4)
    f = library.b200cam_lens_normalise_ex
    assert f(a, a, odd, 16, null, 0, null, 0.0, 0) == E_ALIGN                 # misaligned y
    assert f(odd, a, a, 16, null, 0, null, 0.0, 0) == E_ALIGN
    assert f(null, a, a, 16, null, 0, null, 0.0, 0) == E_NULL
    assert f(a, a, a, 18, null, 0, null, 0.0, 0) == E_BAD_SIZE                # not a multiple of 4
    assert f(a, a, a, 16, null, NOISE, null, 0.01, 0) == E_NULL               # noise requested, none given
    assert f(a, a, a, 16, null, QUANT, null, 0.0, 0) == E_BAD_SIZE            # quant_bits outside 1 ... 16
    assert f(a, a, a, 16, null, QUANT, null, 0.0, 17) == E_BAD_SIZE
    assert f(a, a, a, 16, null, 4, null, 0.0, 0) == E_BAD_SIZE                # unknown flag bit
    assert f(a, a, a, 16, null, NOISE | QUANT | 8, a, 0.01, 8) == E_BAD_SIZE
    assert f(a, a, a, 0, null, NOISE | QUANT, a, 0.01, 8) == 0                # nothing to do: nothing enqueued
