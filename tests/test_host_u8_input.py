"""CPU: the uint8-image entry points of the Face-DeId sensor path are exported and validate their arguments on the host, before
anything is enqueued - no device is touched."""
import ctypes

import pytest

from b200cam import _lib

E_BAD_SIZE, E_NULL, E_WORKSPACE, E_ALIGN = -1, -2, -3, -5
NOISE, QUANT = 1, 2
NEW = ("b200cam_sensor_rows_u8", "b200cam_sensor_fwd_u8", "b200cam_sensor_fwd_u8_bf16", "b200cam_sensor_bwd_u8",
       "b200cam_sensor_bwd_u8_bf16")

null = ctypes.c_void_p(0)
a = ctypes.c_void_p(1 << 20)                  # 16-byte aligned, never dereferenced: validation fails first
odd = ctypes.c_void_p((1 << 20) + 1)          # a valid uint8 address, but not 16-byte aligned


@pytest.fixture(scope="module")
def library():
    _lib.build_library()
    return _lib.load_library()


def _caller(f, ok):
    def call(**kw):
        args = list(ok)
        for i, v in kw.items():
            args[int(i[1:])] = v
        return f(*args)
    return call


def test_u8_symbols_are_exported(library):
    for name in NEW:
        assert name in _lib.EXPORTED_SYMBOLS
        assert getattr(library, name) is not None


def test_sensor_rows_u8_rejects_bad_arguments(library):
    # img spectrum img_max tie_count B N stream
    call = _caller(library.b200cam_sensor_rows_u8, [a, a, a, a, 2, 64, null])
    assert call(_5=32) == E_BAD_SIZE
    assert call(_5=96) == E_BAD_SIZE
    assert call(_4=0) == E_BAD_SIZE
    for i in (0, 1, 2, 3):
        assert call(**{f"_{i}": null}) == E_NULL, i
    for i in (0, 1):
        assert call(**{f"_{i}": odd}) == E_ALIGN, i


def test_sensor_fwd_u8_rejects_bad_arguments(library):
    ws = library.b200cam_sensor_workspace_bytes(64, 2, 1)
    # img psf sensor img_max tie_count tie_pos otf spectrum ws bytes B N stream flags noise scale bits
    call = _caller(library.b200cam_sensor_fwd_u8, [a, a, a, a, a, a, a, null, a, ws, 2, 64, null, 0, null, 0.0, 0])
    assert call(_11=96) == E_BAD_SIZE
    assert call(_11=2048) == E_BAD_SIZE
    assert call(_10=0) == E_BAD_SIZE
    for i in (0, 1, 2, 3, 4, 5, 6, 8):
        assert call(**{f"_{i}": null}) == E_NULL, i
    for i in (0, 1, 2, 6, 7, 8):
        assert call(**{f"_{i}": odd}) == E_ALIGN, i
    assert call(_9=ws - 1) == E_WORKSPACE
    assert call(_13=4) == E_BAD_SIZE                          # unknown flag bit
    assert call(_13=NOISE) == E_NULL                          # noise requested, none given
    assert call(_13=QUANT, _16=17) == E_BAD_SIZE


def test_sensor_fwd_u8_bf16_rejects_bad_arguments(library):
    ws = library.b200cam_sensor_workspace_bytes(128, 3, 1)
    # img psf conv sensor img_max tie_count tie_pos otf spectrum ws bytes B N stream flags noise scale bits
    call = _caller(library.b200cam_sensor_fwd_u8_bf16, [a, a, a, a, a, a, a, a, null, a, ws, 3, 128, null, 0, null, 0.0, 0])
    assert call(_12=100) == E_BAD_SIZE
    assert call(_11=-1) == E_BAD_SIZE
    for i in (0, 1, 2, 3, 4, 5, 6, 7, 9):
        assert call(**{f"_{i}": null}) == E_NULL, i
    for i in (0, 1, 2, 3, 7, 8, 9):
        assert call(**{f"_{i}": odd}) == E_ALIGN, i
    assert call(_10=ws - 1) == E_WORKSPACE
    assert call(_14=NOISE | QUANT | 8, _15=a, _17=8) == E_BAD_SIZE
    assert call(_14=QUANT, _17=0) == E_BAD_SIZE


def test_sensor_bwd_u8_rejects_bad_arguments(library):
    ws = library.b200cam_sensor_workspace_bytes(64, 2, 1)
    ws0 = library.b200cam_sensor_workspace_bytes(64, 2, 0)
    # grad img sensor img_max tie_count tie_pos psf otf spectrum grad_psf grad_img ws bytes B N stream
    call = _caller(library.b200cam_sensor_bwd_u8, [a, a, a, a, a, a, a, a, null, a, a, a, ws, 2, 64, null])
    assert call(_14=2048) == E_BAD_SIZE
    assert call(_13=0) == E_BAD_SIZE
    for i in (0, 1, 2, 3, 4, 5, 6, 7, 9, 11):
        assert call(**{f"_{i}": null}) == E_NULL, i
    for i in (0, 1, 2, 7, 8, 9, 10, 11):
        assert call(**{f"_{i}": odd}) == E_ALIGN, i
    assert call(_12=ws - 1) == E_WORKSPACE                    # dL/dimg asked for: the larger workspace
    assert call(_10=null, _12=ws0 - 1) == E_WORKSPACE


def test_sensor_bwd_u8_bf16_rejects_bad_arguments(library):
    ws = library.b200cam_sensor_workspace_bytes(256, 2, 0)
    # grad img img_max tie_count tie_pos psf otf spectrum grad_psf grad_img ws bytes B N stream
    call = _caller(library.b200cam_sensor_bwd_u8_bf16, [a, a, a, a, a, a, a, null, a, null, a, ws, 2, 256, null])
    assert call(_13=48) == E_BAD_SIZE
    assert call(_12=-2) == E_BAD_SIZE
    for i in (0, 1, 2, 3, 4, 5, 6, 8, 10):
        assert call(**{f"_{i}": null}) == E_NULL, i
    for i in (0, 1, 6, 7, 8, 9, 10):
        assert call(**{f"_{i}": odd}) == E_ALIGN, i
    assert call(_11=ws - 1) == E_WORKSPACE


def test_sensor_fwd_u8_needs_the_fp32_workspace_size(library):
    """the uint8 calls take the workspace sizes of the fp32 calls (no extra room for a converted batch)"""
    for N in (64, 128, 256, 512, 1024):
        for B in (1, 7):
            ws = library.b200cam_sensor_workspace_bytes(N, B, 0)
            f = library.b200cam_sensor_fwd_u8
            assert f(a, a, a, a, a, a, a, null, a, ws - 1, B, N, null, 0, null, 0.0, 0) == E_WORKSPACE
