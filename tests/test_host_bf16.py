"""CPU: the bf16 entry points of both cameras (bf16 sensor image out, bf16 gradient in) are exported and validate their
arguments on the host, before anything is enqueued - no device is touched."""
import ctypes

import pytest

from b200cam import _lib

E_BAD_SIZE, E_NULL, E_WORKSPACE, E_ALIGN = -1, -2, -3, -5
NOISE, QUANT = 1, 2
NEW = ("b200cam_sensor_fwd_bf16", "b200cam_sensor_finish_bf16", "b200cam_sensor_bwd_bf16",
       "b200cam_lens_normalise_bf16", "b200cam_lens_sensor_dot_bf16", "b200cam_lens_sensor_bwd_bf16")

null = ctypes.c_void_p(0)
a = ctypes.c_void_p(1 << 20)                  # 16-byte aligned, never dereferenced: validation fails first
odd = ctypes.c_void_p((1 << 20) + 2)          # bf16-aligned but not 16-byte aligned


@pytest.fixture(scope="module")
def library():
    _lib.build_library()
    return _lib.load_library()


def test_bf16_symbols_are_exported(library):
    for name in NEW:
        assert name in _lib.EXPORTED_SYMBOLS
        assert getattr(library, name) is not None


def test_sensor_fwd_bf16_rejects_bad_arguments(library):
    f = library.b200cam_sensor_fwd_bf16
    ws = library.b200cam_sensor_workspace_bytes(64, 2, 1)
    # img psf conv sensor img_max tie_count tie_pos otf spectrum ws bytes B N stream flags noise scale bits
    ok = [a, a, a, a, a, a, a, a, null, a, ws, 2, 64, null, 0, null, 0.0, 0]

    def call(**kw):
        args = list(ok)
        for i, v in kw.items():
            args[int(i[1:])] = v
        return f(*args)
    assert call(_12=96) == E_BAD_SIZE
    assert call(_11=0) == E_BAD_SIZE
    for i in (0, 1, 2, 3, 4, 5, 6, 7, 9):
        assert call(**{f"_{i}": null}) == E_NULL, i
    for i in (0, 1, 2, 3, 7, 8, 9):
        assert call(**{f"_{i}": odd}) == E_ALIGN, i
    assert call(_10=ws - 1) == E_WORKSPACE
    assert call(_14=4) == E_BAD_SIZE                          # unknown flag bit
    assert call(_14=NOISE) == E_NULL                          # noise requested, none given
    assert call(_14=QUANT, _17=17) == E_BAD_SIZE


def test_sensor_finish_bf16_rejects_bad_arguments(library):
    f = library.b200cam_sensor_finish_bf16
    ws = library.b200cam_sensor_workspace_bytes(128, 3, 1)
    # psf conv sensor img_max tie_count tie_pos otf spectrum otf_ready ws bytes B N stream flags noise scale bits
    ok = [a, a, a, a, a, a, a, a, 0, a, ws, 3, 128, null, 0, null, 0.0, 0]

    def call(**kw):
        args = list(ok)
        for i, v in kw.items():
            args[int(i[1:])] = v
        return f(*args)
    assert call(_12=100) == E_BAD_SIZE
    assert call(_11=-1) == E_BAD_SIZE
    for i in (0, 1, 2, 3, 4, 5, 6, 7, 9):
        assert call(**{f"_{i}": null}) == E_NULL, i
    for i in (0, 1, 2, 6, 7, 9):
        assert call(**{f"_{i}": odd}) == E_ALIGN, i
    assert call(_10=ws - 1) == E_WORKSPACE
    assert call(_14=NOISE | QUANT | 8, _15=a, _17=8) == E_BAD_SIZE
    assert call(_14=QUANT, _17=0) == E_BAD_SIZE


def test_sensor_bwd_bf16_rejects_bad_arguments(library):
    f = library.b200cam_sensor_bwd_bf16
    ws = library.b200cam_sensor_workspace_bytes(64, 2, 1)
    # grad img img_max tie_count tie_pos psf otf spectrum grad_psf grad_img ws bytes B N stream
    ok = [a, a, a, a, a, a, a, null, a, null, a, ws, 2, 64, null]

    def call(**kw):
        args = list(ok)
        for i, v in kw.items():
            args[int(i[1:])] = v
        return f(*args)
    assert call(_13=2048) == E_BAD_SIZE
    assert call(_12=0) == E_BAD_SIZE
    for i in (0, 1, 2, 3, 4, 5, 6, 8, 10):
        assert call(**{f"_{i}": null}) == E_NULL, i
    for i in (0, 1, 6, 7, 8, 9, 10):
        assert call(**{f"_{i}": odd}) == E_ALIGN, i
    assert call(_11=ws - 1) == E_WORKSPACE


def test_lens_normalise_bf16_rejects_bad_arguments(library):
    f = library.b200cam_lens_normalise_bf16
    assert f(a, a, odd, 16, null, 0, null, 0.0, 0) == E_ALIGN                 # misaligned y
    assert f(odd, a, a, 16, null, 0, null, 0.0, 0) == E_ALIGN
    assert f(null, a, a, 16, null, 0, null, 0.0, 0) == E_NULL
    assert f(a, null, a, 16, null, 0, null, 0.0, 0) == E_NULL
    assert f(a, a, null, 16, null, 0, null, 0.0, 0) == E_NULL
    assert f(a, a, a, 18, null, 0, null, 0.0, 0) == E_BAD_SIZE                # not a multiple of 4
    assert f(a, a, a, -4, null, 0, null, 0.0, 0) == E_BAD_SIZE
    assert f(a, a, a, 16, null, NOISE, null, 0.01, 0) == E_NULL               # noise requested, none given
    assert f(a, a, a, 16, null, QUANT, null, 0.0, 0) == E_BAD_SIZE            # quant_bits outside 1 ... 16
    assert f(a, a, a, 16, null, 4, null, 0.0, 0) == E_BAD_SIZE                # unknown flag bit
    assert f(a, a, a, 0, null, NOISE | QUANT, a, 0.01, 8) == 0                # nothing to do: nothing enqueued


def test_lens_dot_and_bwd_bf16_reject_bad_arguments(library):
    ws = library.b200cam_lens_sensor_workspace_bytes(128, 2)
    dot = library.b200cam_lens_sensor_dot_bf16
    assert dot(a, a, a, a, a, ws, 2, 368, null) == E_BAD_SIZE                 # 736 is not a power of two
    assert dot(a, a, a, a, a, ws, 0, 128, null) == E_BAD_SIZE
    for i in range(5):
        args = [a, a, a, a, a]
        args[i] = null
        assert dot(*args, ws, 2, 128, null) == E_NULL, i
    assert dot(odd, a, a, a, a, ws, 2, 128, null) == E_ALIGN
    assert dot(a, odd, a, a, a, ws, 2, 128, null) == E_ALIGN
    assert dot(a, a, a, a, a, ws - 1, 2, 128, null) == E_WORKSPACE
    bwd = library.b200cam_lens_sensor_bwd_bf16
    # grad raw gmax coef otf spectrum grad_kernel grad_img ws bytes B P stream
    assert bwd(a, a, a, a, a, a, a, null, a, ws, 2, 100, null) == E_BAD_SIZE
    assert bwd(a, a, a, a, a, a, a, null, a, ws, -3, 128, null) == E_BAD_SIZE
    for i in (0, 1, 2, 3, 4, 5, 6, 8):
        args = [a, a, a, a, a, a, a, null, a]
        args[i] = null
        assert bwd(*args, ws, 2, 128, null) == E_NULL, i
    for i in (0, 1, 5, 8):
        args = [a, a, a, a, a, a, a, null, a]
        args[i] = odd
        assert bwd(*args, ws, 2, 128, null) == E_ALIGN, i
    assert bwd(a, a, a, a, a, a, a, null, a, ws - 1, 2, 128, null) == E_WORKSPACE


def test_fp32_readout_entry_points_still_reject_flag_4(library):
    """the bf16 output is its own entry point, not a flag bit of the _ex calls"""
    assert library.b200cam_lens_normalise_ex(a, a, a, 16, null, 4, null, 0.0, 0) == E_BAD_SIZE
    ws = library.b200cam_sensor_workspace_bytes(64, 2, 1)
    assert library.b200cam_sensor_fwd_ex(a, a, a, a, a, a, a, null, a, ws, 2, 64, null, 4, null, 0.0, 0) == E_BAD_SIZE
