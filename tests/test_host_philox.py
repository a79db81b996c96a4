"""CPU: the Philox sensor read-out (B200CAM_SENSOR_NOISE_PHILOX).

* The new entry point is exported, and every entry point rejects a bad seed block before anything is enqueued - no device is
  touched.
* Through the emulator (tests/emu/emu_philox.cpp): the block function gives the Random123 known answers and agrees with a
  numpy Philox4x32-10; the materialiser puts counter first4 + e / 4 (64-bit, carries included) behind element e; the normalise
  body with the Philox epilogue is bitwise the tensor epilogue on the materialised noise."""
import ctypes

import numpy as np
import pytest
import torch

import emu_philox_harness as emu
from b200cam import _lib

E_BAD_SIZE, E_NULL, E_ALIGN = -1, -2, -5
NOISE, QUANT, PHILOX = 1, 2, 4

null = ctypes.c_void_p(0)
a = ctypes.c_void_p(1 << 20)                  # 16-byte aligned, never dereferenced: validation fails first
a8 = ctypes.c_void_p((1 << 20) + 8)           # 8- but not 16-byte aligned
a4 = ctypes.c_void_p((1 << 20) + 4)           # 4-byte aligned only


@pytest.fixture(scope="module")
def library():
    _lib.build_library()
    return _lib.load_library()


def test_sensor_noise_symbol_is_exported(library):
    assert "b200cam_sensor_noise" in _lib.EXPORTED_SYMBOLS
    assert library.b200cam_sensor_noise is not None


def test_sensor_noise_rejects_bad_arguments(library):
    f = library.b200cam_sensor_noise
    assert f(null, a, 16, null) == E_NULL
    assert f(a, null, 16, null) == E_NULL
    assert f(a, a, 18, null) == E_BAD_SIZE                   # count % 4 != 0
    assert f(a, a, -4, null) == E_BAD_SIZE
    assert f(a4, a, 16, null) == E_ALIGN                     # the seed block is 8-aligned
    assert f(a8, a8, 16, null) == E_ALIGN                    # out is 16-aligned
    assert f(a8, a, 0, null) == 0                            # nothing to do (an 8-aligned block is fine)


def _epilogue_calls(library):
    """every epilogue entry point with valid other arguments, as f(flags, noise, scale, bits)"""
    ws = library.b200cam_sensor_workspace_bytes(64, 2, 1)
    L = library
    yield "sensor_fwd_ex", lambda fl, nz, sc, qb: L.b200cam_sensor_fwd_ex(a, a, a, a, a, a, a, null, a, ws, 2, 64, null, fl, nz, sc, qb)
    yield "sensor_finish_ex", lambda fl, nz, sc, qb: L.b200cam_sensor_finish_ex(a, a, a, a, a, a, a, 0, a, ws, 2, 64, null, fl, nz, sc, qb)
    yield "sensor_fwd_bf16", lambda fl, nz, sc, qb: L.b200cam_sensor_fwd_bf16(a, a, a, a, a, a, a, a, null, a, ws, 2, 64, null, fl, nz,
                                                                              sc, qb)
    yield "sensor_finish_bf16", lambda fl, nz, sc, qb: L.b200cam_sensor_finish_bf16(a, a, a, a, a, a, a, a, 0, a, ws, 2, 64, null,
                                                                                    fl, nz, sc, qb)
    yield "sensor_fwd_u8", lambda fl, nz, sc, qb: L.b200cam_sensor_fwd_u8(a, a, a, a, a, a, a, null, a, ws, 2, 64, null, fl, nz, sc, qb)
    yield "sensor_fwd_u8_bf16", lambda fl, nz, sc, qb: L.b200cam_sensor_fwd_u8_bf16(a, a, a, a, a, a, a, a, null, a, ws, 2, 64, null,
                                                                                    fl, nz, sc, qb)
    yield "lens_normalise_ex", lambda fl, nz, sc, qb: L.b200cam_lens_normalise_ex(a, a, a, 16, null, fl, nz, sc, qb)
    yield "lens_normalise_bf16", lambda fl, nz, sc, qb: L.b200cam_lens_normalise_bf16(a, a, a, 16, null, fl, nz, sc, qb)


def test_every_epilogue_entry_point_checks_the_seed_block(library):
    for name, f in _epilogue_calls(library):
        assert f(NOISE | PHILOX, a, 0.01, 0) == E_BAD_SIZE, name          # the two noise sources together
        assert f(NOISE | PHILOX | QUANT, a, 0.01, 8) == E_BAD_SIZE, name
        assert f(PHILOX, null, 0.01, 0) == E_NULL, name
        assert f(PHILOX | QUANT, null, 0.01, 8) == E_NULL, name
        assert f(PHILOX, a4, 0.01, 0) == E_ALIGN, name
        assert f(PHILOX, a, 0.0, 0) == E_BAD_SIZE, name                  # a draw must have an amplitude
        assert f(PHILOX, a, -0.01, 0) == E_BAD_SIZE, name
        assert f(PHILOX, a, float("nan"), 0) == E_BAD_SIZE, name
        assert f(PHILOX | QUANT, a, 0.01, 17) == E_BAD_SIZE, name
        assert f(PHILOX | 8, a, 0.01, 0) == E_BAD_SIZE, name             # unknown flag bit


# ---- the generator, through the emulator --------------------------------------------------------------------------------
M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85


def np_philox(ctr: np.ndarray, key: np.ndarray) -> np.ndarray:
    """Philox4x32-10 (Random123) in numpy: ctr [n, 4], key [n, 2] uint32 -> [n, 4] uint32"""
    c = [ctr[:, i].astype(np.uint64) for i in range(4)]
    k0, k1 = key[:, 0].astype(np.uint64), key[:, 1].astype(np.uint64)
    m32 = np.uint64(0xFFFFFFFF)
    for _ in range(10):
        p0, p1 = np.uint64(M0) * c[0], np.uint64(M1) * c[2]
        c = [((p1 >> np.uint64(32)) ^ c[1] ^ k0) & m32, p1 & m32, ((p0 >> np.uint64(32)) ^ c[3] ^ k1) & m32, p0 & m32]
        k0, k1 = (k0 + np.uint64(W0)) & m32, (k1 + np.uint64(W1)) & m32
    return np.stack(c, axis=1).astype(np.uint32)


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff,) * 2, (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0), (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_random123_known_answers(ctr, key, want):
    got = emu.philox(np.array([ctr], dtype=np.uint32), np.array([key], dtype=np.uint32))
    assert [int(v) for v in got[0]] == list(want)


def test_block_function_matches_numpy_philox():
    rng = np.random.default_rng(7)
    ctr = rng.integers(0, 2**32, size=(4096, 4), dtype=np.uint64).astype(np.uint32)
    key = rng.integers(0, 2**32, size=(4096, 2), dtype=np.uint64).astype(np.uint32)
    assert np.array_equal(emu.philox(ctr, key), np_philox(ctr, key))


def _np_normals(key: int, j: np.ndarray) -> np.ndarray:
    """the normals of counters j (uint64) under `key`, in float64 from the numpy Philox: [len(j) * 4]"""
    ctr = np.zeros((len(j), 4), dtype=np.uint32)
    ctr[:, 0] = (j & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    ctr[:, 1] = (j >> np.uint64(32)).astype(np.uint32)
    kk = np.tile(np.array([[key & 0xFFFFFFFF, key >> 32]], dtype=np.uint32), (len(j), 1))
    x = np_philox(ctr, kk).astype(np.float64)
    u = (2.0 * np.floor(x / 512.0) + 1.0) * 2.0 ** -24
    r0, r1 = np.sqrt(-2.0 * np.log(u[:, 0])), np.sqrt(-2.0 * np.log(u[:, 2]))
    n = np.stack([r0 * np.cos(2 * np.pi * u[:, 1]), r0 * np.sin(2 * np.pi * u[:, 1]),
                  r1 * np.cos(2 * np.pi * u[:, 3]), r1 * np.sin(2 * np.pi * u[:, 3])], axis=1)
    return n.reshape(-1)


@pytest.mark.parametrize("key,first4", [(0, 0), (0x0123456789ABCDEF, 12345), (2**63 - 2, 2**32 - 3), (0x5555AAAA5555AAAA, 2**40 - 1)])
def test_materialised_noise_follows_the_counter_rule(key, first4):
    """element e gets the Box-Muller pair of counter first4 + e / 4 (the 64-bit counter carries into its high word)"""
    count = 4 * 64
    got = emu.noise(key, first4, count).double().numpy()
    j = np.uint64(first4) + np.arange(count // 4, dtype=np.uint64)
    want = _np_normals(key, j)
    np.testing.assert_allclose(got, want, rtol=0, atol=2e-5)
    assert np.abs(got).max() <= 5.77


def test_materialised_noise_does_not_depend_on_the_split():
    key, first4, count = 0xDEADBEEF12345678, 2**32 - 5, 4 * 40
    whole = emu.noise(key, first4, count)
    k = 13                                                       # float4s in the first part
    parts = torch.cat((emu.noise(key, first4, 4 * k), emu.noise(key, first4 + k, count - 4 * k)))
    assert torch.equal(whole.view(torch.int32), parts.view(torch.int32))


def _conv(B, N, seed):
    g = torch.Generator().manual_seed(seed)
    conv = torch.rand(B, 3, N, N, generator=g) * 3.0
    for b in range(B):                                           # exact ties of the maximum
        conv[b, b % 3, 1, 2:5] = 4.0
    return conv, conv.reshape(B, -1).amax(dim=1).contiguous()


@pytest.mark.parametrize("levels", [0.0, 255.0, 15.0])
@pytest.mark.parametrize("first4", [0, 2**32 - 7])
def test_philox_normalise_equals_the_tensor_epilogue_on_the_materialised_noise(levels, first4):
    B, N, key, scale = 3, 16, 0x0F0F0F0F12345678, 0.05
    conv, mx = _conv(B, N, 3)
    y_p, tc_p, tp_p = emu.normalise(conv, mx, seed=(key, first4), noise_scale=scale, levels=levels)
    noise = emu.noise(key, first4, conv.numel()).reshape(conv.shape)
    y_t, tc_t, tp_t = emu.normalise(conv, mx, noise=noise, noise_scale=scale, levels=levels)
    assert torch.equal(y_p.view(torch.int32), y_t.view(torch.int32))
    assert torch.equal(tc_p, tc_t)
    assert torch.equal(tp_p.sort(dim=1).values, tp_t.sort(dim=1).values)
    plain, _, _ = emu.normalise(conv, mx)
    assert not torch.equal(y_p, plain)                           # the noise was applied
