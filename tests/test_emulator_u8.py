"""CPU: the uint8-image kernel bodies, through the emulator (tests/emu/emu_u8.cpp), are bitwise the fp32 bodies on the converted
batch.

The conversion is x * fp32(1/255) - what torch's ``u8.float() / 255.0`` does on the GPU, where a division by a CPU scalar is a
multiplication with its fp32 reciprocal.  On the CPU torch really divides, which differs in the last bit for about half of the
byte values, so the references here are built as ``u.float() * float32(1/255)``, never with CPU torch division."""
import pytest
import torch

import emu_u8_harness as emu

RECIP = torch.tensor(1.0 / 255.0, dtype=torch.float32)


def _convert(u: torch.Tensor) -> torch.Tensor:
    return u.float() * RECIP


def _bits(t: torch.Tensor) -> torch.Tensor:
    return t.contiguous().view(torch.int32)


def _images(B, N, seed):
    """uint8 images with several exact ties per image: a saturated block (255) in one channel, a constant block in another,
    random bytes elsewhere"""
    g = torch.Generator().manual_seed(seed)
    u = torch.randint(0, 240, (B, 3, N, N), generator=g, dtype=torch.uint8)
    for b in range(B):
        u[b, b % 3, 3:3 + N // 8, 5:5 + N // 16] = 255
        u[b, (b + 1) % 3, N // 2:N // 2 + 4, :] = 77
    return u


def test_conversion_is_the_reciprocal_product():
    u = torch.arange(256, dtype=torch.uint8)
    table = emu.convert_table()
    assert torch.equal(_bits(table), _bits(_convert(u)))
    assert table[0] == 0.0 and table[255] == 1.0
    # the rule matters: CPU division gives a different last bit for many bytes
    assert int((_bits(u.float() / 255.0) != _bits(table)).sum()) > 0


@pytest.mark.parametrize("N", [64, 256])
@pytest.mark.parametrize("stream", [False, True])
def test_rows_r2c_u8_is_the_fp32_body_on_the_converted_batch(N, stream):
    u = _images(3, N, seed=N + int(stream))
    st8, mx8, c8 = emu.rows_r2c(u, stream, init=True)
    st32, mx32, c32 = emu.rows_r2c(_convert(u), stream, init=True)
    assert torch.equal(_bits(st8), _bits(st32))
    # the per-image max / tie counters are reset as by the fp32 pass
    assert torch.equal(mx8, mx32) and torch.isinf(mx8).all() and (mx8 < 0).all()
    assert torch.equal(c8, c32) and (c8 == 0).all()


def test_rows_r2c_u8_k1_and_k1s_agree():
    u = _images(2, 128, seed=5)
    assert torch.equal(_bits(emu.rows_r2c(u, False)[0]), _bits(emu.rows_r2c(u, True)[0]))


def _ties(u: torch.Tensor):
    """tie lists as the forward records them: up to 8 positions (flat c*N*N + y*N + x) of the image maximum"""
    B, _, N, _ = u.shape
    tc = torch.zeros(B, dtype=torch.int32)
    tp = torch.zeros(B, 8, dtype=torch.int32)
    for b in range(B):
        flat = u[b].reshape(-1)
        idx = torch.nonzero(flat == flat.max()).reshape(-1)
        tc[b] = idx.numel()
        k = min(8, idx.numel())
        step = max(1, idx.numel() // k)
        tp[b, :k] = idx[::step][:k].to(torch.int32)
    return tc, tp


@pytest.mark.parametrize("N", [64, 256])
def test_tie_term_u8_is_the_fp32_body_on_the_converted_batch(N):
    B = 5
    u = _images(B, N, seed=2 * N)
    u[4] = 255                                   # a fully saturated image: every pixel ties
    tc, tp = _ties(u)
    assert (tc > 1).all() and (tc[:4] >= 8).all()
    g = torch.Generator().manual_seed(N)
    coef = torch.randn(B, generator=g)
    gpsf = torch.randn(3, N, N, generator=g)
    a = emu.tie_term(u, gpsf, tc, tp, coef)
    b = emu.tie_term(_convert(u), gpsf, tc, tp, coef)
    assert torch.equal(_bits(a), _bits(b))
    assert not torch.equal(a, gpsf)              # the term is not empty


def test_tie_term_u8_more_than_sixteen_ties_per_channel():
    """more ties in one channel than one 16-wide batch of the gather: the tail of the second batch is clamped and weighted 0"""
    N, B = 64, 3
    u = torch.zeros(B, 3, N, N, dtype=torch.uint8)
    u[:, 1] = 255
    tc = torch.full((B,), 8, dtype=torch.int32)
    tp = torch.stack([torch.arange(8, dtype=torch.int32) * 37 + N * N + b for b in range(B)])   # all in channel 1: 24 ties
    coef = torch.tensor([0.5, -1.25, 3.0])
    gpsf = torch.randn(3, N, N, generator=torch.Generator().manual_seed(1))
    a = emu.tie_term(u, gpsf, tc, tp, coef)
    b = emu.tie_term(_convert(u), gpsf, tc, tp, coef)
    assert torch.equal(_bits(a), _bits(b))
    assert torch.equal(a[0], gpsf[0]) and torch.equal(a[2], gpsf[2]) and not torch.equal(a[1], gpsf[1])
