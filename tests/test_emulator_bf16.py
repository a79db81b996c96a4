"""CPU: the bf16 variants of the sensor kernel bodies through the test-only emulator (tests/emu/emu_bf16.cpp).

A camera with ``sensor_dtype = torch.bfloat16`` must compute exactly ``camera_fp32(x).to(torch.bfloat16)`` and, in backward,
exactly the fp32 backward on ``g.float()``.  Here that is checked body by body: the bf16 normalise against the fp32 one cast
with torch, the bf16 gradient row passes (K1 and the TMA-staged K1s) against the fp32 ones on the widened gradient, and the
whole emulated backward."""
import pytest
import torch

import emu_bf16_harness as emu16
import emu_harness as emu
import b200cam.synthetic as synth
from oracle import camera_oracle as co


def _same(a: torch.Tensor, b: torch.Tensor) -> bool:
    """bitwise equality (bf16 compared through its bit patterns, so -0 / NaN payloads count)"""
    if a.dtype == torch.bfloat16:
        a, b = a.view(torch.int16), b.view(torch.int16)
    else:
        a, b = a.view(torch.int32), b.view(torch.int32)
    return a.shape == b.shape and torch.equal(a, b)


def test_host_rounding_matches_torch_for_finite_values():
    g = torch.Generator().manual_seed(0)
    # every exponent, random mantissas, plus the halfway cases of round-to-nearest-even and the extremes
    bits = torch.randint(0, 2 ** 31 - 1, (1 << 18,), generator=g, dtype=torch.int64)
    x = bits.to(torch.int32).view(torch.float32)
    x = x[torch.isfinite(x)]
    x = torch.cat([x, -x])
    ties = torch.tensor([0x3f808000, 0x3f818000, 0x3f80ffff, 0x3f817fff, 0x7f7fffff, 0x7f7f8000, 0x00008000, 0x00018000,
                         0x00000001, 0x00800000, 0x00000000, -2 ** 31, 0x7f800000, -8388608], dtype=torch.int64)
    x = torch.cat([x, ties.to(torch.int32).view(torch.float32), torch.tensor([1.0 / 3, 0.1, 1.0, 65504.0])])
    assert _same(emu16.bf16_round(x), x.to(torch.bfloat16))


def _conv_batch(B, N, seed):
    g = torch.Generator().manual_seed(seed)
    conv = torch.rand(B, 3, N, N, generator=g) * 3.0
    m = conv.reshape(B, -1).amax(1)
    return conv, m


@pytest.mark.parametrize("epilogue", [False, True])
def test_normalise_bf16_is_the_fp32_body_cast(epilogue):
    B, N = 3, 64
    conv, m = _conv_batch(B, N, 1)
    noise = torch.randn(B, 3, N, N, generator=torch.Generator().manual_seed(2)) if epilogue else None
    kw = dict(noise=noise, noise_scale=0.02, levels=255.0) if epilogue else {}
    y32, tc32, tp32 = emu16.normalise(conv, m, False, **kw)
    y16, tc16, tp16 = emu16.normalise(conv, m, True, **kw)
    assert y16.dtype == torch.bfloat16
    assert _same(y16, y32.to(torch.bfloat16))
    assert torch.equal(tc16, tc32) and torch.equal(tp16, tp32)
    assert tc32.tolist() == [1] * B


def test_normalise_bf16_records_an_exact_tie():
    B, N = 2, 64
    conv, m = _conv_batch(B, N, 3)
    conv[0, 0, 5, 7] = conv[0, 2, 40, 9] = m[0] = 4.0          # two positions attain the maximum exactly
    y32, tc32, tp32 = emu16.normalise(conv, m, False)
    y16, tc16, tp16 = emu16.normalise(conv, m, True)
    assert tc16[0].item() == 2 and torch.equal(tc16, tc32) and torch.equal(tp16, tp32)
    assert y16[0, 0, 5, 7].item() == 1.0 and y16[0, 2, 40, 9].item() == 1.0
    assert _same(y16, y32.to(torch.bfloat16))


@pytest.mark.parametrize("stream", [False, True], ids=["K1", "K1s"])
@pytest.mark.parametrize("N", [64, 128, 256, 512])
def test_gradient_rows_bf16_equal_fp32_on_widened_gradient(N, stream):
    g16 = (torch.randn(2, 3, N, N, generator=torch.Generator().manual_seed(N)) * 1e-3).to(torch.bfloat16)
    st16 = emu16.rows_r2c(g16, stream)
    st32 = emu16.rows_r2c(g16.float(), stream)
    assert _same(st16, st32)


@pytest.mark.parametrize("want_img_grad", [False, True])
@pytest.mark.parametrize("saved_spectrum", [False, True])
def test_emulated_bf16_pipeline_equals_fp32_on_widened_gradient(want_img_grad, saved_spectrum):
    N, B = 64, 3
    C = co.build_constants(N)
    img, w, h = synth.images(B, N, 21), synth.upstream_grad(B, N, 22), synth.height_map(N, 23)
    psf, _ = co.psf_from_height(h, C)
    psf = psf[0].contiguous()
    s32, m, tc, tp, otf, spec = emu16.sensor_fwd(img, psf, out_bf16=False)
    s16, m16, tc16, tp16, otf16, spec16 = emu16.sensor_fwd(img, psf, out_bf16=True)
    assert _same(s16, s32.to(torch.bfloat16))
    assert torch.equal(m16, m) and torch.equal(tc16, tc) and torch.equal(tp16, tp) and _same(otf16, otf) and _same(spec16, spec)
    g16 = w.to(torch.bfloat16)
    sp = spec if saved_spectrum else None
    gpsf32, gimg32 = emu16.sensor_bwd(g16.float(), img, m, tc, tp, psf, otf, want_img_grad=want_img_grad, spectrum=sp)
    gpsf16, gimg16 = emu16.sensor_bwd(g16, img, m, tc, tp, psf, otf, want_img_grad=want_img_grad, spectrum=sp)
    assert _same(gpsf16, gpsf32)
    if want_img_grad:
        assert _same(gimg16, gimg32)
    # the fp32 reference here is the pipeline of the original emulator (tests/emu/emu.cpp), bit for bit
    ref = emu.sensor_fwd(img, psf, save_spectrum=True)
    assert _same(ref[0], s32) and _same(ref[4], otf) and _same(ref[5], spec)
    gpsf_ref, gimg_ref = emu.sensor_bwd(g16.float(), img, s32, m, tc, tp, psf, otf, want_img_grad=want_img_grad, spectrum=sp)
    assert _same(gpsf_ref, gpsf32)
    if want_img_grad:
        assert _same(gimg_ref, gimg32)
