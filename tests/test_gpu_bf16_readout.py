"""GPU (-m gpu): ``sensor_dtype = torch.bfloat16`` on both cameras.

The contract: the bf16 sensor image is exactly ``camera_fp32(x).to(torch.bfloat16)``, and the backward with a bf16 upstream
gradient ``g`` is exactly the fp32 backward on ``g.float()`` - parameter gradients, regularisers and dL/dimg, bit for bit."""
import ctypes

import pytest
import torch

import b200cam.synthetic as synth
from b200cam import _lib
from b200cam import functional as F
from b200cam.lens import OpticsZernike
from b200cam.optics import Camera
from conftest import rel_l2

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
BF16 = torch.bfloat16


def _bits_equal(a: torch.Tensor, b: torch.Tensor) -> bool:
    if a is None or b is None:
        return a is None and b is None
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    view = torch.int16 if a.dtype == BF16 else (torch.int32 if a.element_size() == 4 else torch.int64)
    return torch.equal(a.contiguous().view(view), b.contiguous().view(view))


# ------------------------------------------------------------------------------------------------------------ Face-DeId
def _camera(N, seed=0, terms=10):
    torch.manual_seed(seed)
    return Camera(device=DEV, N=N, zernike_terms=terms)


def _face_step(cam, img, g, dtype, noise=None, want_img=False):
    """one forward + backward: sensor, loss_rad, centering_loss, dL/dZer_train, dL/dimg"""
    cam.sensor_dtype = dtype
    cam.Zer_train.grad = None
    x = img.clone().requires_grad_(True) if want_img else img
    y = cam(x, noise=noise)
    assert y.dtype == dtype
    gy = g if dtype == BF16 else g.float()
    torch.autograd.backward([y, cam.loss_rad, cam.centering_loss],
                            [gy, torch.tensor(0.3, device=DEV), torch.tensor(1.7, device=DEV)])
    return (y.detach(), cam.loss_rad.detach().clone(), cam.centering_loss.detach().clone(), cam.Zer_train.grad.clone(),
            x.grad if want_img else None)


FACE_CASES = [(64, 2, overlap, u8, epi) for overlap in (True, False) for u8 in (False, True) for epi in (False, True)] + [
    (256, 64, True, False, False), (256, 64, False, False, False), (256, 64, True, True, True),
    (512, 2, True, False, False), (512, 2, False, True, True)]


@pytest.mark.parametrize("N,B,overlap,u8,epi", FACE_CASES)
def test_camera_bf16_is_the_fp32_camera_cast(N, B, overlap, u8, epi):
    cam = _camera(N)
    cam.overlap_psf = overlap
    img = synth.images(B, N, seed=N + B).to(DEV)
    if u8:
        img = (img * 255.0).round().clamp(0, 255).to(torch.uint8)
    g = (synth.upstream_grad(B, N, seed=N + 1) * 1e-2).to(DEV, BF16)
    noise = None
    if epi:
        cam.sensor_noise_sigma, cam.sensor_quant_bits = 0.02, 8
        noise = torch.randn(B, 3, N, N, generator=torch.Generator(device=DEV).manual_seed(5), device=DEV)
    want_img = not u8
    a = _face_step(cam, img, g, torch.float32, noise, want_img)
    b = _face_step(cam, img, g, BF16, noise, want_img)
    assert _bits_equal(b[0], a[0].to(BF16))
    for x, y in zip(b[1:], a[1:]):
        assert _bits_equal(x, y)
    # and a second bf16 step repeats itself
    c = _face_step(cam, img, g, BF16, noise, want_img)
    for x, y in zip(b, c):
        assert _bits_equal(x, y)


def test_camera_bf16_empty_batch():
    cam = _camera(64)
    cam.sensor_dtype = BF16
    y = cam(torch.empty(0, 3, 64, 64, device=DEV))
    assert y.dtype == BF16 and y.shape == (0, 3, 64, 64)


def test_sensor_dtype_is_validated():
    cam = _camera(64)
    img = synth.images(1, 64).to(DEV)
    for bad in (torch.float16, torch.float64, "bf16"):
        cam.sensor_dtype = bad
        with pytest.raises(ValueError):
            cam(img)
    lens = OpticsZernike(input_shape=[1, 64, 64, 3], device=DEV, wave_resolution=(128, 128), patch_size=64, sample_interval=3e-6,
                         zernike_terms=10, height_tolerance=None).to(DEV)
    lens.sensor_dtype = torch.float16
    with pytest.raises(ValueError):
        lens(torch.rand(1, 3, 64, 64, device=DEV))


@pytest.mark.parametrize("overlap", [True, False])
def test_bf16_node_saves_no_fp32_sensor_image(overlap):
    N, B = 64, 3
    img = synth.images(B, N).to(DEV)

    def big_fp32_saved(dtype):
        cam = _camera(N)
        cam.overlap_psf = overlap
        cam.sensor_dtype = dtype
        y = cam(img)
        saved = y.grad_fn.saved_tensors
        return [t for t in saved if t is not None and t.dtype == torch.float32 and tuple(t.shape) == (B, 3, N, N)
                and t.data_ptr() != img.data_ptr()]          # the input image itself is not extra memory
    assert len(big_fp32_saved(torch.float32)) == 1             # the fp32 node keeps its sensor image
    assert big_fp32_saved(BF16) == []


def test_graphed_bf16_step():
    """graphed() in bf16: the replay equals the fp32 graphed step cast (both capture the same multi-kernel PSF chain), repeats
    itself, and agrees with the eager bf16 step to the rounding of the eager (cooperative) PSF chain."""
    N, B = 128, 4
    img = synth.images(B, N, seed=3).to(DEV)
    g = (synth.upstream_grad(B, N, seed=4) * 1e-2).to(DEV, BF16)
    res = {}
    for dtype in (torch.float32, BF16):
        cam = _camera(N, seed=3)
        cam.sensor_dtype = dtype
        step = cam.graphed(img)
        outs = []
        for _ in range(2):
            cam.Zer_train.grad = None
            y, rad, cen = step(img)
            assert y.dtype == dtype
            torch.autograd.backward([y, rad, cen], [g if dtype == BF16 else g.float(), torch.tensor(0.3, device=DEV),
                                                   torch.tensor(1.7, device=DEV)])
            outs.append((y.detach().clone(), cam.Zer_train.grad.clone()))
        assert _bits_equal(outs[0][0], outs[1][0]) and _bits_equal(outs[0][1], outs[1][1])
        res[dtype] = (outs[0], cam)
    (y32, g32), _ = res[torch.float32]
    (y16, g16), cam = res[BF16]
    assert _bits_equal(y16, y32.to(BF16))
    assert _bits_equal(g16, g32)
    ye, _, _, ge, _ = _face_step(cam, img, g, BF16)
    assert rel_l2(ye.float(), y16.float()) <= 1e-3
    assert rel_l2(ge, g16) <= 1e-4


# ------------------------------------------------------------------------------------------------------------ Image_Caption
FUSED = [(896, 256), (128, 64)]
UNFUSED = [(64, 32), (736, 368)]


def _lens(wave, patch, tol=None, terms=10):
    cam = OpticsZernike(input_shape=[1, patch, patch, 3], device=DEV, wave_resolution=(wave, wave), patch_size=patch,
                        sample_interval=3e-6, zernike_terms=terms, height_tolerance=tol).to(DEV)
    with torch.no_grad():
        cam.zernike_coeffs_train.fill_(-22.0 * (wave / 896) ** 2)
        cam.zernike_coeffs_no_train2[0] = 0.3
    return cam


def _lens_step(cam, img, g, dtype, seed, noise=None):
    cam.sensor_dtype = dtype
    torch.manual_seed(seed)
    cam.zernike_coeffs_train.grad = None
    sensor, psf, coeffs, _ = cam(img, noise=noise)
    assert sensor.dtype == dtype and psf.dtype == torch.float32
    sensor.backward(g if dtype == BF16 else g.float())
    return sensor.detach(), psf.detach(), cam.zernike_coeffs_train.grad.clone()


@pytest.mark.parametrize("wave,patch", FUSED + UNFUSED)
def test_caption_bf16_is_the_fp32_camera_cast(wave, patch):
    B = 3 if patch <= 256 else 2
    gen = torch.Generator().manual_seed(patch)
    u8 = torch.randint(0, 256, (B, 3, patch, patch), generator=gen, dtype=torch.uint8).to(DEV)
    g = (torch.rand(B, 3, patch, patch, generator=gen) * 1e-2).to(DEV, BF16)
    noise = torch.randn(B, 3, patch, patch, generator=torch.Generator(device=DEV).manual_seed(9), device=DEV)
    for tol in (None, 20e-9):
        cam = _lens(wave, patch, tol)
        for img in (u8, u8.float() / 255.0):
            for epi in (False, True):
                cam.sensor_noise_sigma, cam.sensor_quant_bits = (0.02, 8) if epi else (0.0, 0)
                nz = noise if epi else None
                a = _lens_step(cam, img, g, torch.float32, seed=7, noise=nz)
                b = _lens_step(cam, img, g, BF16, seed=7, noise=nz)
                assert _bits_equal(b[0], a[0].to(BF16)), (tol, img.dtype, epi)
                assert _bits_equal(b[1], a[1]) and _bits_equal(b[2], a[2]), (tol, img.dtype, epi)


# ------------------------------------------------------------------------------------------------------------ C ABI
def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _same_ties(a, b):
    """the recorded arg-max positions: tie_pos is written only up to tie_count (its other slots are never read)"""
    assert torch.equal(a["tc"], b["tc"])
    for i, n in enumerate(a["tc"].tolist()):
        n = min(n, 8)
        assert sorted(a["tp"][i, :n].tolist()) == sorted(b["tp"][i, :n].tolist())


def test_face_abi_bf16_entry_points_equal_fp32_then_cast():
    N, B = 128, 3
    plan = F.DevicePlan(N, DEV)
    lib = plan.lib
    P = _lib.ptr
    img = synth.images(B, N, seed=8).to(DEV)
    psf = torch.rand(3, N, N, generator=torch.Generator().manual_seed(1)).to(DEV)
    psf /= psf.sum()
    ws = torch.empty(lib.b200cam_sensor_workspace_bytes(N, B, 1), dtype=torch.uint8, device=DEV)
    sbytes = lib.b200cam_spectrum_bytes(N, B) // 4

    def bufs():
        return dict(img_max=torch.empty(B, device=DEV), tc=torch.empty(B, dtype=torch.int32, device=DEV),
                    tp=torch.empty(B, 8, dtype=torch.int32, device=DEV), otf=torch.empty(plan.otf_floats, device=DEV),
                    spec=torch.empty(sbytes, device=DEV))
    a, b = bufs(), bufs()
    y32 = torch.empty(B, 3, N, N, device=DEV)
    conv = torch.empty_like(y32)
    y16 = torch.empty(B, 3, N, N, device=DEV, dtype=BF16)
    _lib.check(lib.b200cam_sensor_fwd_ex(P(img), P(psf), P(y32), P(a["img_max"]), P(a["tc"]), P(a["tp"]), P(a["otf"]), P(a["spec"]),
                                         P(ws), ws.numel(), B, N, _stream(), 0, None, 0.0, 0))
    _lib.check(lib.b200cam_sensor_fwd_bf16(P(img), P(psf), P(conv), P(y16), P(b["img_max"]), P(b["tc"]), P(b["tp"]), P(b["otf"]),
                                           P(b["spec"]), P(ws), ws.numel(), B, N, _stream(), 0, None, 0.0, 0))
    assert _bits_equal(y16, y32.to(BF16))
    for k in ("img_max", "tc", "otf", "spec"):
        assert _bits_equal(a[k], b[k]), k
    _same_ties(a, b)
    # split forward: rows, then finish
    c = bufs()
    y16b = torch.empty_like(y16)
    _lib.check(lib.b200cam_sensor_rows(P(img), P(c["spec"]), P(c["img_max"]), P(c["tc"]), B, N, _stream()))
    _lib.check(lib.b200cam_sensor_finish_bf16(P(psf), P(conv), P(y16b), P(c["img_max"]), P(c["tc"]), P(c["tp"]), P(c["otf"]),
                                              P(c["spec"]), 0, P(ws), ws.numel(), B, N, _stream(), 0, None, 0.0, 0))
    assert _bits_equal(y16b, y16)
    _same_ties(a, c)
    # backward
    g16 = (synth.upstream_grad(B, N, seed=2) * 1e-2).to(DEV, BF16)
    g32 = g16.float()
    out = []
    for bf in (False, True):
        gp = torch.empty(3, N, N, device=DEV)
        gi = torch.empty(B, 3, N, N, device=DEV)
        if bf:
            _lib.check(lib.b200cam_sensor_bwd_bf16(P(g16), P(img), P(a["img_max"]), P(a["tc"]), P(a["tp"]), P(psf), P(a["otf"]),
                                                   P(a["spec"]), P(gp), P(gi), P(ws), ws.numel(), B, N, _stream()))
        else:
            _lib.check(lib.b200cam_sensor_bwd(P(g32), P(img), P(y32), P(a["img_max"]), P(a["tc"]), P(a["tp"]), P(psf), P(a["otf"]),
                                              P(a["spec"]), P(gp), P(gi), P(ws), ws.numel(), B, N, _stream()))
        out.append((gp, gi))
    assert _bits_equal(out[0][0], out[1][0]) and _bits_equal(out[0][1], out[1][1])


def test_lens_abi_bf16_entry_points_equal_fp32_then_cast():
    Pp, B = 64, 2
    n = 2 * Pp
    plan = F.DevicePlan(n, DEV, tables=False)
    lib = plan.lib
    P = _lib.ptr
    gen = torch.Generator().manual_seed(4)
    img = torch.rand(B, 3, Pp, Pp, generator=gen).to(DEV)
    k = torch.rand(3, n, n, generator=gen).to(DEV)
    raw = torch.empty(B, 3, Pp, Pp, device=DEV)
    gmax = torch.zeros(1, device=DEV)
    otf = torch.empty(plan.otf_floats, device=DEV)
    spec = torch.empty(lib.b200cam_spectrum_bytes(n, B) // 4, device=DEV)
    ws = torch.empty(lib.b200cam_lens_sensor_workspace_bytes(Pp, B), dtype=torch.uint8, device=DEV)
    _lib.check(lib.b200cam_lens_sensor_fwd(P(img), P(k), P(raw), P(gmax), P(otf), P(spec), P(ws), ws.numel(), B, Pp, _stream()))
    y32 = torch.empty_like(raw)
    y16 = torch.empty(raw.shape, dtype=BF16, device=DEV)
    _lib.check(lib.b200cam_lens_normalise_ex(P(raw), P(gmax), P(y32), raw.numel(), _stream(), 0, None, 0.0, 0))
    _lib.check(lib.b200cam_lens_normalise_bf16(P(raw), P(gmax), P(y16), raw.numel(), _stream(), 0, None, 0.0, 0))
    assert _bits_equal(y16, y32.to(BF16))
    g16 = (torch.rand(B, 3, Pp, Pp, generator=gen) * 1e-2).to(DEV, BF16)
    g32 = g16.float()
    res = []
    for gy, dot, bwd in ((g32, lib.b200cam_lens_sensor_dot, lib.b200cam_lens_sensor_bwd),
                         (g16, lib.b200cam_lens_sensor_dot_bf16, lib.b200cam_lens_sensor_bwd_bf16)):
        dt = torch.empty(2, device=DEV)
        _lib.check(dot(P(gy), P(raw), P(gmax), P(dt), P(ws), ws.numel(), B, Pp, _stream()))
        coef = (dt[0] / (gmax[0] * dt[1].clamp(min=1.0))).reshape(1)
        gk = torch.empty(3, n, n, device=DEV)
        gi = torch.empty(B, 3, Pp, Pp, device=DEV)
        _lib.check(bwd(P(gy), P(raw), P(gmax), P(coef), P(otf), P(spec), P(gk), P(gi), P(ws), ws.numel(), B, Pp, _stream()))
        res.append((dt, gk, gi))
    for x, y in zip(*res):
        assert _bits_equal(x, y)
