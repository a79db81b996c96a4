"""GPU (-m gpu): the read-out of the Image_Caption camera (``b200cam.lens.OpticsZernike``) - uint8 images read by the sensor
kernels, and the opt-in sensor noise + quantisation epilogue (``sensor_noise_sigma`` / ``sensor_quant_bits``)."""
import ctypes

import pytest
import torch

from b200cam import _lib
from b200cam.lens import OpticsZernike
from conftest import rel_l2

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
# (wave resolution, patch): the shipped geometry, a small fused one, the CircConv path (P = 32) and the torch expression of the
# constructor default patch 368 (736^2 transform, not a power of two)
FUSED = [(896, 256), (128, 64)]
UNFUSED = [(64, 32), (736, 368)]


def make(wave, patch, tol=None, terms=10):
    cam = OpticsZernike(input_shape=[1, patch, patch, 3], device=DEV, wave_resolution=(wave, wave), patch_size=patch,
                        sample_interval=3e-6, zernike_terms=terms, height_tolerance=tol).to(DEV)
    with torch.no_grad():
        cam.zernike_coeffs_train.fill_(-22.0 * (wave / 896) ** 2)
        cam.zernike_coeffs_no_train2[0] = 0.3
    return cam


def images(B, patch, seed):
    g = torch.Generator().manual_seed(seed)
    u8 = torch.randint(0, 256, (B, 3, patch, patch), generator=g, dtype=torch.uint8)
    u8[0, 1, patch // 3, patch // 5] = 255
    w = torch.rand(B, 3, patch, patch, generator=g)
    return u8.to(DEV), w.to(DEV)


def step(cam, img, w, seed=None, **kw):
    """sensor, psf and dL/d(defocus) of one forward + backward; `seed` reseeds torch before the call (tolerance / noise draws)."""
    if seed is not None:
        torch.manual_seed(seed)
    cam.zernike_coeffs_train.grad = None
    sensor, psf, _, _ = cam(img, **kw)
    (sensor * w).sum().backward()
    return sensor.detach(), psf.detach(), cam.zernike_coeffs_train.grad.clone()


@pytest.mark.parametrize("wave,patch", FUSED + UNFUSED)
@pytest.mark.parametrize("tol", [None, 20e-9])
def test_uint8_images_match_float_images_divided_by_255(wave, patch, tol):
    """cam(u8) is bit-identical to cam(u8.float() / 255.0) - sensor, PSF and the gradient of the trainable coefficient - with
    and without the lens tolerance noise (reseeded before each call)."""
    if tol is not None and (wave, patch) in UNFUSED:
        pytest.skip("the tolerance field is drawn the same way on every path; covered by the fused geometries")
    B = 3 if patch <= 256 else 2
    u8, w = images(B, patch, seed=patch + 1)
    cam = make(wave, patch, tol)
    a = step(cam, u8, w, seed=7)
    b = step(cam, u8.float() / 255.0, w, seed=7)
    assert a[0].dtype == torch.float32 and a[0].shape == u8.shape
    assert float(a[0].max()) == 1.0
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def test_uint8_row_kernel_reads_every_value_like_torch():
    """The uint8 loader alone: every value 0 ... 255 in the image, raw output and batch maximum of the forward equal the fp32
    entry point's on u8.float() / 255.0 (torch multiplies by the fp32 reciprocal of the CPU scalar: x * fp32(1/255)).  The
    saved spectrum is not compared: only its live rows are written."""
    from b200cam import functional as F
    P, B = 64, 2
    n = 2 * P
    plan = F.DevicePlan(n, DEV, tables=False)
    lib = plan.lib
    u8 = (torch.arange(B * 3 * P * P, device=DEV) % 256).to(torch.uint8).reshape(B, 3, P, P)
    xf = u8.float() / 255.0
    assert torch.equal(torch.unique(u8), torch.arange(256, device=DEV, dtype=torch.uint8))
    k = torch.rand(3, n, n, generator=torch.Generator().manual_seed(2)).to(DEV)
    outs = []
    for fn, img in ((lib.b200cam_lens_sensor_fwd_u8, u8), (lib.b200cam_lens_sensor_fwd, xf)):
        raw = torch.empty(B, 3, P, P, device=DEV)
        gmax = torch.zeros(1, device=DEV)
        otf = torch.empty(plan.otf_floats, device=DEV)
        spectrum = torch.empty(lib.b200cam_spectrum_bytes(n, B) // 4, device=DEV)
        ws = torch.empty(lib.b200cam_lens_sensor_workspace_bytes(P, B), dtype=torch.uint8, device=DEV)
        _lib.check(fn(_lib.ptr(img), _lib.ptr(k), _lib.ptr(raw), _lib.ptr(gmax), _lib.ptr(otf), _lib.ptr(spectrum), _lib.ptr(ws),
                      ws.numel(), B, P, F._stream()))
        outs.append((raw, gmax))
    for x, y in zip(*outs):
        assert torch.equal(x, y)


@pytest.mark.parametrize("wave,patch", [(128, 64), (896, 256), (736, 368)])
def test_opt_in_sensor_noise_and_quantisation(wave, patch):
    """With sigma and 8 bits the sensor image is round(clamp(y_plain + sigma * n, 0, 1) * L) / L for the SAME torch.randn tensor
    n; a value within float rounding of a quantisation boundary may fall on either side, so at most 0.1 % of the pixels may
    differ, each by exactly one level.  Noise only: rel-L2 <= 1e-4.  The gradient is the plain read-out's (straight through).
    736/368 runs the torch expression of the epilogue, the others the normalise kernel."""
    B = 3 if patch <= 256 else 2
    u8, w = images(B, patch, seed=3)
    img = u8.float() / 255.0
    sigma, bits = 0.02, 8
    L = float(2 ** bits - 1)
    noise = torch.randn(B, 3, patch, patch, generator=torch.Generator(device=DEV).manual_seed(11), device=DEV)
    cam = make(wave, patch)
    y_plain, _, g_plain = step(cam, img, w)
    cam.sensor_noise_sigma, cam.sensor_quant_bits = sigma, bits
    y, _, g = step(cam, img, w, noise=noise)
    ref = torch.round(torch.clamp(y_plain + sigma * noise, 0.0, 1.0) * L) / L
    diff = (y - ref).abs()
    assert float(diff.max()) <= 1.0 / L + 1e-6
    assert float((diff > 1e-6).float().mean()) <= 1e-3
    assert torch.all((y * L - torch.round(y * L)).abs() < 1e-3)                 # on the quantisation grid
    assert torch.equal(g, g_plain)
    cam.sensor_quant_bits = 0
    y2, _, g2 = step(cam, img, w, noise=noise)
    assert rel_l2(y2, y_plain + sigma * noise) <= 1e-4
    assert torch.equal(g2, g_plain)
    # quantisation only: the plain image on the grid
    cam.sensor_noise_sigma, cam.sensor_quant_bits = 0.0, bits
    y3, _, _ = step(cam, u8, w)
    ref3 = torch.round(torch.clamp(y_plain, 0.0, 1.0) * L) / L
    assert float(((y3 - ref3).abs() > 1e-6).float().mean()) <= 1e-3


def test_noise_is_drawn_after_the_tolerance_field():
    """sigma > 0 and no noise given: the module draws torch.randn shaped like the batch AFTER the lens tolerance field, so a
    seeded call equals one given that draw explicitly."""
    wave, patch, B, sigma = 128, 64, 2, 0.05
    u8, w = images(B, patch, seed=5)
    cam = make(wave, patch, tol=20e-9)
    cam.sensor_noise_sigma = sigma
    y, _, _ = step(cam, u8, w, seed=4)
    torch.manual_seed(4)
    torch.rand([1, wave, wave, 1], device=DEV)                                  # the tolerance field (PhasePlate._build)
    noise = torch.randn(u8.shape, device=DEV)
    y2, _, _ = step(cam, u8, w, seed=4, noise=noise)
    assert torch.equal(y, y2)
    y3, _, _ = step(cam, u8, w, seed=5)
    assert not torch.equal(y, y3)


@pytest.mark.parametrize("wave,patch", [(128, 64), (736, 368)])
def test_read_out_off_is_bit_identical_to_the_plain_module(wave, patch):
    """Both attributes at 0 (after having been on) give the output of a module that never had them set."""
    B = 2
    u8, w = images(B, patch, seed=9)
    plain = step(make(wave, patch), u8, w)
    cam = make(wave, patch)
    cam.sensor_noise_sigma, cam.sensor_quant_bits = 0.1, 6
    step(cam, u8, w)
    cam.sensor_noise_sigma, cam.sensor_quant_bits = 0.0, 0
    again = step(cam, u8, w)
    for x, y in zip(plain, again):
        assert torch.equal(x, y)


def test_normalise_ex_without_flags_is_the_plain_division():
    """flags = 0: b200cam_lens_normalise_ex is b200cam_lens_normalise, |raw| / gmax exactly (torch's division on the GPU)."""
    lib = _lib.load_library()
    g = torch.Generator().manual_seed(1)
    raw = (torch.randn(4, 3, 64, 64, generator=g) * 3).to(DEV)
    gmax = raw.abs().max().reshape(1)
    y0, y1 = torch.empty_like(raw), torch.empty_like(raw)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _lib.check(lib.b200cam_lens_normalise(_lib.ptr(raw), _lib.ptr(gmax), _lib.ptr(y0), raw.numel(), stream))
    _lib.check(lib.b200cam_lens_normalise_ex(_lib.ptr(raw), _lib.ptr(gmax), _lib.ptr(y1), raw.numel(), stream, 0, None, 0.0, 0))
    assert torch.equal(y0, y1)
    assert torch.equal(y0, raw.abs() / gmax)


def test_caption_step_with_uint8_and_read_out_is_graph_capturable():
    """Forward + backward with uint8 images and noise + quantisation on, captured in a CUDA graph, replays to the eager
    result (the noise tensor is a static input of the step)."""
    wave, patch, B = 128, 64, 3
    u8, w = images(B, patch, seed=12)
    noise = torch.randn(u8.shape, generator=torch.Generator(device=DEV).manual_seed(2), device=DEV)
    cam = make(wave, patch)
    cam.sensor_noise_sigma, cam.sensor_quant_bits = 0.03, 8
    out = {}

    def run():
        cam.zernike_coeffs_train.grad = None
        sensor, _, _, _ = cam(u8, noise=noise)
        torch.autograd.backward([sensor], [w])
        out["sensor"] = sensor

    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run()
        eager_y, eager_g = out["sensor"].detach().clone(), cam.zernike_coeffs_train.grad.clone()
        run()
    torch.cuda.current_stream().wait_stream(side)
    out.clear()
    cam.zernike_coeffs_train.grad = None
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        run()
    y_static = out["sensor"]
    for _ in range(2):
        cam.zernike_coeffs_train.grad.zero_()
        graph.replay()
        torch.cuda.synchronize()
        assert torch.equal(y_static, eager_y)
        assert torch.equal(cam.zernike_coeffs_train.grad, eager_g)
