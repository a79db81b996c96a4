"""GPU (-m gpu): ``sensor_noise_rng = "philox"`` on both cameras - the opt-in sensor noise drawn inside the normalise kernels
(include/b200cam.h B200CAM_SENSOR_NOISE_PHILOX).

The contract: the output of a Philox step is bit for bit the output of the tensor read-out given
``F.philox_normal(cam.sensor_noise_seed, x.shape)`` as ``noise=``; the value of an element depends only on the key and its
index in the (possibly sharded) batch."""
import numpy as np
import pytest
import torch

import b200cam.synthetic as synth
from b200cam import functional as F
from b200cam.lens import OpticsZernike
from b200cam.optics import Camera

pytestmark = pytest.mark.gpu

DEV = torch.device("cuda", 0)
BF16 = torch.bfloat16
SIGMA = 0.02


def _bits_equal(a: torch.Tensor, b: torch.Tensor) -> bool:
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    view = torch.int16 if a.dtype == BF16 else torch.int32
    return torch.equal(a.contiguous().view(view), b.contiguous().view(view))


# ------------------------------------------------------------------------------------------------------------ Face-DeId
def _camera(N, seed=0, terms=10):
    torch.manual_seed(seed)
    return Camera(device=DEV, N=N, zernike_terms=terms)


def _face_images(B, N, u8, seed):
    img = synth.images(B, N, seed=seed).to(DEV)
    return (img * 255.0).round().clamp(0, 255).to(torch.uint8) if u8 else img


def _face_step(cam, img, g, seed=None, noise=None):
    """sensor and dL/dZer_train of one forward + backward; `seed` reseeds torch before the forward (the key draw)"""
    if seed is not None:
        torch.manual_seed(seed)
    cam.Zer_train.grad = None
    y = cam(img, noise=noise)
    torch.autograd.backward([y, cam.loss_rad, cam.centering_loss],
                            [g.to(y.dtype), torch.tensor(0.3, device=DEV), torch.tensor(1.7, device=DEV)])
    return y.detach(), cam.Zer_train.grad.clone()


FACE_CASES = ([(64, 3, ov, u8, dt, q) for ov in (True, False) for u8 in (False, True) for dt in (torch.float32, BF16)
               for q in (0, 8)]
              + [(256, 8, True, False, torch.float32, 0), (256, 8, False, True, BF16, 8), (256, 8, True, True, torch.float32, 8),
                 (1024, 2, True, False, torch.float32, 8), (1024, 2, False, True, BF16, 0)])


@pytest.mark.parametrize("N,B,overlap,u8,dtype,bits", FACE_CASES)
def test_camera_philox_equals_tensor_read_out_on_materialised_noise(N, B, overlap, u8, dtype, bits):
    cam = _camera(N)
    cam.overlap_psf, cam.sensor_dtype = overlap, dtype
    cam.sensor_noise_sigma, cam.sensor_quant_bits = SIGMA, bits
    img = _face_images(B, N, u8, seed=N + B)
    g = (synth.upstream_grad(B, N, seed=N + 1) * 1e-2).to(DEV)
    cam.sensor_noise_rng = "philox"
    y, gz = _face_step(cam, img, g, seed=11)
    seed = cam.sensor_noise_seed
    assert seed is not None and seed.dtype == torch.int64 and seed.shape == (2,) and int(seed[1]) == 0
    noise = F.philox_normal(seed, img.shape)
    cam.sensor_noise_rng = "torch"
    y_t, gz_t = _face_step(cam, img, g, noise=noise)
    assert cam.sensor_noise_seed is None
    assert _bits_equal(y, y_t)
    # straight through: dL/dZer_train is that of the plain read-out
    cam.sensor_noise_sigma, cam.sensor_quant_bits = 0.0, 0
    _, gz_plain = _face_step(cam, img, g)
    assert _bits_equal(gz, gz_plain) and _bits_equal(gz_t, gz_plain)
    # the noise is there
    assert not torch.equal(y.float(), _face_step(cam, img, g)[0].float())


def test_camera_philox_is_reproducible_and_drawn_at_the_start_of_forward():
    N, B = 64, 3
    cam = _camera(N)
    cam.sensor_noise_sigma, cam.sensor_noise_rng = SIGMA, "philox"
    img = _face_images(B, N, False, seed=2)
    g = (synth.upstream_grad(B, N, seed=3) * 1e-2).to(DEV)
    a = _face_step(cam, img, g, seed=4)[0]
    key_a = cam.sensor_noise_seed.clone()
    b = _face_step(cam, img, g, seed=4)[0]
    c = _face_step(cam, img, g, seed=5)[0]
    assert torch.equal(a, b) and not torch.equal(a, c)
    torch.manual_seed(4)
    key = torch.randint(2**63 - 1, (1,), dtype=torch.int64, device=DEV)
    assert int(key_a[0]) == int(key) and int(key_a[1]) == 0


def test_sigma_zero_draws_nothing_and_the_default_is_unchanged():
    N, B = 64, 2
    img = _face_images(B, N, False, seed=6)
    g = (synth.upstream_grad(B, N, seed=7) * 1e-2).to(DEV)
    cam = _camera(N)
    cam.sensor_noise_rng = "philox"
    torch.manual_seed(1)
    y = _face_step(cam, img, g)[0]
    after = torch.cuda.get_rng_state(DEV)
    assert cam.sensor_noise_seed is None
    torch.manual_seed(1)
    assert torch.equal(after, torch.cuda.get_rng_state(DEV))            # no key was drawn
    cam2 = _camera(N)
    assert torch.equal(y, _face_step(cam2, img, g)[0])
    cam.sensor_noise_rng = "numpy"
    with pytest.raises(ValueError):
        cam(img)


def test_face_sensor_forward_is_split_invariant():
    """the sensor forward on x[:k] and x[k:], each with its first4, concatenates to the forward on x (one seed block)"""
    N, B, k = 128, 5, 2
    cam = _camera(N)
    img = _face_images(B, N, False, seed=8)
    with torch.no_grad():
        psf = cam.get_psf()
        torch.cuda.synchronize()
        plan = cam._plan(DEV)
        key = 0x1234_5678_9ABC_DEF0
        per4 = 3 * N * N // 4
        blk = lambda f4: torch.tensor([key, f4], dtype=torch.int64, device=DEV)       # noqa: E731
        whole = F.sensor_conv(img, psf, plan, None, (blk(0), SIGMA, 8))
        parts = torch.cat((F.sensor_conv(img[:k], psf, plan, None, (blk(0), SIGMA, 8)),
                           F.sensor_conv(img[k:], psf, plan, None, (blk(k * per4), SIGMA, 8))))
    assert _bits_equal(whole, parts)


def test_materialised_images_are_rows_of_the_whole_batch():
    B, N, k, m = 6, 64, 2, 3
    key = 987654321987654321
    whole = F.philox_normal(torch.tensor([key, 0], dtype=torch.int64, device=DEV), (B, 3, N, N))
    part = F.philox_normal(torch.tensor([key, k * 3 * N * N // 4], dtype=torch.int64, device=DEV), (m, 3, N, N))
    assert torch.equal(whole[k:k + m], part)


def test_graphed_step_draws_a_new_key_on_every_replay():
    """each replay gives a new image, which is the noise-free graphed image plus sigma * the materialised noise of that replay's
    seed block (to the rounding of the addition)"""
    N, B = 128, 4
    img = _face_images(B, N, False, seed=9)
    plain_cam = _camera(N, seed=3)
    plain = plain_cam.graphed(img)(img)[0].detach().clone()
    cam = _camera(N, seed=3)
    cam.sensor_noise_sigma, cam.sensor_noise_rng = SIGMA, "philox"
    step = cam.graphed(img)
    ys, seeds = [], []
    for _ in range(3):
        y = step(img)[0]
        torch.cuda.synchronize()
        ys.append(y.detach().clone())
        seeds.append(cam.sensor_noise_seed.clone())
    assert len({int(s[0]) for s in seeds}) == 3
    assert not torch.equal(ys[0], ys[1]) and not torch.equal(ys[1], ys[2])
    for y, s in zip(ys, seeds):
        n = F.philox_normal(s, img.shape)
        assert float((y - plain - SIGMA * n).abs().max()) <= 1e-6


@pytest.mark.parametrize("overlap", [False, True])
def test_peak_memory_drops_by_the_noise_tensor(overlap):
    """peak allocated memory of an eager forward, "torch" against "philox" on the same camera: the B*3*N*N fp32 noise tensor
    is not allocated (the seed block takes one 512-byte allocator block)"""
    N, B = 256, 16
    img = _face_images(B, N, False, seed=10)
    cam = _camera(N)
    cam.overlap_psf, cam.sensor_noise_sigma = overlap, SIGMA
    peaks = {}
    for rng in ("torch", "philox", "torch", "philox"):
        cam.sensor_noise_rng = rng
        with torch.no_grad():
            cam(img)                                   # warm: plans, workspaces, the previous step's tensors released
            torch.cuda.synchronize()
            base = torch.cuda.memory_allocated(DEV)
            torch.cuda.reset_peak_memory_stats(DEV)
            y = cam(img)
            torch.cuda.synchronize()
        peaks[rng] = torch.cuda.max_memory_allocated(DEV) - base
        del y
    noise_bytes = B * 3 * N * N * 4
    assert abs((peaks["torch"] - peaks["philox"]) - noise_bytes) <= 4096, peaks


# ------------------------------------------------------------------------------------------------------------ statistics
def test_noise_statistics():
    shape = (16, 3, 512, 512)                          # 12.6 M draws
    key = 0x0DDBA11CAFEF00D
    z = F.philox_normal(torch.tensor([key, 0], dtype=torch.int64, device=DEV), shape).double()
    n = z.numel()
    assert abs(float(z.mean())) < 5 / np.sqrt(n)
    assert abs(float(z.var()) - 1.0) < 5 * np.sqrt(2 / n)
    assert float(z.abs().max()) <= 5.77

    def corr(a, b):
        a, b = a.reshape(-1), b.reshape(-1)
        return float(((a - a.mean()) * (b - b.mean())).mean() / (a.std() * b.std())), a.numel()

    z2 = F.philox_normal(torch.tensor([key + 1, 0], dtype=torch.int64, device=DEV), shape).double()
    for name, (r, m) in {"x": corr(z[..., :-1], z[..., 1:]), "y": corr(z[..., :-1, :], z[..., 1:, :]),
                         "channel": corr(z[:, :-1], z[:, 1:]), "image": corr(z[:-1], z[1:]), "key": corr(z, z2)}.items():
        assert abs(r) < 5 / np.sqrt(m), (name, r)
    from scipy import stats
    sub = z.reshape(-1)[torch.randperm(n, generator=torch.Generator().manual_seed(0))[:1_000_000].to(DEV)].cpu().numpy()
    assert stats.kstest(sub, "norm").pvalue > 1e-4


# ------------------------------------------------------------------------------------------------------------ caption camera
def _lens(wave, patch, tol=None, terms=10):
    cam = OpticsZernike(input_shape=[1, patch, patch, 3], device=DEV, wave_resolution=(wave, wave), patch_size=patch,
                        sample_interval=3e-6, zernike_terms=terms, height_tolerance=tol).to(DEV)
    with torch.no_grad():
        cam.zernike_coeffs_train.fill_(-22.0 * (wave / 896) ** 2)
        cam.zernike_coeffs_no_train2[0] = 0.3
    return cam


def _lens_images(B, patch, u8, seed):
    g = torch.Generator().manual_seed(seed)
    x = torch.randint(0, 256, (B, 3, patch, patch), generator=g, dtype=torch.uint8)
    w = torch.rand(B, 3, patch, patch, generator=g)
    return (x if u8 else x.float() / 255.0).to(DEV), w.to(DEV)


def _lens_step(cam, img, w, seed=None, noise=None):
    if seed is not None:
        torch.manual_seed(seed)
    cam.zernike_coeffs_train.grad = None
    sensor, _, _, _ = cam(img, noise=noise)
    (sensor.float() * w).sum().backward()
    return sensor.detach(), cam.zernike_coeffs_train.grad.clone()


LENS_CASES = ([(128, 64, u8, dt, q) for u8 in (False, True) for dt in (torch.float32, BF16) for q in (0, 8)]
              + [(896, 256, True, torch.float32, 8), (896, 256, False, BF16, 0), (64, 32, False, torch.float32, 8),
                 (64, 32, True, BF16, 0), (736, 368, False, torch.float32, 8), (736, 368, True, torch.float32, 0)])


@pytest.mark.parametrize("wave,patch,u8,dtype,bits", LENS_CASES)
def test_caption_philox_equals_tensor_read_out_on_materialised_noise(wave, patch, u8, dtype, bits):
    """the fused geometries (P = 64, 256) and the others (P = 32 CircConv, P = 368 torch expression)"""
    B = 3 if patch <= 256 else 2
    cam = _lens(wave, patch, tol=20e-9)
    cam.sensor_dtype = dtype
    cam.sensor_noise_sigma, cam.sensor_quant_bits = SIGMA, bits
    img, w = _lens_images(B, patch, u8, seed=patch)
    cam.sensor_noise_rng = "philox"
    y, gz = _lens_step(cam, img, w, seed=7)
    seed = cam.sensor_noise_seed
    assert seed is not None and int(seed[1]) == 0
    noise = F.philox_normal(seed, img.shape)
    cam.sensor_noise_rng = "torch"
    y_t, gz_t = _lens_step(cam, img, w, seed=7, noise=noise)
    assert _bits_equal(y, y_t)
    cam.sensor_noise_sigma, cam.sensor_quant_bits = 0.0, 0
    _, gz_plain = _lens_step(cam, img, w, seed=7)
    assert _bits_equal(gz, gz_plain) and _bits_equal(gz_t, gz_plain)


def test_caption_key_is_drawn_after_the_tolerance_field():
    wave, patch, B = 128, 64, 2
    img, w = _lens_images(B, patch, True, seed=5)
    cam = _lens(wave, patch, tol=20e-9)
    cam.sensor_noise_sigma, cam.sensor_noise_rng = SIGMA, "philox"
    y, _ = _lens_step(cam, img, w, seed=4)
    torch.manual_seed(4)
    torch.rand([1, wave, wave, 1], device=DEV)                                  # the tolerance field (PhasePlate._build)
    key = torch.randint(2**63 - 1, (1,), dtype=torch.int64, device=DEV)
    assert int(cam.sensor_noise_seed[0]) == int(key)
    y2, _ = _lens_step(cam, img, w, seed=4)
    y3, _ = _lens_step(cam, img, w, seed=5)
    assert torch.equal(y, y2) and not torch.equal(y, y3)
