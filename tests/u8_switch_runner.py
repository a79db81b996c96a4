"""GPU check, for use under an environment switch (B200CAM_TIE_SPECTRAL=1, B200CAM_ONE_PASS=1, B200CAM_PLANE=1, B200CAM_COOP=0):
the Face-DeId camera fed uint8 images equals, bit for bit, the camera fed the same batch converted on the GPU with
``u8.to(torch.float32).div_(255.0)`` - sensor image, PSF, both regularisers and dL/dZer_train.  The switches are read once per
process, so tests/test_gpu_u8_input.py runs this file in a subprocess per switch.  With B200CAM_COOP=0 (the eager PSF chain is
then the multi-kernel one a CUDA graph captures) it also checks that a ``graphed()`` step from uint8 replays the eager step bit
for bit.  Prints one ``U8_SWITCH ... ok=<bool>`` line."""
import os
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import b200cam.synthetic as synth          # noqa: E402
from b200cam.optics import Camera          # noqa: E402

DEV = torch.device("cuda", 0)
BF16 = torch.bfloat16


def u8_images(B, N, seed):
    """a uint8 batch with exact ties: image 0 saturated (every pixel 255), image 1 a constant block, the rest synthetic"""
    u = (synth.images(B, N, seed=seed) * 255.0).round().clamp(0, 255).to(torch.uint8)
    u[0] = 255
    if B > 1:
        u[1, :, N // 4:N // 2, N // 4:N // 2] = 200
    return u.to(DEV)


def bits_equal(a, b) -> bool:
    if a is None or b is None:
        return a is None and b is None
    if a.dtype != b.dtype or a.shape != b.shape:
        return False
    view = {2: torch.int16, 4: torch.int32, 8: torch.int64}[a.element_size()]
    return torch.equal(a.contiguous().view(view), b.contiguous().view(view))


def camera(N, seed=0, terms=10):
    torch.manual_seed(seed)
    return Camera(device=DEV, N=N, zernike_terms=terms)


def face_step(cam, img, g, dtype=torch.float32, noise=None):
    """one eager forward + backward -> (sensor, psf, loss_rad, centering_loss, dL/dZer_train)"""
    cam.sensor_dtype = dtype
    cam.Zer_train.grad = None
    y = cam(img, noise=noise)
    assert y.dtype == dtype
    torch.autograd.backward([y, cam.loss_rad, cam.centering_loss],
                            [g.to(dtype), torch.tensor(0.3, device=DEV), torch.tensor(1.7, device=DEV)])
    return (y.detach().clone(), cam.psfs.detach().clone(), cam.loss_rad.detach().clone(), cam.centering_loss.detach().clone(),
            cam.Zer_train.grad.clone())


def u8_equals_converted(N, B, overlap, dtype, epi, seed=0):
    cam = camera(N, seed)
    cam.overlap_psf = overlap
    u = u8_images(B, N, seed=N + B + seed)
    g = (synth.upstream_grad(B, N, seed=N + 1) * 1e-2).to(DEV)
    noise = None
    if epi:
        cam.sensor_noise_sigma, cam.sensor_quant_bits = 0.02, 8
        noise = torch.randn(B, 3, N, N, generator=torch.Generator(device=DEV).manual_seed(5), device=DEV)
    a = face_step(cam, u, g, dtype, noise)
    b = face_step(cam, u.to(torch.float32).div_(255.0), g, dtype, noise)
    return [bits_equal(x, y) for x, y in zip(a, b)]


def graphed_equals_eager(N=128, B=4):
    cam = camera(N, seed=3)
    u = u8_images(B, N, seed=11)
    g = (synth.upstream_grad(B, N, seed=4) * 1e-2).to(DEV)
    step = cam.graphed(u)
    outs = []
    for _ in range(2):
        cam.Zer_train.grad = None
        y, rad, cen = step(u)
        torch.autograd.backward([y, rad, cen], [g, torch.tensor(0.3, device=DEV), torch.tensor(1.7, device=DEV)])
        outs.append((y.detach().clone(), rad.detach().clone(), cen.detach().clone(), cam.Zer_train.grad.clone()))
    e = face_step(cam, u, g)
    eager = (e[0], e[2], e[3], e[4])
    return [bits_equal(x, y) for x, y in zip(outs[0], outs[1])] + [bits_equal(x, y) for x, y in zip(outs[1], eager)]


def rows_u8_refused(N=256, B=2) -> bool:
    """with the plane kernels selected at N = 256, b200cam_sensor_rows_u8 returns B200CAM_E_BAD_SIZE (the finish call would
    expect the plane layout) and enqueues nothing"""
    import ctypes
    from b200cam import _lib
    from b200cam import functional as F
    plan = F.DevicePlan(N, DEV)
    u = u8_images(B, N, seed=1)
    spec = torch.full((plan.lib.b200cam_spectrum_bytes(N, B) // 4,), 7.0, device=DEV)
    mx, tc = torch.zeros(B, device=DEV), torch.full((B,), 3, dtype=torch.int32, device=DEV)
    rc = plan.lib.b200cam_sensor_rows_u8(_lib.ptr(u), _lib.ptr(spec), _lib.ptr(mx), _lib.ptr(tc), B, N,
                                         ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc == -1 and bool((spec == 7.0).all()) and bool((tc == 3).all())


def main():
    checks = {}
    for N, B in ((256, 5), (128, 3)):
        for overlap in (True, False):
            for dtype in (torch.float32, BF16):
                checks[f"N={N} overlap={overlap} {str(dtype).split('.')[-1]}"] = u8_equals_converted(N, B, overlap, dtype, False)
    if os.environ.get("B200CAM_PLANE") != "1":     # (the opt-in plane kernels have no read-out epilogue)
        checks["N=256 epilogue"] = u8_equals_converted(256, 3, True, torch.float32, True)
    if os.environ.get("B200CAM_COOP") == "0":
        checks["graphed==eager"] = graphed_equals_eager()
    if os.environ.get("B200CAM_PLANE") == "1":
        checks["rows_u8 refuses the plane layout"] = [rows_u8_refused()]
    torch.cuda.synchronize()
    bad = [k for k, v in checks.items() if not all(v)]
    for k in bad:
        print(f"mismatch {k}: {checks[k]}", flush=True)
    switches = " ".join(f"{k}={v}" for k, v in os.environ.items() if k in ("B200CAM_TIE_SPECTRAL", "B200CAM_ONE_PASS",
                                                                          "B200CAM_PLANE", "B200CAM_COOP"))
    print(f"U8_SWITCH {switches} checks={len(checks)} ok={not bad}", flush=True)
    sys.exit(0 if not bad else 1)


if __name__ == "__main__":
    main()
