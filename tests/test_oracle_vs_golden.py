"""CPU: pin the oracle (oracle/camera_oracle.py) to the reference.

1. against the committed golden vectors (outputs of the unmodified reference Camera,
   written by oracle/make_golden.py) - runs anywhere;
2. against the live reference module when B200CAM_REFERENCE_ROOT names a reference checkout.
"""
import pytest
import torch

from conftest import GOLDEN_CASES, load_golden, rel_l2
from oracle import camera_oracle as co
from oracle import ref_shim
import b200cam.synthetic as synth


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_forward_matches_golden(name):
    gold = load_golden(name)
    C = co.build_constants(gold["N"])
    out = co.camera_forward(gold["img"], gold["h"], C)
    # same torch build -> bit-exact; tolerance only guards against a different FFT backend
    assert rel_l2(out["sensor"], gold["sensor"]) <= 1e-6
    assert rel_l2(out["psf"], gold["psf"]) <= 1e-6
    assert abs(out["loss_rad"].item() - gold["loss_rad"].item()) <= 1e-6 * abs(gold["loss_rad"].item())
    assert abs(out["centering_loss"].item() - gold["centering_loss"].item()) <= 1e-5 * abs(gold["centering_loss"].item())


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_autograd_matches_golden(name):
    gold = load_golden(name)
    C = co.build_constants(gold["N"])
    h = gold["h"].clone().requires_grad_(True)
    out = co.camera_forward(gold["img"], h, C)
    ((out["sensor"] * gold["w"]).sum() + out["loss_rad"] + out["centering_loss"]).backward()
    assert rel_l2(h.grad, gold["grad_h"]) <= 1e-5


@pytest.mark.parametrize("name", GOLDEN_CASES)
def test_oracle_closed_form_backward_matches_golden(name):
    """The hand-derived adjoints (what the CUDA kernels implement) reproduce the reference gradient."""
    gold = load_golden(name)
    N = gold["N"]
    C = co.build_constants(N)
    psf, _ = co.psf_from_height(gold["h"], C)
    gpsf, _ = co.sensor_backward(gold["w"], gold["img"], psf, N)
    gpsf = gpsf + co.regulariser_grads(psf, C, 1.0, 1.0)
    gh = co.psf_backward(gpsf, gold["h"], C)
    assert rel_l2(gh, gold["grad_h"]) <= 1e-5


def test_oracle_closed_form_backward_fp64_vs_autograd():
    N, B = 64, 2
    C = co.build_constants(N, torch.float64)
    h = synth.height_map(N).double().requires_grad_(True)
    img = synth.images(B, N).double().requires_grad_(True)
    w = synth.upstream_grad(B, N).double()
    out = co.camera_forward(img, h, C)
    ((out["sensor"] * w).sum() + 0.3 * out["loss_rad"] + 0.7 * out["centering_loss"]).backward()
    with torch.no_grad():
        psf = out["psf"].detach()
        gpsf, gimg = co.sensor_backward(w, img.detach(), psf, N, want_img_grad=True)
        gpsf = gpsf + co.regulariser_grads(psf, C, 0.3, 0.7)
        gh = co.psf_backward(gpsf, h.detach(), C)
    assert rel_l2(gh, h.grad) <= 1e-10
    assert rel_l2(gimg, img.grad) <= 1e-10


def test_amax_tie_splitting_matches_torch():
    """Exact ties of the per-image maximum split the gradient evenly (torch amax backward)."""
    N = 64
    img = torch.zeros(1, 3, N, N, dtype=torch.float64)
    img[0, 0, 5, 7] = 1.0
    img[0, 2, 40, 9] = 1.0                       # two identical impulses -> exact tie after the blur
    psf = torch.zeros(1, 3, N, N, dtype=torch.float64)
    psf[0, :, N // 2, N // 2] = 0.25
    psf[0, :, N // 2 + 1, N // 2] = 0.08
    psf = psf.requires_grad_(True)
    w = synth.upstream_grad(1, N).double()
    y, conv, m = co.sensor_from_psf(img, psf, N)
    assert int((conv == m.reshape(-1, 1, 1, 1)).sum()) == 2
    (y * w).sum().backward()
    gpsf, _ = co.sensor_backward(w, img, psf.detach(), N)
    assert rel_l2(gpsf, psf.grad) <= 1e-12


@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference sources not present (B200CAM_REFERENCE_ROOT)")
@pytest.mark.parametrize("N,B", [(128, 2), (256, 1)])
def test_oracle_matches_live_reference(N, B):
    Camera = ref_shim.load_face_deid_camera()
    torch.manual_seed(0)
    cam = Camera(device="cpu", N=N, zernike_terms=8)
    C = co.build_constants(N)
    # (a) constants
    for name in ("XY", "FF", "XY2", "rho"):
        assert torch.equal(getattr(cam, name), getattr(C, name)), name
    assert torch.equal(cam.rad, C.rad) and torch.equal(cam.flmb, C.flmb) and torch.equal(cam.k, C.k)
    # (b) height map through the Zernike parameters (Optics.py:79-83)
    h_ref = cam.get_Heith_Map()
    h_orc = co.height_map(cam.Zer_no_train, cam.Zer_train, cam.zernike_volume)
    assert torch.equal(h_ref, h_orc)
    # (c) forward + backward with the default-init lens
    img = synth.images(B, N, 77)
    w = synth.upstream_grad(B, N, 78)
    y = cam(img)
    (y * w).sum().add(cam.loss_rad).add(cam.centering_loss).backward()
    zt = cam.Zer_train.detach().clone().requires_grad_(True)
    h2 = co.height_map(cam.Zer_no_train, zt, cam.zernike_volume)
    out = co.camera_forward(img, h2, C)
    ((out["sensor"] * w).sum() + out["loss_rad"] + out["centering_loss"]).backward()
    assert rel_l2(out["sensor"], y) <= 1e-6
    assert rel_l2(out["psf"], cam.psfs) <= 1e-6
    assert rel_l2(zt.grad, cam.Zer_train.grad) <= 1e-5
