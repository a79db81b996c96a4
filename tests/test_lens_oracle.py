"""CPU: pins ``oracle/lens_oracle.py`` (Image_Caption camera restatement) to the UNMODIFIED reference module
``Image_Caption/Camera/Lens.py`` (imported through ``oracle/ref_shim.py`` when B200CAM_REFERENCE_ROOT is set) and to
the committed golden vectors written from it by ``oracle/make_golden.py``."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR, rel_l2
from oracle import lens_oracle as lo
from oracle import ref_shim
import b200cam.zernike as zern

CASES = {"caption_w128_p64_b2": dict(wave=128, patch=64, B=2, terms=10),
         # the shipped geometry (train.py:64-66: wave 896 -> 1344^2 propagation, patch 256 -> 512^2 convolution), few terms
         "caption_w896_p256_b2": dict(wave=896, patch=256, B=2, terms=10)}


def inputs(case):
    c = CASES[case]
    g = torch.Generator().manual_seed(77)
    img = torch.rand(c["B"], 3, c["patch"], c["patch"], generator=g)
    img[:, :, c["patch"] // 3, c["patch"] // 2] += 3.0          # a clear maximum (arg-max margin for the global max)
    w = torch.rand(c["B"], 3, c["patch"], c["patch"], generator=g)
    coeffs = torch.zeros(c["terms"], 1, 1)
    coeffs[3] = -22.0
    coeffs[5] = 0.7
    coeffs[8] = -0.4
    return img, w, coeffs


def oracle_run(case):
    c = CASES[case]
    img, w, coeffs = inputs(case)
    cfg = lo.LensConfig(wave_res=c["wave"], patch=c["patch"], sample_interval=3e-6)
    vol = torch.tensor(zern.zernike_volume(c["wave"], c["terms"], 1e-6).astype(np.float32))
    cz = coeffs.clone().requires_grad_(True)
    out = lo.lens_forward(img, cz, vol, cfg)
    (out["sensor"] * w).sum().backward()
    return out, cz.grad


@pytest.mark.parametrize("case", list(CASES))
def test_oracle_matches_golden(case):
    gold = np.load(GOLDEN_DIR / f"{case}.npz")
    out, g = oracle_run(case)
    assert rel_l2(out["sensor"], torch.from_numpy(gold["sensor"])) <= 1e-6
    assert rel_l2(out["psf"], torch.from_numpy(gold["psf"])) <= 1e-6
    assert abs(float(g[3]) - float(gold["grad_defocus"].reshape(-1)[0])) <= 1e-4 * abs(float(gold["grad_defocus"].reshape(-1)[0]))


@pytest.mark.skipif(not ref_shim.reference_available(), reason="reference sources not present (B200CAM_REFERENCE_ROOT)")
@pytest.mark.parametrize("case", list(CASES))
def test_oracle_matches_live_reference(case, tmp_path, monkeypatch):
    monkeypatch.chdir(tmp_path)                                  # the reference caches its Zernike volume in cwd
    c = CASES[case]
    img, w, coeffs = inputs(case)
    Lens = ref_shim.load_image_caption_lens()
    cam = Lens.OpticsZernike(input_shape=[1, c["patch"], c["patch"], 3], device=torch.device("cpu"),
                             wave_resolution=(c["wave"], c["wave"]), patch_size=c["patch"], sample_interval=3e-6,
                             zernike_terms=c["terms"], height_tolerance=None)
    with torch.no_grad():
        cam.zernike_coeffs_train.copy_(coeffs[3])
        cam.zernike_coeffs_no_train2.copy_(coeffs[4:])
    sensor, psf, zc, loss = cam(img)
    (sensor * w).sum().backward()
    out, g = oracle_run(case)
    assert loss is None and out["loss"] is None
    assert torch.equal(zc.detach(), coeffs)
    assert rel_l2(out["sensor"], sensor) <= 1e-6
    assert rel_l2(out["psf"], psf) <= 1e-6
    assert abs(float(g[3]) - float(cam.zernike_coeffs_train.grad)) <= 1e-4 * abs(float(g[3]))
