"""TEST INFRASTRUCTURE ONLY - generate tests/golden/facedeid_*.npz from the live reference.

Run with a checkout of the reference named by ``B200CAM_REFERENCE_ROOT``:

    B200CAM_REFERENCE_ROOT=<reference checkout> python oracle/make_golden.py

Each fixture holds the outputs of the UNMODIFIED reference ``Camera``
(``Face-DeId/Camera/Optics.py:9``, imported through ``oracle/ref_shim.py``) on the
synthetic inputs of ``privacy-preserving-vision_b200/synthetic.py``:
forward sensor image, PSF, the two regulariser scalars and dL/dh for
``L = sum(sensor*w) + loss_rad + centering_loss`` with the height map injected through
``cam.get_Heith_Map = lambda: h`` (SURVEY.md section 8c).  Small cases store their inputs
too; the N=256 case stores only a checksum of the inputs (they are regenerated from
the seed) to keep the repository small.
"""
from __future__ import annotations

import hashlib
import sys
from pathlib import Path

import numpy as np
import torch

REPO = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(REPO))

from oracle import ref_shim  # noqa: E402
import b200cam.synthetic as synth  # noqa: E402

CASES = [
    # name, N, B, store_inputs
    ("facedeid_n64_b2", 64, 2, True),
    ("facedeid_n128_b3", 128, 3, True),
    ("facedeid_n256_b2", 256, 2, False),
]


def digest(*tensors: torch.Tensor) -> str:
    m = hashlib.sha256()
    for t in tensors:
        m.update(t.contiguous().numpy().tobytes())
    return m.hexdigest()


def run_reference(N: int, B: int, seed_img: int = 1000, seed_w: int = 2000, seed_h: int = 1234):
    Camera = ref_shim.load_face_deid_camera()
    torch.manual_seed(0)
    cam = Camera(device="cpu", N=N, zernike_terms=6)   # basis unused: height map is injected
    h = synth.height_map(N, seed_h).requires_grad_(True)
    cam.get_Heith_Map = lambda: h
    img = synth.images(B, N, seed_img)
    w = synth.upstream_grad(B, N, seed_w)
    y = cam(img)
    loss = (y * w).sum() + cam.loss_rad + cam.centering_loss
    loss.backward()
    conv_gap = None
    with torch.no_grad():
        Utils = ref_shim.load_face_deid_utils()
        conv = Utils.conv2D(img, torch.roll(cam.psfs, (-(N // 2), -(N // 2)), (-2, -1)))
        conv_gap = synth.top2_relative_gap(conv).min().item()
    return {
        "img": img, "w": w, "h": h.detach(),
        "sensor": y.detach(), "psf": cam.psfs.detach(),
        "loss_rad": cam.loss_rad.detach().reshape(1), "centering_loss": cam.centering_loss.detach().reshape(1),
        "grad_h": h.grad.detach(), "min_top2_gap": torch.tensor([conv_gap]),
    }


def main() -> None:
    out_dir = REPO / "tests" / "golden"
    out_dir.mkdir(parents=True, exist_ok=True)
    for name, N, B, store_inputs in CASES:
        r = run_reference(N, B)
        assert r["min_top2_gap"].item() >= 1e-5, f"{name}: amax margin too small ({r['min_top2_gap'].item()})"
        payload = {k: v.numpy() for k, v in r.items() if store_inputs or k not in ("img", "w", "h")}
        payload["N"] = np.array([N]); payload["B"] = np.array([B])
        payload["seeds"] = np.array([1000, 2000, 1234])
        payload["input_sha256"] = np.array([digest(r["img"], r["w"], r["h"])])
        payload["torch_version"] = np.array([torch.__version__])
        np.savez_compressed(out_dir / f"{name}.npz", **payload)
        print(name, "gap", r["min_top2_gap"].item(), "loss_rad", r["loss_rad"].item(),
              "centering", r["centering_loss"].item(), "bytes", (out_dir / f"{name}.npz").stat().st_size)
    make_caption_fixture(out_dir)
    make_camera_init_fixture(out_dir, ref_shim.load_face_deid_camera(), "reference")


CAMERA_INIT_ATTRS = ("XY", "FF", "XY2", "rho", "rad", "k", "flmb", "lamb", "u", "x2", "fx1", "r", "r2")


def make_camera_init_fixture(out_dir: Path, Camera, source: str) -> None:
    """tests/golden/camera_init_n64_t10.npz: what ``Camera(N=64, zernike_terms=10)`` holds right after construction
    under torch seed 3 - its state_dict, the buffers the forward reads, the initial lens's height map and phase shift
    and the names of the trainable parameters.  ``source`` records which ``Camera`` class wrote the file."""
    torch.manual_seed(3)
    cam = Camera(N=64, zernike_terms=10)
    sd = cam.state_dict()
    payload = {"source": np.array([source]), "torch_version": np.array([torch.__version__]),
               "state_keys": np.array(list(sd)),
               "trainable": np.array([n for n, p in cam.named_parameters() if p.requires_grad])}
    payload.update({f"sd.{k}": v.detach().numpy() for k, v in sd.items()})
    payload.update({f"attr.{n}": getattr(cam, n).detach().numpy() for n in CAMERA_INIT_ATTRS})
    with torch.no_grad():
        payload["heith_map"] = cam.get_Heith_Map().numpy()
        payload["phase_shift"] = cam.get_phase_shift().numpy()
    np.savez_compressed(out_dir / "camera_init_n64_t10.npz", **payload)
    print("wrote camera_init_n64_t10 from", source)


def make_caption_fixture(out_dir: Path) -> None:
    """tests/golden/caption_*.npz: outputs of the UNMODIFIED ``OpticsZernike`` (Image_Caption/Camera/Lens.py:11) on
    the seeded inputs of tests/test_lens_oracle.py (height tolerance off; small wave grid so the file stays small)."""
    import os
    import tempfile
    sys.path.insert(0, str(REPO / "tests"))
    import test_lens_oracle as tlo
    Lens = ref_shim.load_image_caption_lens()
    for case, c in tlo.CASES.items():
        img, w, coeffs = tlo.inputs(case)
        cwd = os.getcwd()
        with tempfile.TemporaryDirectory() as tmp:
            os.chdir(tmp)                      # the reference writes zernike_volumes/*.npy into cwd
            try:
                cam = Lens.OpticsZernike(input_shape=[1, c["patch"], c["patch"], 3], device=torch.device("cpu"),
                                         wave_resolution=(c["wave"], c["wave"]), patch_size=c["patch"],
                                         sample_interval=3e-6, zernike_terms=c["terms"], height_tolerance=None)
                with torch.no_grad():
                    cam.zernike_coeffs_train.copy_(coeffs[3])
                    cam.zernike_coeffs_no_train2.copy_(coeffs[4:])
                sensor, psf, _, _ = cam(img)
                (sensor * w).sum().backward()
            finally:
                os.chdir(cwd)
        np.savez_compressed(out_dir / f"{case}.npz", sensor=sensor.detach().numpy(), psf=psf.detach().numpy(),
                            grad_defocus=cam.zernike_coeffs_train.grad.numpy())
        print("wrote", case)


if __name__ == "__main__":
    main()
