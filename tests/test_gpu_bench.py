"""GPU (-m gpu): ``bench.py --dump-outputs`` writes what the last timed step returned to its caller.  Each test runs the
benchmark in a subprocess for a few steps and repeats that last step eagerly through the module on the same inputs."""
import subprocess
import sys

import numpy as np
import pytest
import torch

import b200cam.synthetic as synth
from conftest import REPO, rel_l2

pytestmark = pytest.mark.gpu
STEPS, SETS = 3, 4                   # the last timed step uses input set (STEPS - 1) % SETS


def run_bench(out_dir, *args):
    cmd = [sys.executable, str(REPO / "bench.py"), "--steps", str(STEPS), "--warmup", "1", "--input-sets", str(SETS),
           "--dump-outputs", str(out_dir), *args]
    res = subprocess.run(cmd, cwd=REPO, capture_output=True, text=True, timeout=900)
    assert res.returncode == 0, (res.stdout + res.stderr)[-3000:]
    return {p.stem: torch.from_numpy(np.load(p)) for p in out_dir.glob("*.npy")}


def test_dump_is_the_last_timed_step_config2(tmp_path):
    from b200cam.optics import Camera
    N, B = 256, 8
    got = run_bench(tmp_path, "--quick", "--batch", str(B))
    assert sorted(got) == ["centering_loss", "grad_h", "loss_rad", "psf", "sensor"]
    assert all(t.dtype == torch.float32 for t in got.values())
    dev = torch.device("cuda", 0)
    torch.manual_seed(0)                                       # bench.py: Camera(..., zernike_terms=12) after this seed
    cam = Camera(device=dev, N=N, zernike_terms=12)
    h = synth.height_map(N).to(dev).requires_grad_(True)
    cam.get_Heith_Map = lambda: h
    r = (STEPS - 1) % SETS
    y = cam(synth.images(B, N, seed=1000 + r).to(dev))
    torch.autograd.backward([y, cam.loss_rad, cam.centering_loss],
                            [synth.upstream_grad(B, N, seed=2000 + r).to(dev), torch.ones((), device=dev),
                             torch.ones((), device=dev)])
    assert rel_l2(got["sensor"], y) <= 1e-5
    assert rel_l2(got["psf"], cam.psfs) <= 1e-5
    assert rel_l2(got["grad_h"], h.grad) <= 1e-5
    assert rel_l2(got["loss_rad"], cam.loss_rad) <= 1e-5 and rel_l2(got["centering_loss"], cam.centering_loss) <= 1e-5
    y_other = cam(synth.images(B, N, seed=1000 + (r + 1) % SETS).to(dev))
    assert rel_l2(got["sensor"], y_other) > 1e-2                # another input set is told apart


def test_dump_is_the_last_timed_step_caption_camera(tmp_path):
    """--config 3cam: every step draws the lens tolerance noise from torch's generator; the benchmark seeds it before the
    timed steps, so the last of them is reproduced by seeding and running that many eager steps."""
    from b200cam.lens import OpticsZernike
    B, P = 2, 256
    got = run_bench(tmp_path, "--config", "3cam", "--batch", str(B))
    assert sorted(got) == ["grad_defocus", "psf", "sensor"]
    dev = torch.device("cuda", 0)
    cam = OpticsZernike(input_shape=[None, P, P, 3], device=dev, zernike_terms=350, patch_size=P, height_tolerance=2e-8,
                        sensor_distance=0.025, wave_resolution=[896, 896], sample_interval=3e-06, upsample=False).to(dev)
    g = torch.Generator().manual_seed(5)                       # bench.py's input sets: images, then upstream gradients
    imgs = [torch.rand(B, 3, P, P, generator=g).to(dev) for _ in range(SETS)]
    ws = [torch.rand(B, 3, P, P, generator=g).to(dev) for _ in range(SETS)]

    def last_step(seed):
        torch.manual_seed(seed)
        for i in range(STEPS):
            cam.zero_grad(set_to_none=True)
            sensor, psf, _, _ = cam(imgs[i % SETS])
            torch.autograd.backward([sensor], [ws[i % SETS]])
        return sensor.detach(), psf.detach(), cam.zernike_coeffs_train.grad.detach().clone()

    sensor, psf, gd = last_step(0)
    assert rel_l2(got["sensor"], sensor) <= 1e-5
    assert rel_l2(got["psf"], psf) <= 1e-5
    assert rel_l2(got["grad_defocus"], gd) <= 1e-4
    _, psf_other, _ = last_step(1)
    assert rel_l2(got["psf"], psf_other) > 1e-4                 # other tolerance noise is told apart
