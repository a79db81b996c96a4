"""The opt-in sensor noise drawn in the normalise kernels (``sensor_noise_rng = "philox"``) against the torch.randn tensor
(``"torch"``, the default) on both cameras.

Workloads: the Face-DeId ``Camera(N=256, zernike_terms=50)`` (config 2) and the Image_Caption ``OpticsZernike`` 896/256/T=350
with the height tolerance on (the 3cam geometry, uint8 images), each at batch 64 and 128.  One training step = camera forward
with ``sensor_noise_sigma = 0.01`` (and ``sensor_quant_bits`` 0 or 8) + ``(y * w).sum()`` (+ the Face-DeId regularisers) +
backward into the camera parameters.  Two arms per (workload, quantisation):
  torch  : the noise is a torch.randn tensor shaped like the batch, written by torch's kernel and read by the normalise kernel
  philox : one torch.randint key; the normalise kernel draws the noise itself (Philox4x32-10 + Box-Muller per float4)
Per arm:
  * step_ms   : the step replayed from a CUDA graph (a new key / a new randn draw on every replay), CUDA events over --steps
                replays after warm-up; the two arms alternate --reps times (every sample is reported, and the median)
  * kernel_us : mean device time per launch of the normalise kernels and of torch's normal-distribution kernel, from
                torch.profiler over eager steps in a run of its own (after the timed legs)
  * peak_mb   : torch.cuda.max_memory_allocated over one eager step, minus what was allocated before it
The card's name, power limit and max SM clock are read in the same run.  Prints one JSON line; --out FILE also writes it.

  python tools/philox_noise_bench.py [--steps 200] [--reps 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import statistics
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
sys.path.insert(0, str(Path(__file__).resolve().parent))
import b200cam.synthetic as synth               # noqa: E402
from b200cam.lens import OpticsZernike          # noqa: E402
from b200cam.optics import Camera               # noqa: E402
from bf16_readout_bench import capture, gpu_info, peak_memory, time_replays   # noqa: E402

ARMS = ("torch", "philox")
SIGMA = 0.01


def make_workload(camera: str, B: int, dev):
    """(module, step(arm) -> tensor, description)"""
    g = torch.Generator().manual_seed(B)
    if camera == "face_deid":
        N = 256
        torch.manual_seed(0)
        cam = Camera(device=dev, N=N, zernike_terms=50)
        img = synth.images(B, N, seed=B).to(dev)
        w = synth.upstream_grad(B, N, seed=B + 1).to(dev)
        desc = f"Camera N={N} T=50, batch {B}, fwd + (y * w).sum() + bwd into Zer_train"

        def step(arm):
            cam.sensor_noise_rng = arm
            cam.Zer_train.grad = None
            y = cam(img)
            ((y * w).sum() + 0.3 * cam.loss_rad + 1.7 * cam.centering_loss).backward()
            return cam.Zer_train.grad.reshape(-1)[0]
    else:
        P = 256
        cam = OpticsZernike(input_shape=[None, P, P, 3], device=dev, zernike_terms=350, patch_size=P, height_tolerance=2e-8,
                            sensor_distance=0.025, wave_resolution=[896, 896], sample_interval=3e-06, upsample=False).to(dev)
        img = torch.randint(0, 256, (B, 3, P, P), generator=g, dtype=torch.uint8).to(dev)
        w = torch.rand(B, 3, P, P, generator=g).to(dev)
        desc = f"OpticsZernike 896/{P}/T=350, height tolerance 2e-8, uint8 images, batch {B}, fwd + (y * w).sum() + bwd"

        def step(arm):
            cam.sensor_noise_rng = arm
            cam.zernike_coeffs_train.grad = None
            y, _, _, _ = cam(img)
            (y * w).sum().backward()
            return cam.zernike_coeffs_train.grad.reshape(-1)[0]
    cam.sensor_noise_sigma = SIGMA
    return cam, step, desc


def kernel_group(key: str):
    """normalise: the Face-DeId K4 / the caption normalise (the Philox arm runs their _philox instantiations); randn: torch's
    normal-distribution kernel that writes the noise tensor of the torch arm"""
    if "k_normalise" in key or "k_lnormalise" in key:
        return "normalise"
    if "normal" in key and "distribution" in key:
        return "randn"
    return None


def profile_kernels(step, arm, steps=10):
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        step(arm)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step(arm)
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        group = kernel_group(ev.key)
        if group is None:
            continue
        t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
        out[ev.key[:160]] = {"group": group, "us_per_launch": t / max(ev.count, 1), "launches_per_step": ev.count / steps,
                             "us_per_step": t / steps}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(dev), "sigma": SIGMA, "steps": args.steps, "reps": args.reps, "workloads": {}}
    for camera in ("face_deid", "caption"):
        for B in (64, 128):
            cam, step, desc = make_workload(camera, B, dev)
            for bits in (0, 8):
                cam.sensor_quant_bits = bits
                graphs = {arm: capture(step, arm, dev) for arm in ARMS}
                samples = {arm: [] for arm in ARMS}
                for _ in range(args.reps):                   # the arms alternate
                    for arm in ARMS:
                        samples[arm].append(time_replays(graphs[arm], args.steps))
                del graphs
                torch.cuda.synchronize()
                entry = {"workload": desc, "quant_bits": bits}
                for arm in ARMS:
                    entry[arm] = {"step_ms_median": statistics.median(samples[arm]), "step_ms_samples": samples[arm],
                                  "peak_mb": peak_memory(step, arm, dev)}
                for arm in ARMS:
                    entry[arm]["kernels"] = profile_kernels(step, arm)
                entry["philox_minus_torch_ms"] = entry["philox"]["step_ms_median"] - entry["torch"]["step_ms_median"]
                name = f"{camera}_B{B}_q{bits}"
                res["workloads"][name] = entry
                print(json.dumps({name: {arm: entry[arm]["step_ms_median"] for arm in ARMS}}), flush=True)
            del cam, step
            torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
