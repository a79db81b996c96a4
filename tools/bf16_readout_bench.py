"""bf16 hand-over of the sensor image to a bf16 downstream network: fp32 camera + cast against ``sensor_dtype = torch.bfloat16``.

For each camera at the two batch sizes of the project's workloads (sensor 256 x 256: config 2 = batch 64, the 3cam geometry =
batch 128; Face-DeId ``Camera(N=256, zernike_terms=50)``, Image_Caption ``OpticsZernike`` 896/256/T=350 with the height
tolerance on), one training step = camera forward + a bf16 consumer stand-in ``(y.to(bf16) * w_bf16).sum()`` (+ the
Face-DeId regularisers) + backward into the camera parameters.  Two arms:
  fp32_cast : sensor_dtype = float32; the .to(bf16) is a cast kernel each way (autocast's boundary)
  bf16      : sensor_dtype = bfloat16; the .to(bf16) is a no-op, the kernels write y / read dL/dy in bf16
Per arm:
  * step_ms   : the step replayed from a CUDA graph, CUDA events over --steps replays after warm-up; the two arms alternate
                --reps times (every sample is reported, and the median)
  * kernel_us : mean device time per launch of the normalise and gradient-row kernels and of the cast kernels, from
                torch.profiler over eager steps in a run of its own (after the timed legs)
  * peak_mb   : torch.cuda.max_memory_allocated over one eager step, minus what was allocated before it
The card's name, power limit and max SM clock are read in the same run.  Prints one JSON line; --out FILE also writes it.

  python tools/bf16_readout_bench.py [--steps 200] [--reps 5] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import b200cam.synthetic as synth               # noqa: E402
from b200cam.lens import OpticsZernike          # noqa: E402
from b200cam.optics import Camera               # noqa: E402

BF16 = torch.bfloat16
ARMS = (("fp32_cast", torch.float32), ("bf16", BF16))


def gpu_info(dev) -> dict:
    info = {"name": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", f"--id={dev.index}", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"unavailable ({exc})"
    return info


def make_workload(camera: str, B: int, dev):
    """(module, images, step(dtype) -> tensor checksum, description)"""
    g = torch.Generator().manual_seed(B)
    if camera == "face_deid":
        N = 256
        torch.manual_seed(0)
        cam = Camera(device=dev, N=N, zernike_terms=50)
        img = synth.images(B, N, seed=B).to(dev)
        w = synth.upstream_grad(B, N, seed=B + 1).to(dev, BF16)
        desc = f"Camera N={N} T=50, batch {B}, fwd + bf16 consumer + bwd into Zer_train"

        def step(dtype):
            cam.sensor_dtype = dtype
            cam.Zer_train.grad = None
            y = cam(img)
            loss = (y.to(BF16) * w).sum().float() + 0.3 * cam.loss_rad + 1.7 * cam.centering_loss
            loss.backward()
            return cam.Zer_train.grad.reshape(-1)[0]
    else:
        P = 256
        cam = OpticsZernike(input_shape=[None, P, P, 3], device=dev, zernike_terms=350, patch_size=P, height_tolerance=2e-8,
                            sensor_distance=0.025, wave_resolution=[896, 896], sample_interval=3e-06, upsample=False).to(dev)
        img = torch.randint(0, 256, (B, 3, P, P), generator=g, dtype=torch.uint8).to(dev)
        w = torch.rand(B, 3, P, P, generator=g).to(dev, BF16)
        desc = f"OpticsZernike 896/{P}/T=350, height tolerance 2e-8, uint8 images, batch {B}, fwd + bf16 consumer + bwd"

        def step(dtype):
            cam.sensor_dtype = dtype
            cam.zernike_coeffs_train.grad = None
            y, _, _, _ = cam(img)
            (y.to(BF16) * w).sum().float().backward()
            return cam.zernike_coeffs_train.grad.reshape(-1)[0]
    return cam, step, desc


def capture(step, dtype, dev):
    cur = torch.cuda.current_stream(dev)
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        for _ in range(3):
            step(dtype)
    cur.wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        step(dtype)
    return graph


def time_replays(graph, n, warmup=10):
    for _ in range(warmup):
        graph.replay()
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    for _ in range(n):
        graph.replay()
    t1.record()
    torch.cuda.synchronize()
    return t0.elapsed_time(t1) / n


def kernel_group(key: str):
    """normalise: K4 / the caption normalise; grad_rows: the persistent row kernel (Face-DeId: it also runs the image rows of
    the forward - the fp32 arm then shows 2 launches per step, the bf16 arm one of each instantiation) and the caption's
    gradient row kernel; elementwise: torch's element-wise kernels, the dtype casts among them"""
    if "k_normalise" in key or "k_lnormalise" in key:
        return "normalise"
    if "k_rows_r2c_persist" in key or ("k_lrows_r2c" in key and "GradLoad" in key):
        return "grad_rows"
    if "copy_kernel" in key or "elementwise_kernel" in key:
        return "elementwise"
    return None


def profile_kernels(step, dtype, steps=10):
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        step(dtype)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step(dtype)
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


def peak_memory(step, dtype, dev):
    step(dtype)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    step(dtype)
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated(dev) - base) / 2 ** 20


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
    res = {"gpu": gpu_info(dev), "steps": args.steps, "reps": args.reps, "workloads": {}}
    for camera in ("face_deid", "caption"):
        for B in (64, 128):
            cam, step, desc = make_workload(camera, B, dev)
            graphs = {name: capture(step, dtype, dev) for name, dtype in ARMS}
            samples = {name: [] for name, _ in ARMS}
            for _ in range(args.reps):                       # the arms alternate
                for name, _ in ARMS:
                    samples[name].append(time_replays(graphs[name], args.steps))
            del graphs
            torch.cuda.synchronize()
            entry = {"workload": desc}
            for name, dtype in ARMS:
                entry[name] = {"step_ms_median": statistics.median(samples[name]), "step_ms_samples": samples[name],
                               "peak_mb": peak_memory(step, dtype, dev)}
            for name, dtype in ARMS:
                entry[name]["kernels"] = profile_kernels(step, dtype)
            a, b = entry["fp32_cast"]["step_ms_median"], entry["bf16"]["step_ms_median"]
            entry["bf16_minus_fp32_cast_ms"] = b - a
            res["workloads"][f"{camera}_B{B}"] = entry
            print(json.dumps({f"{camera}_B{B}": {k: entry[k]["step_ms_median"] for k, _ in ARMS}}), flush=True)
            del cam, step
            torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
