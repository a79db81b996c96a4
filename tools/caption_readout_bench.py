"""Read-out of the Image_Caption camera on the GPU: fp32 against uint8 images, and the cost of the noise + quantisation epilogue.

Workload: bench.py --config 3cam (OpticsZernike 896/256/T=350, height tolerance on, batch 128, forward + backward into the
trainable coefficient), with that bench's loops:
* step_*   : the module step replayed from a CUDA graph, images resident on the GPU (fp32, uint8, fp32 + 8-bit quantiser with
             sigma = 0.01 noise drawn by the module), CUDA events over `--steps` replays;
* e2e_*    : pinned host images copied on a copy stream beside the compute of the previous step (two device buffers), the
             step replayed from a CUDA graph per buffer, sensor checksum + gradient read back every step;
* kernel_us: the forward row kernel k_lrows_r2c<512, ImgLoad> against <512, ImgLoadU8>, mean device time per launch from a
             torch.profiler run of its own (after the timed legs).
Prints one JSON line with the GPU name and power limit read in the same run; --out FILE also writes it there.

  python tools/caption_readout_bench.py [--steps 100] [--batch 128] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from b200cam.lens import OpticsZernike      # noqa: E402

P = 256


def gpu_info(dev) -> dict:
    info = {"name": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", f"--id={dev.index}", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"unavailable ({exc})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--batch", type=int, default=128)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    B = args.batch
    cam = OpticsZernike(input_shape=[None, P, P, 3], device=dev, zernike_terms=350, patch_size=P, height_tolerance=2e-8,
                        sensor_distance=0.025, wave_resolution=[896, 896], sample_interval=3e-06, upsample=False).to(dev)
    g = torch.Generator().manual_seed(5)
    host_u8 = torch.randint(0, 256, (B, 3, P, P), generator=g, dtype=torch.uint8).pin_memory()
    host_f32 = (host_u8.float() / 255.0).pin_memory()
    w = torch.rand(B, 3, P, P, generator=g).to(dev)
    cur = torch.cuda.current_stream(dev)

    def compute(img):
        cam.zero_grad(set_to_none=True)
        sensor, _, _, _ = cam(img)
        torch.autograd.backward([sensor], [w])
        return torch.stack([sensor.detach().sum(), cam.zernike_coeffs_train.grad.reshape(-1)[0]])

    def capture(img):
        side = torch.cuda.Stream(device=dev)
        side.wait_stream(cur)
        with torch.cuda.stream(side):
            for _ in range(2):
                compute(img)
        cur.wait_stream(side)
        torch.cuda.synchronize()
        cam.zero_grad(set_to_none=True)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = compute(img)
        return graph, out

    def time_replays(graph, n):
        for _ in range(5):
            graph.replay()
        torch.cuda.synchronize()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(n):
            graph.replay()
        t1.record()
        torch.cuda.synchronize()
        return t0.elapsed_time(t1) / n

    res = {"workload": f"OpticsZernike 896/256/T=350, height tolerance 2e-8, batch {B}, fwd+bwd into the trainable coefficient",
           "gpu": gpu_info(dev), "steps": args.steps}
    # device step: images resident on the GPU
    dev_f32, dev_u8 = host_f32.to(dev), host_u8.to(dev)
    for name, img, sigma, bits in (("step_f32", dev_f32, 0.0, 0), ("step_u8", dev_u8, 0.0, 0),
                                   ("step_f32_noise_quant8", dev_f32, 0.01, 8), ("step_u8_noise_quant8", dev_u8, 0.01, 8)):
        cam.sensor_noise_sigma, cam.sensor_quant_bits = sigma, bits
        graph, _ = capture(img)
        ms = time_replays(graph, args.steps)
        res[name] = {"ms": ms, "images_per_s": B / (ms * 1e-3)}
        del graph
    cam.sensor_noise_sigma, cam.sensor_quant_bits = 0.0, 0

    # end to end from pinned host images
    copy_stream = torch.cuda.Stream(device=dev)
    out_host = torch.empty(2).pin_memory()
    e2e_steps = max(5, min(args.steps, 30))
    for name, host in (("e2e_f32", host_f32), ("e2e_u8", host_u8)):
        bufs = [torch.empty_like(host, device=dev) for _ in range(2)]
        ready = [torch.cuda.Event() for _ in range(2)]
        freed = [torch.cuda.Event() for _ in range(2)]
        caps = [capture(bufs[k]) for k in range(2)]
        torch.cuda.synchronize()
        for k in range(2):
            freed[k].record(cur)

        def upload(i):
            k = i % 2
            with torch.cuda.stream(copy_stream):
                copy_stream.wait_event(freed[k])
                bufs[k].copy_(host, non_blocking=True)
                ready[k].record(copy_stream)

        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for timed in (False, True):
            n = e2e_steps if timed else 3
            if timed:
                t0.record()
            upload(0)
            for i in range(n):
                if i + 1 < n:
                    upload(i + 1)
                k = i % 2
                cur.wait_event(ready[k])
                caps[k][0].replay()
                freed[k].record(cur)
                out_host.copy_(caps[k][1], non_blocking=True)
            if timed:
                t1.record()
            torch.cuda.synchronize()
        ms = t0.elapsed_time(t1) / e2e_steps
        res[name] = {"images_per_s": B / (ms * 1e-3), "ms_per_step": ms, "h2d_bytes_per_step": host.numel() * host.element_size(),
                     "h2d_GBps": host.numel() * host.element_size() / (ms * 1e-3) / 1e9, "steps": e2e_steps}
        del caps, bufs

    # per-kernel device time of the forward row pass, fp32 against uint8 loader (a profiled run of its own)
    from torch.profiler import ProfilerActivity, profile
    kernels = {}
    for img in (dev_f32, dev_u8):
        with torch.no_grad():
            for _ in range(3):
                cam(img)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            with torch.no_grad():
                for _ in range(20):
                    cam(img)
            torch.cuda.synchronize()
        for ev in prof.key_averages():
            if "k_lrows_r2c" in ev.key and ("ImgLoad>" in ev.key or "ImgLoadU8>" in ev.key):
                t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0.0)
                kernels["ImgLoadU8" if "ImgLoadU8" in ev.key else "ImgLoad"] = {"us_per_launch": t / max(ev.count, 1),
                                                                                "launches": ev.count}
    res["kernel_us"] = kernels
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
