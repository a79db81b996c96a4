"""uint8 images on the Face-DeId camera: the sensor kernels reading the bytes against torch conversion + the fp32 kernels.

Workload: config 2's camera (``Camera(N=256, zernike_terms=50)``) at batch 64 and 128, one training step = forward + the
regularisers + backward into Zer_train, from a device-resident uint8 batch.  Two arms:
  u8         : cam(u8)                                   - the kernels read the bytes (x * fp32(1/255) in registers)
  convert    : cam(u8.to(torch.float32).div_(255.0))     - what the camera did before: a torch kernel + the fp32 kernels
Per arm:
  * step_ms   : the step replayed from a CUDA graph, CUDA events over --steps replays after warm-up; the arms alternate --reps
                times (every sample is reported, and the median)
  * e2e       : images/s of bench.py's e2e_u8 loop - pinned host uint8 batches copied on a second stream into two device
                buffers, the graph-captured step replayed on each - over --e2e-steps steps, the arms alternating --reps times
  * peak_mb   : torch.cuda.max_memory_allocated over one eager step, minus what was allocated before it
  * kernels   : mean device time per launch of the persistent row kernel (both instantiations) and of torch's element-wise
                kernels (the conversion), from torch.profiler over eager steps in a run of its own (after the timed legs)
The outputs of the two arms are compared bit for bit (eager steps, after the timed legs).  The card's name, power limit and max SM clock are read in the same
run.  Prints one JSON line; --out FILE also writes it.

  python tools/u8_input_bench.py [--steps 200] [--reps 5] [--e2e-steps 200] [--out FILE]
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
from b200cam.optics import Camera               # noqa: E402

ARMS = ("u8", "convert")


def gpu_info(dev) -> dict:
    info = {"name": torch.cuda.get_device_name(dev)}
    try:
        q = subprocess.run(["nvidia-smi", f"--id={dev.index}", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        info["nvidia_smi"] = q.stdout.strip()
    except (OSError, subprocess.SubprocessError) as exc:
        info["nvidia_smi"] = f"unavailable ({exc})"
    return info


def make_workload(B: int, dev):
    N = 256
    torch.manual_seed(0)
    cam = Camera(device=dev, N=N, zernike_terms=50)
    w = synth.upstream_grad(B, N, seed=B + 1).to(dev)
    one = torch.ones((), device=dev)

    def step(arm, img):
        cam.Zer_train.grad = None
        x = img if arm == "u8" else img.to(torch.float32).div_(255.0)
        y = cam(x)
        torch.autograd.backward([y, cam.loss_rad, cam.centering_loss], [w, one, one])
        return y, cam.Zer_train.grad
    return cam, step


def capture(step, arm, img, dev, side):
    cur = torch.cuda.current_stream(dev)
    side.wait_stream(cur)
    with torch.cuda.stream(side):
        for _ in range(3):
            step(arm, img)
    cur.wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        outs = step(arm, img)
    return graph, outs


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


def e2e(caps, bufs, host, n):
    """bench.py's e2e loop: copy of batch i on `copy` overlapping the replay of batch i-1 -> images/s"""
    cur = torch.cuda.current_stream()
    copy = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]

    def loop(m):
        for i in range(m + 1):
            if i < m:
                s = i % 2
                with torch.cuda.stream(copy):
                    copy.wait_event(freed[s])
                    bufs[s].copy_(host[i % len(host)], non_blocking=True)
                    ready[s].record(copy)
            if i >= 1:
                s = (i - 1) % 2
                cur.wait_event(ready[s])
                caps[s].replay()
                freed[s].record(cur)

    torch.cuda.synchronize()
    for s in range(2):
        freed[s].record(cur)
    loop(3)
    torch.cuda.synchronize()
    t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0.record()
    loop(n)
    t1.record()
    torch.cuda.synchronize()
    return bufs[0].shape[0] * n / (t0.elapsed_time(t1) * 1e-3)


def kernel_group(key: str):
    if "k_rows_r2c_persist" in key:
        return "rows_persist"
    if "copy_kernel" in key or "elementwise_kernel" in key:
        return "elementwise"
    return None


def profile_kernels(step, arm, img, steps=10):
    from torch.profiler import ProfilerActivity, profile
    for _ in range(3):
        step(arm, img)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            step(arm, img)
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


def peak_memory(step, arm, img, dev):
    step(arm, img)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    base = torch.cuda.memory_allocated(dev)
    torch.cuda.reset_peak_memory_stats(dev)
    step(arm, img)
    torch.cuda.synchronize()
    return (torch.cuda.max_memory_allocated(dev) - base) / 2 ** 20


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--e2e-steps", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    res = {"gpu": gpu_info(dev), "steps": args.steps, "reps": args.reps, "e2e_steps": args.e2e_steps, "workloads": {}}
    N, R = 256, 4
    for B in (64, 128):
        cam, step = make_workload(B, dev)
        host = [(synth.images(B, N, seed=1000 + r) * 255.0).round().to(torch.uint8).pin_memory() for r in range(R)]
        # every graph is captured before the first eager step (make_graphed_callables' rule: gradient-accumulation nodes made on
        # the default stream cannot join a capture); graph s of an arm reads device buffer s (the e2e loop's double buffer)
        bufs = [host[s].to(dev) for s in range(2)]
        side = torch.cuda.Stream(device=dev)
        caps = {arm: [capture(step, arm, bufs[s], dev, side)[0] for s in range(2)] for arm in ARMS}
        samples = {arm: [] for arm in ARMS}
        for _ in range(args.reps):                       # the arms alternate
            for arm in ARMS:
                samples[arm].append(time_replays(caps[arm][0], args.steps))
        e2e_samples = {arm: [] for arm in ARMS}
        for _ in range(args.reps):
            for arm in ARMS:
                e2e_samples[arm].append(e2e(caps[arm], bufs, host, args.e2e_steps))
        del caps
        torch.cuda.synchronize()
        img = host[0].to(dev)
        # the two arms compute the same thing: checked on the timed workload itself (eager steps)
        ya, ga = (t.detach().clone() for t in step("u8", img))
        yb, gb = (t.detach().clone() for t in step("convert", img))
        same = torch.equal(ya, yb) and torch.equal(ga, gb)
        entry = {"workload": f"Camera N={N} T=50, batch {B}, device-resident uint8 images, fwd + regularisers + bwd into Zer_train",
                 "outputs_bit_identical": same}
        for arm in ARMS:
            entry[arm] = {"step_ms_median": statistics.median(samples[arm]), "step_ms_samples": samples[arm],
                          "e2e_images_per_s_median": statistics.median(e2e_samples[arm]), "e2e_images_per_s_samples": e2e_samples[arm],
                          "peak_mb": peak_memory(step, arm, img, dev)}
        for arm in ARMS:
            entry[arm]["kernels"] = profile_kernels(step, arm, img)
        entry["u8_minus_convert_ms"] = entry["u8"]["step_ms_median"] - entry["convert"]["step_ms_median"]
        res["workloads"][f"face_deid_B{B}"] = entry
        print(json.dumps({f"face_deid_B{B}": {arm: [entry[arm]["step_ms_median"], entry[arm]["e2e_images_per_s_median"],
                                                     entry[arm]["peak_mb"]] for arm in ARMS}, "same": same}), flush=True)
        del cam, step
        torch.cuda.empty_cache()
    line = json.dumps(res)
    print(line, flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
