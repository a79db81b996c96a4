#!/usr/bin/env python
"""bench.py - encoded images/s, forward+backward, of the optical-encoder camera on B200.

Workload (BASELINE.json configs[1]): Face-DeId Camera forward + backward into the height map,
batch 64 of synthetic 256x256 RGB images per GPU, loss = sum(sensor*w) + loss_rad + centering_loss.
A "step" is one such forward+backward over one batch.  Prints ONE JSON line (rank 0).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--size N] [--impl reference] [--dump-outputs DIR]

* value      : images/s over all ranks, inputs resident in HBM, CUDA-graph replay of the step,
               CUDA events, barrier + synchronize on both sides, max over ranks.
* e2e        : the same step through the public nn.Module API with HOST (pinned) image buffers:
               H2D copy of every batch and D2H read of loss + dL/dh inside the timed region.
* roofline   : algorithmic bytes (48*N^2 per image, SURVEY 8d) / measured step time vs the measured
               HBM copy bandwidth in MEASURED_PEAKS.json; `breakdown_us` times the four C-ABI calls.
* cpu_baseline: the oracle port (oracle/camera_oracle.py, torch CPU, all host threads) on a bounded
               sample of the same workload - reported, not the target.
* --impl reference : times only that CPU implementation (the reference itself is PyTorch code that is
               not present on the GPU box; the oracle is its bit-exact restatement).
* --dump-outputs DIR : after the timed steps, writes what the last timed step returned to its caller (sensor
               images, PSF, regularisers, gradient) as DIR/<name>.npy, so that two builds can be compared output
               for output on the same seeded inputs.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time
from pathlib import Path

REPO = Path(__file__).resolve().parent
sys.path.insert(0, str(REPO))

import torch  # noqa: E402

METRIC = "encoded images/s fwd+bwd @1/2/4/8 B200; achieved HBM GB/s vs roofline"   # BASELINE.json: metric
UNIT = "images/s"
FALLBACK_HBM_GBS = 6650.0   # /opt/skills/guides/B200_PROFILING.md fallback


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default 2000; --impl reference: 20)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--batch", type=int, default=64, help="images per GPU")
    ap.add_argument("--size", type=int, default=256, help="image side N")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--input-sets", type=int, default=4, help="distinct resident input batches rotated through")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="budget of the cpu_baseline leg")
    ap.add_argument("--quick", action="store_true", help="timed loop only (for ncu): no breakdown / e2e / cpu legs")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32, at most 64 MB in all)")
    ap.add_argument("--config", default="2", choices=["1", "2", "3cam", "4cam", "5"],
                    help="BASELINE.json config: 1 = forward only, batch 8 (CPU-reference shape); 2 = fwd+bwd batch 64 (headline, "
                         "default); 3cam = the Image_Caption camera of config 3 (896/256/T=350, batch 128) without the caption "
                         "nets; 4cam = the camera half of config 4 (global batch 512 split over the ranks: STRONG scaling, all-reduce of dL/dh; the "
                         "FAN heat-map regressor is the reference's own model and is not on the GPU box: \"downstream\": \"absent\"); "
                         "5 = hi-res sweep (use --size 512|1024; the batch defaults to what fits the bench comfortably)")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.impl == "reference" else 2000      # a CPU step of the oracle port takes ~70 ms
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA implementation, not to --impl reference")
    if args.config == "1":
        args.batch = 8 if args.batch == 64 else args.batch
    if args.config == "5":
        if args.size == 256:
            args.size = 512
        if args.batch == 64:
            args.batch = 32 if args.size == 512 else 8
    if args.config == "3cam" and args.batch == 64:
        args.batch = 128
    if args.config == "4cam":                       # BASELINE config 4: global batch 512 over the ranks
        world = int(os.environ.get("WORLD_SIZE", str(max(1, args.gpus))))
        args.batch = max(1, 512 // max(1, world))
    return args


DUMP_BYTES = 64_000_000         # --dump-outputs: bytes written in all, at most


def dump_outputs(out_dir: str, outs: dict) -> None:
    """Write each output as <out_dir>/<name>.npy (float32).  When together they exceed DUMP_BYTES, the largest is cut to
    a fixed seeded sample of its leading (batch) dimension and the kept indices go to <name>_index.npy (float64): runs
    with the same arguments write the same sample."""
    import numpy as np
    arrays = {k: v.detach().float().cpu().numpy() for k, v in outs.items()}
    budget = DUMP_BYTES - 1024 * (len(arrays) + 1)             # room for the .npy headers
    total = sum(a.nbytes for a in arrays.values())
    if total > budget:
        big = max(arrays, key=lambda k: arrays[k].nbytes)
        a = arrays[big]
        keep_n = (budget - (total - a.nbytes)) // (a[0].nbytes + 8)
        if keep_n < 1:
            raise RuntimeError(f"--dump-outputs: one row of {big} {tuple(a.shape)} does not fit in {DUMP_BYTES} bytes")
        keep = np.sort(np.random.default_rng(0).choice(a.shape[0], size=keep_n, replace=False))
        arrays[big] = np.ascontiguousarray(a[keep])
        arrays[big + "_index"] = keep.astype(np.float64)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in arrays.items():
        np.save(out / f"{name}.npy", a)


# --------------------------------------------------------------------------------------------
# CPU arm: oracle port on the host cores
# --------------------------------------------------------------------------------------------
def cpu_port_rate(N: int, B: int, budget_s: float, steps: int | None = None, warmup: int = 1, forward_only: bool = False,
                  device: str = "cpu"):
    """images/s of the oracle (fwd+bwd into h, or forward only) with all host threads; bounded by budget_s.
    device="cuda": the same restatement on stock torch / cuFFT kernels of the GPU (the on-GPU comparison bar, SURVEY 2b)."""
    from oracle import camera_oracle as co
    import b200cam.synthetic as synth
    torch.set_num_threads(os.cpu_count() or 1)
    C = co.build_constants(N)
    img, w = synth.images(B, N), synth.upstream_grad(B, N)
    h = synth.height_map(N)
    if device != "cpu":
        import dataclasses
        C = dataclasses.replace(C, **{f.name: getattr(C, f.name).to(device) for f in dataclasses.fields(C)
                                      if torch.is_tensor(getattr(C, f.name))})
        img, w, h = img.to(device), w.to(device), h.to(device)
    h.requires_grad_(not forward_only)
    sync = torch.cuda.synchronize if device != "cpu" else (lambda: None)

    def step():
        if forward_only:
            with torch.no_grad():
                co.camera_forward(img, h, C)
            return
        h.grad = None
        out = co.camera_forward(img, h, C)
        ((out["sensor"] * w).sum() + out["loss_rad"] + out["centering_loss"]).backward()

    for _ in range(max(1, warmup)):
        step()
    sync()
    times = []
    t_end = time.perf_counter() + budget_s
    while (steps is None and time.perf_counter() < t_end and len(times) < 50) or (steps is not None and len(times) < steps):
        t0 = time.perf_counter()
        step()
        sync()
        times.append(time.perf_counter() - t0)
    times.sort()
    med = times[len(times) // 2]
    return B / med, med, len(times), torch.get_num_threads()


def workload_config(args, world: int, launch: str) -> dict:
    N, B, R = args.size, args.batch, max(1, args.input_sets)
    what = "forward only" if args.config == "1" else "fwd+bwd into height map"
    extra = {}
    if args.config == "4cam":
        what += " (camera half of the optical encoder + heat-map regressor step, global batch 512)"
        extra = {"downstream": "absent"}     # FAN (Face-DeId/core/wing.py) is the reference's own cuDNN model; not on the GPU box
    return {"workload": f"Face-DeId Camera {what}, batch {B}/GPU of {N}x{N} RGB, random height map",
            "baseline_config": args.config, **extra,
            "global_batch": B * world, "size": N, "parallelism": f"dp{world}" if world > 1 else "single",
            "l2": (f"{R} distinct resident input sets rotated: {R * 2 * B * 3 * N * N * 4 / 1e6:.0f} MB of inputs "
                   + ("(larger than the 126 MB L2)" if R * 2 * B * 3 * N * N * 4 > 126e6 else "(SMALLER than L2 - not a valid bench size)")),
            "launch": launch}


def module_step_with_zernike(dev, N: int, B: int, imgs, ws, T: int = 300, steps: int = 200) -> dict:
    """Forward + backward of the module with its own height map (Zernike projection of T coefficients and its adjoint
    included), CUDA-graph replay, device-timed.  Informational: BASELINE config 2 injects a random height map."""
    from b200cam.optics import Camera
    torch.manual_seed(0)
    cam = Camera(device=dev, N=N, zernike_terms=T)
    one = torch.ones((), device=dev)
    R = len(imgs)

    def step(i):
        cam.Zer_train.grad = None
        y = cam(imgs[i % R])
        torch.autograd.backward([y, cam.loss_rad, cam.centering_loss], [ws[i % R], one, one])

    def drop():
        cam.psfs = None
        cam.loss_rad = cam.centering_loss = cam._pending_centering = None
        cam.Zer_train.grad = None

    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream(dev))
    with torch.cuda.stream(side):
        for i in range(3):
            step(i)
    torch.cuda.current_stream(dev).wait_stream(side)
    torch.cuda.synchronize()
    graphs = []
    for r in range(R):
        drop()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            step(r)
        graphs.append(g)
    for i in range(20):
        graphs[i % R].replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        graphs[i % R].replay()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    return {"value": B / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms, "steps": steps, "zernike_terms": T,
            "note": "Camera with its own T-term Zernike height map (projection + adjoint over the basis volume every step), "
                    "gradient into Zer_train; extra information beside the contract's injected-height-map step"}


def run_reference(args) -> None:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    N, B = args.size, args.batch
    steps = args.steps
    warm = max(1, min(args.warmup, 10))            # the warm-up the caller asked for (a CPU step is ~70 ms: cheap)
    rate, med, n, cores = cpu_port_rate(N, B, budget_s=120.0, steps=steps, warmup=warm, forward_only=args.config == "1")
    line = {
        "impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": n,
        "warmup": warm, "ms_per_step": med * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, max(1, args.gpus), f"torch {torch.__version__} CPU, {cores} threads, rank 0 only"),
        "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{n} steps of batch {B} at N={N}, median (reference PyTorch module is not on the GPU box; "
                                   "oracle/camera_oracle.py is its bit-exact torch restatement)"},
        "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------------
# clocks sampler
# --------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines: list[str] = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "power_w_max": max(pw), "samples": len(sm),
                "reasons": sorted(reasons)}


# --------------------------------------------------------------------------------------------
# GPU arm
# --------------------------------------------------------------------------------------------
def hbm_peak():
    p = REPO / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def run_b200(args) -> None:
    import torch.distributed as dist
    import b200cam.synthetic as synth
    from b200cam import _lib
    from b200cam.optics import Camera

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a CUDA device; there is no CPU fallback for the b200 arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)
    N, B, R = args.size, args.batch, max(1, args.input_sets)
    lib = _lib.load_library()

    # the camera's PSF chain runs on a side stream by design; autograd's advisory about it is not an error
    try:
        torch.autograd.graph.set_warn_on_accumulate_grad_stream_mismatch(False)
    except AttributeError:
        pass
    torch.manual_seed(0)
    cam = Camera(device=dev, N=N, zernike_terms=12)
    h = synth.height_map(N).to(dev).requires_grad_(True)     # "random height map" (configs[0..1])
    cam.get_Heith_Map = lambda: h
    if world > 1:
        cam.data_parallel(average=True)
    imgs_host = [synth.images(B, N, seed=1000 + 17 * rank + r).pin_memory() for r in range(R)]
    imgs = [t.to(dev) for t in imgs_host]
    ws = [synth.upstream_grad(B, N, seed=2000 + 17 * rank + r).to(dev) for r in range(R)]

    one = torch.ones((), device=dev)
    fwd_only = args.config == "1"

    def step(i: int) -> dict:
        """forward + backward into h; upstream gradients: w for the sensor image, 1 for the two regularisers
        (i.e. L = sum(sensor*w) + loss_rad + centering_loss without materialising the product).
        Config 1: the forward alone (no autograd graph).  Returns what the caller receives (detached)."""
        if fwd_only:
            with torch.no_grad():
                y = cam(imgs[i % R])
        else:
            h.grad = None
            y = cam(imgs[i % R])
            torch.autograd.backward([y, cam.loss_rad, cam.centering_loss], [ws[i % R], one, one])
        outs = {"sensor": y.detach(), "psf": cam.psfs.detach(), "loss_rad": cam.loss_rad.detach(),
                "centering_loss": cam.centering_loss.detach()}
        if not fwd_only:
            outs["grad_h"] = h.grad
        return outs

    def drop_graph_refs():
        # the module keeps psfs / loss tensors (like the reference); they pin the previous autograd graph and
        # its AccumulateGrad stream, which breaks stream capture - release them before capturing
        cam.psfs = None
        cam.loss_rad = cam.centering_loss = cam._pending_centering = None
        h.grad = None

    # eager warm-up (also builds the per-device plan outside any capture) + count our kernel launches per step
    step(0)
    torch.cuda.synchronize()
    c0 = lib.b200cam_launch_count()
    step(1)
    torch.cuda.synchronize()
    launches_per_step = int(lib.b200cam_launch_count() - c0)

    graphs = None
    drop_graph_refs()
    if not args.no_graph:
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for r in range(R):
                    step(r)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graphs, graph_outs = [], []          # graph_outs[r]: the static output tensors that replays of graphs[r] rewrite
            for r in range(R):
                g = torch.cuda.CUDAGraph()
                drop_graph_refs()
                with torch.cuda.graph(g):
                    graph_outs.append(step(r))
                graphs.append(g)
        except Exception as exc:   # e.g. NCCL capture unsupported: fall back to eager launches of the same kernels
            if rank == 0:
                print(f"[bench] CUDA graph capture failed ({exc}); timing eager launches", file=sys.stderr)
            graphs = None
            torch.cuda.synchronize()

    def run_step(i: int) -> dict:
        if graphs is not None:
            graphs[i % R].replay()
            return graph_outs[i % R]
        return step(i)

    # rough step time (same code path on every rank) to size the load phase before the timed region
    torch.cuda.synchronize()
    t_est = time.perf_counter()
    for i in range(10):
        run_step(i)
    torch.cuda.synchronize()
    est_ms = (time.perf_counter() - t_est) * 100.0
    if world > 1:
        t = torch.tensor([est_ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        est_ms = float(t.item())

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # nvidia-smi needs ~1 s before its first sample: keep every rank under load for a FIXED number of steps
    # (identical on all ranks - the steps contain a collective)
    spin_steps = int(min(5000, max(100, 1.0 / max(est_ms * 1e-3, 1e-5))))
    for i in range(spin_steps):
        run_step(i)
    torch.cuda.synchronize()
    for i in range(max(3, args.warmup)):
        run_step(i)
    sync_all()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        last = run_step(i)
    e1.record()
    sync_all()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    total_ms = float(ms.item())
    clocks = sampler.stop() if rank == 0 else None
    ms_per_step = total_ms / args.steps
    value = world * B * args.steps / (total_ms * 1e-3)
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, last)          # before the passes below replay the graphs again

    if args.quick:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
                              "ms_per_step": ms_per_step, "quick": True, "launches_per_step": launches_per_step,
                              "clocks": clocks}), flush=True)
        graphs = None
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
            sys.stdout.flush()
            os._exit(0)
        return

    # ---- per-kernel durations of the replayed step (CUPTI activity records through torch.profiler; a separate pass
    #      AFTER the timed region - nothing above was measured under it).  Bytes = what that kernel must read + write.
    kernel_table = None
    if graphs is not None:
        try:
            from torch.profiler import ProfilerActivity, profile
            reps = 8                                    # every rank replays them (the step holds a collective)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                for i in range(reps):
                    run_step(i)
                torch.cuda.synchronize()
            P = B * 3 * N * N * 4                       # one batch of real planes
            S = B * 3 * (N // 2 + 1) * N * 8            # one batch of half spectra
            model = {"k_rows_r2c_persist": P + S, "k_cols_conv": 2 * S, "k_rows_c2r_persist": S + P, "k_normalise": 2 * P,
                     "k_cols_accum": 2 * S}
            agg = {}
            for e in prof.events():
                if e.device_type == torch.autograd.DeviceType.CUDA and e.time_range is not None and "k_" in e.name:
                    name = e.name.replace("void ", "").replace("b200cam::", "").split("(")[0]
                    a = agg.setdefault(name, [0, 0.0])
                    a[0] += 1
                    a[1] += e.time_range.end - e.time_range.start
            kernel_table = []
            for name, (cnt, tot) in sorted(agg.items(), key=lambda kv: -kv[1][1]):
                us = tot / cnt
                row = {"kernel": name, "launches_per_step": round(cnt / reps, 2), "avg_us": round(us, 2)}
                key = name.split("<")[0]
                if key in model and cnt / reps < 2.5:
                    nbytes = model[key]
                    row["bytes"] = nbytes
                    row["GBps"] = round(nbytes / us * 1e-3, 1)
                kernel_table.append(row)
        except Exception as exc:    # CUPTI not available: the table is optional
            kernel_table = [{"error": str(exc)[:200]}]

    # ---- per-call breakdown (each C-ABI call timed alone over the same rotating inputs) -----------------
    from b200cam import functional as F
    plan = cam._plan(dev)
    breakdown = {}

    def time_call(name, fn, reps=20):
        for i in range(3):
            fn(i)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for i in range(reps):
            fn(i)
        b.record()
        torch.cuda.synchronize()
        breakdown[name] = a.elapsed_time(b) / reps * 1e3

    with torch.no_grad():
        hd = h.detach()
        time_call("psf_fwd", lambda i: F.PsfSynth.apply(hd, plan))
        psf = F.PsfSynth.apply(hd, plan)[0]
        time_call("sensor_fwd", lambda i: F.SensorConv.apply(imgs[i % R], psf, plan))
    if not fwd_only:
        p_req = psf.clone().requires_grad_(True)
        ys = [F.sensor_conv(imgs[r], p_req, plan) for r in range(R)]
        time_call("sensor_bwd", lambda i: torch.autograd.grad(ys[i % R], p_req, ws[i % R], retain_graph=True))
        hr = h.detach().clone().requires_grad_(True)
        pp, _l1, _l2 = F.psf_synth(hr, plan)
        gp = torch.rand_like(pp)
        time_call("psf_bwd", lambda i: torch.autograd.grad(pp, hr, gp, retain_graph=True))
        del ys, p_req, pp

    # ---- data parallel: is the fused peer-memory all-reduce right?  (outside every timed region)  dL/dh of one step through
    #      b200cam_psf_bwd_allreduce (the path timed above) against the same step with dist.all_reduce, and bitwise equality
    #      of the result across ranks.
    allreduce_check = None
    if world > 1 and not fwd_only:
        def grad_once(camera):
            h.grad = None
            y = camera(imgs[0])
            torch.autograd.backward([y, camera.loss_rad, camera.centering_loss], [ws[0], one, one])
            torch.cuda.synchronize()
            return h.grad.detach().clone()
        g_peer = grad_once(cam)
        fused_path = cam._plan(dev).peer_comm is not None
        cam_ref = Camera(device=dev, N=N, zernike_terms=12)
        cam_ref.get_Heith_Map = lambda: h
        cam_ref.data_parallel(average=True, peer_memory=False)
        g_nccl = grad_once(cam_ref)
        gathered = [torch.empty_like(g_peer) for _ in range(world)]
        dist.all_gather(gathered, g_peer)
        allreduce_check = {"rel": float((g_peer - g_nccl).norm() / g_nccl.norm()),
                           "ranks_bitwise_equal": bool(all(torch.equal(t, gathered[0]) for t in gathered)),
                           "fused_peer_path": bool(fused_path), "finite": bool(torch.isfinite(g_peer).all())}
        cam.check_device_errors()

    # ---- end to end through the module API with host image buffers ------------------------------------
    # Every step: H2D copy of that step's pinned host images (copy stream, two device buffers), the module's forward +
    # backward on them, D2H of the step's results (loss + dL/dh; config 1: the sensor images).  The module call is made
    # the way a training loop that cares about speed makes it - captured once per device buffer in a CUDA graph
    # (torch.cuda.graph around `cam(img)` + backward; static input = the device buffer the copy lands in) and replayed;
    # the same loop with eager module calls is reported beside it as `e2e_eager` (an eager step costs ~0.4 ms of Python,
    # ctypes and autograd for ~0.17 ms of device work: that bounds the uint8 loop, the fp32 one is PCIe-bound either way).
    copy_stream = torch.cuda.Stream()
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    gh_host = torch.empty(1, N, N).pin_memory()
    loss_host = torch.empty(1).pin_memory()
    y_host = torch.empty(B, 3, N, N).pin_memory() if fwd_only else None
    e2e_steps = max(10, min(args.steps, 50))

    def e2e_compute(buf, j):
        if fwd_only:                                      # config 1: the sensor images themselves are the result
            with torch.no_grad():
                return (cam(buf),)
        h.grad = None
        y = cam(buf)
        torch.autograd.backward([y, cam.loss_rad, cam.centering_loss], [ws[j % R], one, one])
        return (h.grad, (cam.loss_rad + cam.centering_loss).detach().reshape(1))

    def measure_e2e(host_list, bufs, graphed):
        """images/s of the whole job; (value, "cuda-graph replay" | "eager")"""
        cur = torch.cuda.current_stream()
        caps = None
        if graphed:
            try:
                caps = []
                for s in range(2):
                    drop_graph_refs()
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        outs = e2e_compute(bufs[s], s)
                    caps.append((g, outs))
            except Exception as exc:
                if rank == 0:
                    print(f"[bench] e2e graph capture failed ({exc}); eager module calls", file=sys.stderr)
                caps = None
                torch.cuda.synchronize()

        def loop(n):
            for i in range(n + 1):
                if i < n:                                 # prefetch batch i
                    s = i % 2
                    with torch.cuda.stream(copy_stream):
                        copy_stream.wait_event(freed[s])
                        bufs[s].copy_(host_list[i % R], non_blocking=True)
                        ready[s].record(copy_stream)
                if i >= 1:                                # compute batch i-1
                    s = (i - 1) % 2
                    cur.wait_event(ready[s])
                    if caps is not None:
                        caps[s][0].replay()
                        outs = caps[s][1]
                    else:
                        outs = e2e_compute(bufs[s], i - 1)
                    freed[s].record(cur)
                    if fwd_only:
                        y_host.copy_(outs[0], non_blocking=True)
                    else:
                        gh_host.copy_(outs[0], non_blocking=True)
                        loss_host.copy_(outs[1], non_blocking=True)

        sync_all()
        for s in range(2):
            freed[s].record(cur)
        loop(3)
        sync_all()
        t0, t1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0.record()
        loop(e2e_steps)
        t1.record()
        sync_all()
        ems = torch.tensor([t0.elapsed_time(t1)], device=dev)
        if world > 1:
            dist.all_reduce(ems, op=dist.ReduceOp.MAX)
        drop_graph_refs()
        return world * B * e2e_steps / (float(ems.item()) * 1e-3), ("cuda-graph replay" if caps is not None else "eager")

    dev_bufs = [torch.empty_like(imgs[0]) for _ in range(2)]
    # the same loop with uint8 host images (what an image decoder yields; the reference's loader converts to fp32 on the
    # host before the copy).  Reported beside `e2e`, not instead of it.
    imgs_u8_host = [(t * 255.0).round().to(torch.uint8).pin_memory() for t in imgs_host]
    dev_u8 = [torch.empty(B, 3, N, N, dtype=torch.uint8, device=dev) for _ in range(2)]
    want_graph = graphs is not None
    e2e_value, e2e_launch = measure_e2e(imgs_host, dev_bufs, want_graph)
    e2e_u8_value, e2e_u8_launch = measure_e2e(imgs_u8_host, dev_u8, want_graph)
    e2e_eager_value, _ = measure_e2e(imgs_host, dev_bufs, False)
    e2e_u8_eager_value, _ = measure_e2e(imgs_u8_host, dev_u8, False)

    def finish():
        # captured graphs hold NCCL work: drop them and drain the device before tearing the communicator down
        nonlocal graphs
        graphs = None
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()
            sys.stdout.flush()
            sys.stderr.flush()
            os._exit(0)      # skip destroy_process_group(): it can block on graph-captured collectives

    if rank != 0:
        finish()
        return

    peak, peak_src = hbm_peak()
    bytes_per_image = (24 if fwd_only else 48) * N * N
    achieved = B * bytes_per_image / (ms_per_step * 1e-3) / 1e9          # per GPU
    # DRAM traffic of one step: NOT measured by this run (it needs ncu) - the committed ncu capture of the same command
    # is quoted as `traffic_static` with its source; `traffic` stays null unless a live counter is available
    traffic_static = None
    tpath = REPO / "profiles" / "traffic.json"
    if tpath.exists() and not fwd_only:
        try:
            tj = json.loads(tpath.read_text())
            if f"N{N}_B{B}" in tj:
                traffic_static = {"bytes_per_step": tj[f"N{N}_B{B}"], "source": tj.get("source", "profiles/traffic.json")}
        except Exception:
            traffic_static = None
    cpu = None
    torch_cuda = None
    if world == 1:
        what = "forward" if fwd_only else "fwd+bwd"
        rate, med, n, cores = cpu_port_rate(N, B, args.cpu_seconds, forward_only=fwd_only)
        cpu = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
               "sample": f"{n} {what} steps of batch {B} at N={N} (median), oracle/camera_oracle.py on torch CPU"}
        # the on-GPU bar (SURVEY 2b): the same restatement of the reference module on stock torch + cuFFT, this GPU
        try:
            trate, tmed, tn, _ = cpu_port_rate(N, B, 3.0, warmup=3, forward_only=fwd_only, device=str(dev))
            torch_cuda = {"value": trate, "unit": UNIT, "ms_per_step": tmed * 1e3, "steps": tn,
                          "kind": "oracle restatement of the reference Camera on stock torch/cuFFT kernels, eager, same GPU",
                          "speedup_of_this_repo": value / trate}
        except Exception as exc:
            torch_cuda = {"error": str(exc)[:200]}
    # Extra information (not the contract's number): the module as a training loop drives it - height map from the T = 300
    # Zernike coefficients (solver.py:30) instead of an injected one, gradient into Zer_train.  Adds the projection
    # h = sum coef_j Z_j and its adjoint (2 x 79 MB over the basis volume at N = 256) to every step.
    module_step = None
    if world == 1 and args.config == "2" and not fwd_only:
        try:
            module_step = module_step_with_zernike(dev, N, B, imgs, ws)
        except Exception as exc:
            module_step = {"error": str(exc)[:200]}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(3, args.warmup),
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong" if args.config == "4cam" else "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, world, "cuda-graph replay" if graphs is not None else "eager"),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": B * 3 * N * N * 4,
                "d2h_bytes_per_step": B * 3 * N * N * 4 if fwd_only else N * N * 4 + 4,
                "steps": e2e_steps, "launch": e2e_launch,
                "h2d_GBps": e2e_value / world / B * (B * 3 * N * N * 4) / 1e9,      # per GPU; ~55 GB/s = the PCIe ceiling of the box
                "note": "nn.Module API (cam(img) + backward), pinned host images, double-buffered H2D on a copy stream, "
                        "loss + dL/dh read back every step"},
        "e2e_eager": {"value": e2e_eager_value, "unit": UNIT, "note": "the same loop with eager module calls (fp32 images: PCIe-bound either way; uint8: see e2e_u8.eager_value)"},
        "e2e_u8": {"value": e2e_u8_value, "unit": UNIT, "h2d_bytes_per_step": B * 3 * N * N,
                   "d2h_bytes_per_step": B * 3 * N * N * 4 if fwd_only else N * N * 4 + 4,
                   "steps": e2e_steps, "launch": e2e_u8_launch, "eager_value": e2e_u8_eager_value,
                   "h2d_GBps": e2e_u8_value / world / B * (B * 3 * N * N) / 1e9,
                   "note": "same loop, uint8 host images (decoder output), /255 on the GPU: extra information, "
                           "the fp32 `e2e` above is the contract's number"},
        "gpu_launches": launches_per_step * args.steps,
        "launches_per_step": launches_per_step,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": None, "traffic_static": traffic_static, "peak_source": peak_src,
                     "scope": ("whole step: every kernel of the forward (algorithmic bytes 24*N^2 per image)" if fwd_only else
                               "whole step: every kernel of fwd+bwd (algorithmic bytes 48*N^2 per image, SURVEY 8d)"),
                     "breakdown_us": {k: round(v, 2) for k, v in breakdown.items()},
                     "kernels_cupti": kernel_table},
        "clocks": clocks,
    }
    if module_step is not None:
        line["module_step_with_zernike"] = module_step
    if cpu is not None:
        line["cpu_baseline"] = cpu
    if torch_cuda is not None:
        line["torch_cuda_baseline"] = torch_cuda
    if allreduce_check is not None:
        line["allreduce_check"] = allreduce_check
    print(json.dumps(line), flush=True)
    finish()


# --------------------------------------------------------------------------------------------
# config "3cam": the Image_Caption camera of BASELINE config 3 (OpticsZernike, shipped geometry of
# Image_Caption/train.py:64-66: wave 896, patch 256, T = 350, batch 128) - forward + backward into the trainable Zernike
# coefficient, WITHOUT the caption nets (ResNet-101 / LSTM are cuDNN / cuBLAS work outside the hot path, SURVEY 2 #19).
# --------------------------------------------------------------------------------------------
def run_caption_camera(args) -> None:
    from b200cam.lens import OpticsZernike
    from b200cam import _lib
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    dev = torch.device("cuda", int(os.environ.get("LOCAL_RANK", "0")))
    torch.cuda.set_device(dev)
    B, P = args.batch, 256
    lib = _lib.load_library()
    cam = OpticsZernike(input_shape=[None, P, P, 3], device=dev, zernike_terms=350, patch_size=P, height_tolerance=2e-8,
                        sensor_distance=0.025, wave_resolution=[896, 896], sample_interval=3e-06, upsample=False).to(dev)
    R = max(1, args.input_sets)
    g = torch.Generator().manual_seed(5)
    imgs_host = [torch.rand(B, 3, P, P, generator=g).pin_memory() for _ in range(R)]
    imgs = [t.to(dev) for t in imgs_host]
    ws = [torch.rand(B, 3, P, P, generator=g).to(dev) for _ in range(R)]

    def step(i) -> dict:
        cam.zero_grad(set_to_none=True)
        sensor, psf, coeffs, loss = cam(imgs[i % R])
        torch.autograd.backward([sensor], [ws[i % R]])
        return {"sensor": sensor.detach(), "psf": psf.detach(), "grad_defocus": cam.zernike_coeffs_train.grad}

    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    c0 = lib.b200cam_launch_count()
    step(0)
    torch.cuda.synchronize()
    launches = int(lib.b200cam_launch_count() - c0)
    # the timed loop replays the step from CUDA graphs (one per input set), as config 2 does; eager launches if capture fails
    graphs = None
    if not args.no_graph:
        try:
            side = torch.cuda.Stream(device=dev)
            side.wait_stream(torch.cuda.current_stream(dev))
            with torch.cuda.stream(side):
                for i in range(2):
                    step(i)
            torch.cuda.current_stream(dev).wait_stream(side)
            torch.cuda.synchronize()
            graphs, graph_outs = [], []
            for r in range(R):
                cam.zero_grad(set_to_none=True)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    graph_outs.append(step(r))
                graphs.append(g)
        except Exception as exc:
            print(f"[bench] CUDA graph capture of the caption camera failed ({exc}); timing eager launches", file=sys.stderr)
            graphs = None
            torch.cuda.synchronize()

    def run_step(i) -> dict:
        if graphs is not None:
            graphs[i % R].replay()
            return graph_outs[i % R]
        return step(i)

    sampler = ClockSampler(dev.index)
    sampler.start()
    t_spin = time.perf_counter()
    i = 0
    while time.perf_counter() - t_spin < 1.2:
        run_step(i); i += 1
    for i in range(max(3, args.warmup)):
        run_step(i)
    torch.cuda.synchronize()
    steps = args.steps
    # every step draws the lens tolerance noise from torch's generator (a graph replay reads its state when it runs), and
    # the spin above runs for a wall-clock time: seed here, so that the timed steps see the same noise on every run
    torch.manual_seed(0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        last = run_step(i)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / steps
    clocks = sampler.stop()
    if args.dump_outputs is not None:
        dump_outputs(args.dump_outputs, last)
    # end to end: pinned host images in, sensor checksum + coefficient gradient out; the host-to-device copy of step i+1 runs on
    # a copy stream beside the compute of step i (two device buffers), as the config-2 e2e leg does.  The module call
    # (cam(img) + backward) is captured once per device buffer in a CUDA graph and replayed; `e2e_eager` = eager calls.
    out_host = torch.empty(2).pin_memory()
    dbufs = [torch.empty_like(imgs[0]) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    ready = [torch.cuda.Event() for _ in range(2)]
    freed = [torch.cuda.Event() for _ in range(2)]
    cur = torch.cuda.current_stream(dev)
    e2e_steps = max(5, min(steps, 30))

    def e2e_compute(k, j):
        cam.zero_grad(set_to_none=True)
        sensor, psf, coeffs, loss = cam(dbufs[k])
        torch.autograd.backward([sensor], [ws[j % R]])
        return torch.stack([sensor.detach().sum(), cam.zernike_coeffs_train.grad.reshape(-1)[0]])

    def upload(i):
        k = i % 2
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(freed[k])                  # the step that last read this buffer is done
            dbufs[k].copy_(imgs_host[i % R], non_blocking=True)
            ready[k].record(copy_stream)

    def measure_e2e(graphed):
        caps = None
        if graphed:
            try:
                caps = []
                for k in range(2):
                    cam.zero_grad(set_to_none=True)
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g):
                        out = e2e_compute(k, k)
                    caps.append((g, out))
            except Exception as exc:
                print(f"[bench] e2e graph capture failed ({exc}); eager module calls", file=sys.stderr)
                caps = None
        torch.cuda.synchronize()
        for k in range(2):
            freed[k].record(cur)
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
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
                if caps is not None:
                    caps[k][0].replay()
                    out = caps[k][1]
                else:
                    out = e2e_compute(k, i)
                freed[k].record(cur)
                out_host.copy_(out, non_blocking=True)
            if timed:
                t1.record()
            torch.cuda.synchronize()
        cam.zero_grad(set_to_none=True)
        return B * e2e_steps / (t0.elapsed_time(t1) * 1e-3), ("cuda-graph replay" if caps is not None else "eager")

    e2e, e2e_launch = measure_e2e(graphs is not None)
    e2e_eager, _ = measure_e2e(False)
    peak, peak_src = hbm_peak()
    achieved = B * 48 * P * P / (ms * 1e-3) / 1e9
    # CPU baseline: the oracle restatement of the reference module, bounded sample (one step of batch 4 is ~1.5 s)
    from oracle import lens_oracle as lo
    import b200cam.zernike as zern
    import numpy as np
    torch.set_num_threads(os.cpu_count() or 1)
    cfg = lo.LensConfig()
    vol = cam.zernike_volume.detach().cpu() if hasattr(cam, "zernike_volume") else torch.tensor(
        zern.zernike_volume(896, 350, 1e-6).astype(np.float32))
    coeffs = torch.zeros(350, 1, 1); coeffs[3] = -22.0
    bs = 4
    img_c, w_c = imgs_host[0][:bs].clone(), ws[0][:bs].cpu()
    times = []
    for k in range(3):
        cz = coeffs.clone().requires_grad_(True)
        tt = time.perf_counter()
        out = lo.lens_forward(img_c, cz, vol, cfg)
        (out["sensor"] * w_c).sum().backward()
        times.append(time.perf_counter() - tt)
    cpu_rate = bs / sorted(times)[1]
    line = {"metric": METRIC, "value": B / (ms * 1e-3), "unit": UNIT, "n_gpus": 1, "steps": steps, "warmup": max(3, args.warmup),
            "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": f"Image_Caption camera (OpticsZernike 896/256/T=350) fwd+bwd into the trainable coefficient, batch {B} "
                                   "of 256x256 RGB; caption nets not included", "baseline_config": "3cam", "global_batch": B,
                       "l2": f"{R} input sets rotated: {R * 2 * B * 3 * P * P * 4 / 1e6:.0f} MB", "launch": "cuda-graph replay" if graphs is not None else "eager"},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": B * 3 * P * P * 4, "d2h_bytes_per_step": 8, "steps": e2e_steps,
                    "launch": e2e_launch, "h2d_GBps": e2e * 3 * P * P * 4 / 1e9},     # ~55 GB/s = the PCIe ceiling of the box
            "e2e_eager": {"value": e2e_eager, "unit": UNIT},
            "gpu_launches": launches * steps, "launches_per_step": launches,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": None,
                         "peak_source": peak_src,
                         "scope": "whole step: PSF synthesis (1344^2 mixed-radix kernels), pruned 512^2 sensor convolution, backward into the trainable coefficient; algorithmic bytes 48*P^2 per image - the path is FP32-compute bound, SURVEY 8a"},
            "clocks": clocks,
            "cpu_baseline": {"value": cpu_rate, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"3 fwd+bwd steps of batch {bs} (median), oracle/lens_oracle.py on torch CPU"}}
    print(json.dumps(line), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    elif args.config == "3cam":
        run_caption_camera(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
