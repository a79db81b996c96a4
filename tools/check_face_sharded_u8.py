"""Multi-GPU check (run under torchrun, one rank per GPU): the Face-DeId camera with its batch sharded over the ranks
(`Camera.data_parallel`: dL/dh all-reduced inside the PSF backward) fed uint8 shards must give, on every rank, the sensor image
and the all-reduced dL/dh of the same camera fed the shards converted on the GPU with ``u8.to(torch.float32).div_(255.0)`` -
bit for bit.
usage: python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/check_face_sharded_u8.py [--bf16]
--bf16: sensor_dtype = torch.bfloat16 (bf16 sensor images, bf16 upstream gradient).
"""
import sys
from pathlib import Path

import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import b200cam.synthetic as synth          # noqa: E402
from b200cam import parallel               # noqa: E402
from b200cam.optics import Camera          # noqa: E402


def main():
    out_dtype = torch.bfloat16 if "--bf16" in sys.argv[1:] else torch.float32
    rank, world, local = parallel.init_from_env("nccl")
    dev = torch.device("cuda", local)
    N, per = 128, 3
    B = per * world
    u8 = (synth.images(B, N, seed=21) * 255.0).round().clamp(0, 255).to(torch.uint8)
    u8[B - 1] = 255                               # a saturated image on the last rank's shard
    w = synth.upstream_grad(B, N, seed=22) * 1e-2
    h_cpu = synth.height_map(N, 23)
    sl = slice(rank * per, (rank + 1) * per)
    shard = u8[sl].to(dev)

    def step(img):
        torch.manual_seed(0)
        cam = Camera(device=dev, N=N, zernike_terms=8).data_parallel()
        cam.sensor_dtype = out_dtype
        h = h_cpu.to(dev).requires_grad_(True)
        cam.get_Heith_Map = lambda: h
        y = cam(img)
        ((y.float() * w[sl].to(dev)).sum() + cam.loss_rad + cam.centering_loss).backward()
        cam.check_device_errors()
        return y.detach(), h.grad.detach()

    y8, g8 = step(shard)
    y32, g32 = step(shard.to(torch.float32).div_(255.0))
    view = torch.int16 if out_dtype == torch.bfloat16 else torch.int32
    ok = (y8.dtype == out_dtype and torch.equal(y8.view(view), y32.view(view))
          and torch.equal(g8.view(torch.int32), g32.view(torch.int32)))
    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print(f"FACE_SHARDED_U8 world={world} dtype={str(out_dtype).split('.')[-1]} ok={bool(flag.item())}", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
