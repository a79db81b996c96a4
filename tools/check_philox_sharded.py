"""Multi-GPU check (run under torchrun, one rank per GPU): with ``sensor_noise_rng = "philox"`` and every rank seeded alike,
both cameras with their batch sharded over the ranks (``data_parallel``) must give, on every rank, the rows of the one-GPU
sensor image of the whole batch - bit for bit, noise included (the shard's Philox counter starts at rank * shard elements / 4).
usage: python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/check_philox_sharded.py
"""
import sys
from pathlib import Path

import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import b200cam.synthetic as synth          # noqa: E402
from b200cam import parallel               # noqa: E402
from b200cam.lens import OpticsZernike     # noqa: E402
from b200cam.optics import Camera          # noqa: E402


def main():
    rank, world, local = parallel.init_from_env("nccl")
    dev = torch.device("cuda", local)
    per, sigma, bits = 3, 0.02, 8
    B = per * world
    sl = slice(rank * per, (rank + 1) * per)
    ok = True

    # Face-DeId camera (per-image maximum)
    N = 128
    img = synth.images(B, N, seed=41).to(dev)
    torch.manual_seed(0)
    cam = Camera(device=dev, N=N, zernike_terms=8)
    cam.sensor_noise_sigma, cam.sensor_quant_bits, cam.sensor_noise_rng = sigma, bits, "philox"
    with torch.no_grad():
        torch.manual_seed(5)
        whole = cam(img)
        cam.data_parallel(peer_memory=False)
        torch.manual_seed(5)
        shard = cam(img[sl].contiguous())
    ok &= torch.equal(whole[sl].view(torch.int32), shard.view(torch.int32))
    ok &= int(cam.sensor_noise_seed[1]) == rank * per * 3 * N * N // 4

    # Image_Caption camera (batch-global maximum, all-reduced by data_parallel)
    wave, patch = 128, 64
    g = torch.Generator().manual_seed(42)
    x = torch.rand(B, 3, patch, patch, generator=g).to(dev)
    lens = OpticsZernike(input_shape=[1, patch, patch, 3], device=dev, wave_resolution=(wave, wave), patch_size=patch,
                         sample_interval=3e-6, zernike_terms=10, height_tolerance=20e-9).to(dev)
    lens.sensor_noise_sigma, lens.sensor_quant_bits, lens.sensor_noise_rng = sigma, bits, "philox"
    with torch.no_grad():
        torch.manual_seed(6)
        whole = lens(x)[0]
        lens.data_parallel()
        torch.manual_seed(6)
        shard = lens(x[sl].contiguous())[0]
    ok &= torch.equal(whole[sl].view(torch.int32), shard.view(torch.int32))

    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print(f"PHILOX_SHARDED world={world} ok={bool(flag.item())}", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
