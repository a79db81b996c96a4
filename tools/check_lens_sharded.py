"""Multi-GPU check (run under torchrun, one rank per GPU): the Image_Caption camera with its batch sharded over the ranks
(`OpticsZernike.data_parallel`: all-reduce MAX of the batch-global maximum, SUM of sum(g*y) and of the tie count) must
reproduce the single-GPU result on the whole batch - sensor images and the gradient of the trainable coefficient
(summed over ranks).  Lens.py:312 couples all images of a batch; T5 in SURVEY 8.
usage: python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 tools/check_lens_sharded.py [--bf16] [--u8]
--bf16: both cameras with sensor_dtype = torch.bfloat16 (bf16 sensor images, bf16 upstream gradient).
--u8: uint8 images; the sharded camera fed the uint8 shards must also equal, bit for bit, the sharded camera fed the shards
converted on the GPU (u8.to(torch.float32).div_(255.0)): sensor images and the all-reduced coefficient gradient.
"""
import sys
from pathlib import Path

import torch
import torch.distributed as dist

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from b200cam import parallel               # noqa: E402
from b200cam.lens import OpticsZernike     # noqa: E402


def main():
    out_dtype = torch.bfloat16 if "--bf16" in sys.argv[1:] else torch.float32
    u8 = "--u8" in sys.argv[1:]
    rank, world, local = parallel.init_from_env("nccl")
    dev = torch.device("cuda", local)
    wave, patch, terms, per = 128, 64, 10, 3
    B = per * world

    def build():
        cam = OpticsZernike(input_shape=[1, patch, patch, 3], device=dev, wave_resolution=(wave, wave), patch_size=patch,
                            sample_interval=3e-6, zernike_terms=terms, height_tolerance=None).to(dev)
        with torch.no_grad():
            cam.zernike_coeffs_train.fill_(-0.45)
            cam.zernike_coeffs_no_train2[1] = 0.3
        cam.sensor_dtype = out_dtype
        return cam

    g = torch.Generator().manual_seed(31)
    img = torch.rand(B, 3, patch, patch, generator=g)
    img[B - 2, 1, 20, 33] += 5.0                  # the batch maximum lives on the LAST rank's shard
    w = torch.rand(B, 3, patch, patch, generator=g)
    if u8:
        img = (img * 255.0).round().clamp(0, 255).to(torch.uint8)
        img[B - 2, 1, 16:24, 30:36] = 255         # a saturated patch on the last rank's shard

    whole = build()
    y_all, _, _, _ = whole(img.to(dev))
    (y_all * w.to(dev, out_dtype)).sum().backward()
    g_all = whole.zernike_coeffs_train.grad.clone()

    shard = build().data_parallel()
    sl = slice(rank * per, (rank + 1) * per)
    y, _, _, _ = shard(img[sl].to(dev))
    (y * w[sl].to(dev, out_dtype)).sum().backward()
    g_sum = shard.zernike_coeffs_train.grad.clone()
    dist.all_reduce(g_sum)

    same = True
    if u8:                                        # the same shards converted on the GPU: bit for bit
        conv = build().data_parallel()
        y32, _, _, _ = conv(img[sl].to(dev).to(torch.float32).div_(255.0))
        (y32 * w[sl].to(dev, out_dtype)).sum().backward()
        g32 = conv.zernike_coeffs_train.grad.clone()
        dist.all_reduce(g32)
        same = torch.equal(y.detach().float(), y32.detach().float()) and torch.equal(g_sum, g32)

    assert y.dtype == out_dtype
    y, y_ref = y.float(), y_all[sl].float()
    e_y = float((y - y_ref).norm() / y_ref.norm())
    e_g = float((g_sum - g_all).abs().max() / g_all.abs().max())
    ok = e_y <= 1e-6 and e_g <= 1e-4 and same
    flag = torch.tensor([1.0 if ok else 0.0], device=dev)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if rank == 0:
        print(f"LENS_SHARDED world={world} dtype={str(out_dtype).split('.')[-1]} u8={u8} sensor_rel={e_y:.2e} grad_rel={e_g:.2e} "
              f"ok={bool(flag.item())}", flush=True)
    dist.destroy_process_group()
    sys.exit(0 if flag.item() == 1.0 else 1)


if __name__ == "__main__":
    main()
