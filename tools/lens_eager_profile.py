import sys, time
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import torch
from b200cam.lens import OpticsZernike
dev = torch.device("cuda", 0)
B = 128
cam = OpticsZernike(input_shape=[None, 256, 256, 3], device=dev, zernike_terms=350, patch_size=256, height_tolerance=2e-8,
                    sensor_distance=0.025, wave_resolution=[896, 896], sample_interval=3e-06, upsample=False).to(dev)
img = torch.rand(B, 3, 256, 256, device=dev); w = torch.rand(B, 3, 256, 256, device=dev)
def step():
    cam.zero_grad(set_to_none=True)
    s, p, c, l = cam(img)
    torch.autograd.backward([s], [w])
for _ in range(5): step()
torch.cuda.synchronize()
t0 = time.perf_counter()
for _ in range(20): step()
t_launch = (time.perf_counter() - t0) / 20
torch.cuda.synchronize()
t_total = (time.perf_counter() - t0) / 20
print(f"host time to enqueue one step {t_launch*1e3:.2f} ms; wall per step incl. GPU {t_total*1e3:.2f} ms")
import cProfile, pstats
pr = cProfile.Profile(); pr.enable()
for _ in range(10): step()
pr.disable(); torch.cuda.synchronize()
pstats.Stats(pr).sort_stats("cumulative").print_stats(18)
