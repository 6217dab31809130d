"""graph-replay timing of the U-Net step / VAE decode at the bench shape (CUDA events over N replays)"""
import sys, os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch
import bench
from v2v_b200.models import VideoToVideoDiffusion
B = int(sys.argv[1]) if len(sys.argv) > 1 else 4
N = int(sys.argv[2]) if len(sys.argv) > 2 else 60
dev = torch.device("cuda:0")
torch.manual_seed(0)
m = VideoToVideoDiffusion(bench.load_cfg()).eval().to(dev)
x = torch.randn((B, 8, 48, 48, 48), device=dev); c = torch.randn_like(x); t = torch.full((B,), 500, device=dev)
def timeit(fn, n):
    for _ in range(3): fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n): fn()
    e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n
tu = timeit(lambda: m.unet(x, t, c), N)
td = timeit(lambda: m.vae.decode(x), 5)
v = torch.rand((B, 1, 8, 192, 192), device=dev) * 2 - 1
te = timeit(lambda: m.vae.encode(v), 5)
print(f"B={B}: unet_step {tu:.3f} ms  decode {td:.3f} ms  encode {te:.3f} ms")
