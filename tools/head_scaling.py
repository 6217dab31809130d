import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from v2v_b200 import ops
dev = torch.device("cuda:0")
g = torch.Generator().manual_seed(0)
for cout in (1, 8):
    for (B, D, H) in [(1, 48, 96), (1, 48, 192), (4, 48, 192)] if cout == 1 else [(1, 48, 48), (4, 48, 48), (4, 48, 96)]:
        x16 = torch.randn((B, D, H, H, 128), device=dev, dtype=torch.float16)
        w = torch.randn((cout, 128, 3, 3, 3), generator=g) / 60.0
        conv = ops.Conv(0, w, torch.zeros(cout), 128, 0, cout)
        for _ in range(2):
            conv(x16, out_fp32=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(5):
            conv(x16, out_fp32=True)
        e1.record(); torch.cuda.synchronize()
        pos = B * D * H * H
        print(f"cout={cout} positions={pos/1e6:.2f}M  {e0.elapsed_time(e1)/5:.4f} ms  P={27*cout*pos*4/1e6:.0f} MB in={pos*256/1e6:.0f} MB")
        del x16, conv
