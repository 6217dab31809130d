"""Cost of the DPM-Solver++(2M) sampler on the B200, in one process:
  * the card (name, power limit, SM clock) and a device-to-device copy rate measured in the same run;
  * the dpmpp_update kernel (ODE: 20 B per element, SDE: 24 B) and ddim_update (12 B) at the benchmark's batch-4 latent
    (4, 8, 48, 48, 48), by CUDA events, inputs rotated over buffers larger than L2, as bytes/s against the copy rate;
  * generate() at the benchmark shape (batch 4, 8 -> 48 slices, 192^2) for DDIM-50 and dpmpp_2m at 10 / 15 / 20 / 25
    steps, alternated A/B over 3 repetitions: ms per batch and patch-volumes/s.
usage: python tools/time_samplers.py [OUT_DIR]   (writes time_samplers.txt and time_samplers.json there; default: the
current directory)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402
from v2v_b200 import ops  # noqa: E402
from v2v_b200.inference.sampler import dpmpp_coefficients  # noqa: E402
from v2v_b200.models import GaussianDiffusion, VideoToVideoDiffusion  # noqa: E402

out_dir = sys.argv[1] if len(sys.argv) > 1 else os.getcwd()
os.makedirs(out_dir, exist_ok=True)
lines, res = [], {}


def say(s):
    print(s, flush=True)
    lines.append(s)


def events_ms(fn, n, warm=3):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


dev = torch.device("cuda:0")
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip().splitlines()[0]
res["card"] = q
say(f"card (name, power limit, SM clock, max SM clock): {q}")

src = torch.empty(1 << 29, dtype=torch.float32, device=dev).normal_()  # 2 GiB per copy, read + write counted
dst = torch.empty_like(src)
ms = events_ms(lambda: dst.copy_(src), 20)
copy_rate = 2 * src.numel() * 4 / ms / 1e6  # GB/s
res["copy_GBps"] = copy_rate
say(f"device-to-device copy: {copy_rate:.0f} GB/s (2 GiB buffers, read + write)")
del src, dst

# the update kernels at the batch-4 latent, rotating over > 400 MB of inputs (L2 is 126 MB)
numel = 4 * 8 * 48 * 48 * 48
nbuf = max(2, -(-400 * (1 << 20) // (4 * numel * 4)))
g = torch.Generator(device=dev).manual_seed(0)
z = [torch.randn(numel, device=dev, generator=g) for _ in range(nbuf)]
eps = [torch.randn(numel, device=dev, generator=g) for _ in range(nbuf)]
x0p = [torch.randn(numel, device=dev, generator=g) for _ in range(nbuf)]
nz = [torch.randn(numel, device=dev, generator=g) for _ in range(nbuf)]
acp = GaussianDiffusion("cosine", 1000).alphas_cumprod.float()  # the benchmark config's schedule
ts = np.array([500, 480, 460, 0], dtype=np.int64)
row_ode = dpmpp_coefficients(ts, acp, 2, False)[1].to(dev)  # an order-2 row (x0_prev read)
row_sde = dpmpp_coefficients(ts, acp, 2, True)[1].to(dev)
a_t, a_p = acp[500], acp[480]
ddim_coef = torch.tensor([float(torch.sqrt(1 - a_t + 1e-8)), float(torch.sqrt(a_t + 1e-8) + 1e-8),
                          float(torch.sqrt(a_p + 1e-8)), float(torch.sqrt(1 - a_p + 1e-8)), 0, 0, 0, 0], device=dev)
it = [0]


def nxt():
    it[0] += 1
    return it[0] % nbuf


kern = {
    "ddim_update": (lambda: (lambda k: ops.ddim_update(z[k], eps[k], ddim_coef))(nxt()), 12),
    "dpmpp_update_ode": (lambda: (lambda k: ops.dpmpp_update(z[k], x0p[k], eps[k], row_ode))(nxt()), 20),
    "dpmpp_update_sde": (lambda: (lambda k: ops.dpmpp_update(z[k], x0p[k], eps[k], row_sde, nz[k]))(nxt()), 24),
}
res["kernels"] = {}


def kernel_us(fn, kname, n=200):
    """mean device time of the kernel `kname` over n calls, from torch.profiler's CUDA activity records"""
    fn()
    torch.cuda.synchronize()
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    tot = cnt = 0
    for e in prof.key_averages():
        if kname in e.key:
            tot += getattr(e, "device_time_total", None) or e.cuda_time_total
            cnt += e.count
    return tot / cnt


for name, (fn, bpe) in kern.items():
    # per call through the Python op wrapper (ctypes call, NaN-flag allocation): host-bound at this size
    call_us = events_ms(fn, 200, warm=10) * 1e3
    us = kernel_us(fn, "ddim_update_kernel" if name == "ddim_update" else "dpmpp_update_kernel")
    rate = numel * bpe / us / 1e3
    res["kernels"][name] = dict(kernel_us=us, call_us=call_us, bytes_per_elem=bpe, GBps=rate,
                                frac_of_copy=rate / copy_rate)
    say(f"{name:18s} numel {numel}: kernel {us:6.1f} us (profiler), {bpe} B/elem -> {rate:.0f} GB/s = "
        f"{100 * rate / copy_rate:.0f} % of the copy rate; {call_us:.1f} us per wrapper call ({nbuf} rotating buffer sets)")
for k in ("dpmpp_update_ode", "dpmpp_update_sde"):
    extra = res["kernels"][k]["kernel_us"] - res["kernels"]["ddim_update"]["kernel_us"]
    res["kernels"][k]["us_over_ddim"] = extra
    say(f"{k} - ddim_update: {extra:+.1f} us per step (kernel time)")
del z, eps, x0p, nz

# generate() at the benchmark shape, alternated
torch.manual_seed(0)
m = VideoToVideoDiffusion(bench.load_cfg()).eval().to(dev)
B = 4
v = torch.rand((B, 1, 8, 192, 192), device=dev, generator=g) * 2 - 1
runs = [("ddim", 50)] + [("dpmpp_2m", s) for s in (10, 15, 20, 25)]
for s, n in runs:  # warm-up: program build, graph capture, time-embedding tables
    m.generate(v, s, n, target_depth=48)
times = {f"{s}-{n}": [] for s, n in runs}
for rep in range(3):
    for s, n in runs:
        torch.manual_seed(7)
        times[f"{s}-{n}"].append(events_ms(lambda: m.generate(v, s, n, target_depth=48), 1, warm=0))
res["generate_ms_per_batch"] = times
base = min(times["ddim-50"])
for key, ts_ in times.items():
    best = min(ts_)
    res.setdefault("summary", {})[key] = dict(best_ms=best, patch_volumes_per_s=B * 1000 / best, vs_ddim50=best / base)
    say(f"generate {key:12s} batch {B}: " + ", ".join(f"{t:.1f}" for t in ts_) + f" ms; best {best:.1f} ms = "
        f"{B * 1000 / best:.2f} patch-volumes/s, {best / base:.3f}x DDIM-50")

open(os.path.join(out_dir, "time_samplers.txt"), "w").write("\n".join(lines) + "\n")
json.dump(res, open(os.path.join(out_dir, "time_samplers.json"), "w"), indent=1)
