"""Cost of ensemble generation on the B200, in one process:
  * the card (name, power limit, SM clock) and a device-to-device copy rate measured in the same run;
  * the ensemble_stats kernel (K*4 + 8 B per voxel) at K = 4 / B = 4 / 48 x 192^2 and at K = 8 / B = 1 / 48 x 512^2, by
    torch.profiler kernel time, inputs rotated over buffers larger than L2, as bytes/s against the copy rate;
  * at batch 1, 8 -> 48 slices at 192^2, dpmpp_2m-10 with K = 4: generate_ensemble, four sequential generate() calls,
    and one generate() on the input repeated 4 times (the same sampling at batch K*B, K encodes), alternated over 3
    repetitions.
usage: python tools/time_ensemble.py [OUT_DIR]   (writes time_ensemble.txt and time_ensemble.json there; default: the
current directory)"""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from v2v_b200 import ops  # noqa: E402
from v2v_b200.inference.ensemble import generate_ensemble  # noqa: E402
from v2v_b200.models import VideoToVideoDiffusion  # noqa: E402

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


def kernel_us(fn, kname, n=50):
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

# the statistics kernel, rotating over > 400 MB of members (L2 is 126 MB)
g = torch.Generator(device=dev).manual_seed(0)
res["ensemble_stats"] = {}
for K, B, D, H in ((4, 4, 48, 192), (8, 1, 48, 512)):
    n = B * D * H * H
    nbuf = max(2, -(-400 * (1 << 20) // (K * n * 4)))
    mem = [torch.rand((K, n), device=dev, generator=g) * 2 - 1 for _ in range(nbuf)]
    it = [0]

    def fn():
        it[0] += 1
        ops.ensemble_stats(mem[it[0] % nbuf])
    us = kernel_us(fn, "ensemble_stats_kernel")
    nbytes = n * (4 * K + 8)
    rate = nbytes / us / 1e3
    key = f"K{K}_B{B}_{D}x{H}^2"
    res["ensemble_stats"][key] = dict(kernel_us=us, bytes=nbytes, GBps=rate, frac_of_copy=rate / copy_rate)
    say(f"ensemble_stats {key}: {nbytes / 1e6:.1f} MB in {us:.1f} us (profiler) -> {rate:.0f} GB/s = "
        f"{100 * rate / copy_rate:.0f} % of the copy rate ({nbuf} rotating buffers)")
    del mem

# batch 1, K = 4, dpmpp_2m-10 at the benchmark's patch shape
torch.manual_seed(0)
m = VideoToVideoDiffusion(bench.load_cfg()).eval().to(dev)
K, steps = 4, 10
v = torch.rand((1, 1, 8, 192, 192), device=dev, generator=g) * 2 - 1
v_rep = v.repeat(K, 1, 1, 1, 1).contiguous()


def sequential():
    for _ in range(K):
        m.generate(v, "dpmpp_2m", steps, target_depth=48)


arms = {"generate_ensemble": lambda: generate_ensemble(m, v, "dpmpp_2m", steps, K, target_depth=48),
        "4x generate() batch 1": sequential,
        "generate() on the repeated input, batch 4": lambda: m.generate(v_rep, "dpmpp_2m", steps, target_depth=48)}
for fn in arms.values():  # warm-up: program build, graph capture, time-embedding tables, workspaces
    fn()
times = {k: [] for k in arms}
for rep in range(3):
    for k, fn in arms.items():
        torch.manual_seed(7)
        times[k].append(events_ms(fn, 1, warm=0))
res["ms"] = times
best = {k: min(t) for k, t in times.items()}
base = best["generate() on the repeated input, batch 4"]
for k, t in times.items():
    say(f"{k:42s}: " + ", ".join(f"{x:.1f}" for x in t) + f" ms; best {best[k]:.1f} ms = {best[k] / base:.3f}x the "
        "repeated-input generate()")
res["ensemble_vs_repeated"] = best["generate_ensemble"] / base
res["ensemble_vs_sequential"] = best["generate_ensemble"] / best["4x generate() batch 1"]
say(f"generate_ensemble / 4 sequential generate(): {res['ensemble_vs_sequential']:.3f}")

open(os.path.join(out_dir, "time_ensemble.txt"), "w").write("\n".join(lines) + "\n")
json.dump(res, open(os.path.join(out_dir, "time_ensemble.json"), "w"), indent=1)
