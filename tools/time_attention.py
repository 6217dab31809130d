"""Cost of the softmax attention mode on the B200, in one process:
  * the card (name, power limit, SM clock) and a device-to-device copy rate measured in the same run;
  * the temporal_attention kernel at the level-1 (C 256, 24x24) and level-2 (C 512, 12x12) batch-4 shapes of the
    benchmark, by CUDA events, inputs rotated over buffers larger than L2, and its rate on the algorithmic bytes
    B*T*P*(3C + C)*2 (qkv read once, o written once);
  * the U-Net step and the DDIM-50 generate() at batch 4 in reference and softmax mode, alternated A/B (>= 3 reps);
  * the per-op profile (b2v_unet_profile) of the softmax-mode step.
usage: python tools/time_attention.py [OUT_DIR]   (writes time_attention.txt and time_attention.json there; default:
the current directory)"""
import ctypes
import copy
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import bench  # noqa: E402
from v2v_b200 import _lib, ops  # noqa: E402
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


dev = torch.device("cuda:0")
q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                   capture_output=True, text=True).stdout.strip().splitlines()[0]
res["card"] = q
say(f"card (name, power limit, SM clock, max SM clock): {q}")

# device-to-device copy rate: 2 GiB per copy, read + write counted
src = torch.empty(1 << 30, dtype=torch.float16, device=dev).normal_()
dst = torch.empty_like(src)
ms = events_ms(lambda: dst.copy_(src), 20)
copy_rate = 2 * src.numel() * 2 / ms / 1e6  # GB/s
res["copy_GBps"] = copy_rate
say(f"device-to-device copy: {copy_rate:.0f} GB/s (2 GiB buffers, read + write)")
del src, dst

# the kernel at the benchmark's batch-4 attention shapes
res["kernel"] = []
for name, C, S in (("level1", 256, 24), ("level2", 512, 12)):
    B, T, heads = 4, 48, 4
    P = S * S
    one = B * T * P * 3 * C * 2
    nbuf = max(2, -(-400 * (1 << 20) // one))  # rotate over > 400 MB (L2 is 126 MB)
    g = torch.Generator(device=dev).manual_seed(C)
    qkv = [torch.randn((B, T, S, S, 3 * C), device=dev, generator=g).half() for _ in range(nbuf)]
    outs = [torch.empty((B, T, S, S, C), dtype=torch.float16, device=dev) for _ in range(nbuf)]
    L = _lib.lib()
    st = _lib.stream()
    i = [0]

    def run():
        k = i[0] % nbuf
        i[0] += 1
        _lib.check(L.b2v_temporal_attention(_lib.dptr(qkv[k], torch.float16), _lib.dptr(outs[k], torch.float16), B, T,
                                            P, C, heads, st), "temporal_attention")

    ms = events_ms(run, 200, warm=10)
    nbytes = B * T * P * (3 * C + C) * 2
    rate = nbytes / ms / 1e6
    r = dict(shape=name, B=B, C=C, HW=f"{S}x{S}", T=T, heads=heads, ms=ms, bytes=nbytes, GBps=rate,
             frac_of_copy=rate / copy_rate, buffers=nbuf)
    res["kernel"].append(r)
    say(f"temporal_attention {name} (B {B}, C {C}, {S}x{S}, T {T}, hd {C // heads}): {ms * 1e3:.1f} us, "
        f"{nbytes / 1e6:.0f} MB algorithmic -> {rate:.0f} GB/s = {100 * rate / copy_rate:.0f} % of the copy rate "
        f"({nbuf} rotating buffers)")
    del qkv, outs

# U-Net step and generate() in both modes, alternated
torch.manual_seed(0)
m_ref = VideoToVideoDiffusion(bench.load_cfg()).eval().to(dev)
m_sm = copy.deepcopy(m_ref)
m_sm.unet.set_attention_mode("softmax")
B = 4
g = torch.Generator(device=dev).manual_seed(1)
x = torch.randn((B, 8, 48, 48, 48), device=dev, generator=g)
c = torch.randn_like(x)
t = torch.full((B,), 500, device=dev)
v = torch.rand((B, 1, 8, 192, 192), device=dev, generator=g) * 2 - 1
steps = {"reference": [], "softmax": []}
gens = {"reference": [], "softmax": []}
models = {"reference": m_ref, "softmax": m_sm}
for mode, m in models.items():  # warm-up: program build, graph capture
    m.unet(x, t, c)
    m.generate(v, "ddim", 2, target_depth=48)
for rep in range(3):
    for mode, m in models.items():
        steps[mode].append(events_ms(lambda: m.unet(x, t, c), 30))
    for mode, m in models.items():
        torch.manual_seed(7)
        gens[mode].append(events_ms(lambda: m.generate(v, "ddim", 50, target_depth=48), 1, warm=0))
res["unet_step_ms"] = steps
res["generate_ddim50_ms_per_batch"] = gens
for mode in models:
    say(f"U-Net step, batch {B}, {mode:9s}: " + ", ".join(f"{s:.3f}" for s in steps[mode]) + " ms;  "
        f"DDIM-50 generate per batch: " + ", ".join(f"{s:.1f}" for s in gens[mode]) + " ms")
ratio = min(steps["softmax"]) / min(steps["reference"])
gratio = min(gens["softmax"]) / min(gens["reference"])
res["step_ratio"], res["generate_ratio"] = ratio, gratio
say(f"softmax / reference (best of 3): U-Net step {ratio:.3f}x, generate {gratio:.3f}x")

# per-op profile of the softmax-mode step
m_sm.unet(x, t, c)
torch.cuda.synchronize()
buf = ctypes.create_string_buffer(1 << 20)
_lib.check(_lib.lib().b2v_unet_profile(m_sm.unet.native(dev), 5, buf, len(buf), _lib.stream()), "unet_profile")
prof = json.loads(buf.value.decode())
res["softmax_step_profile"] = prof
tot = sum(o["ms"] for o in prof)
att = [o for o in prof if ".attn." in o["name"]]
say(f"softmax-mode step, per-op profile: {tot:.3f} ms in {len(prof)} ops; attention ops {sum(o['ms'] for o in att):.3f} ms")
for o in att:
    gb = o["bytes"] / o["ms"] / 1e6 if o["bytes"] else 0
    say(f"  {o['name']:28s} {o['ms']:8.4f} ms  {gb:7.0f} GB/s")

open(os.path.join(out_dir, "time_attention.txt"), "w").write("\n".join(lines) + "\n")
json.dump(res, open(os.path.join(out_dir, "time_attention.json"), "w"), indent=1)
