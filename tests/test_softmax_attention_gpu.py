"""The opt-in softmax temporal attention on the B200: the fused tcgen05 kernel against fp32 attention, GroupNorm mode 2,
and the U-Net / generate() in softmax mode against the fp32 softmax oracle (tests/softmax_oracle.py)."""
import os

import pytest
import torch
import torch.nn.functional as F

from helpers import TINY_UNET, rel_l2
from oracle import ref_port as R
import softmax_oracle as S

pytestmark = pytest.mark.gpu
EPS_TOL = 1e-2


@pytest.fixture(scope="module")
def dev():
    if not torch.cuda.is_available():
        pytest.skip("no GPU")
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return torch.device("cuda:0")


def _sd(m, d):
    return {k: v.to(d) for k, v in m.state_dict().items()}


def _attention_fp32(qkv, heads):
    """fp32 attention of an fp16 qkv tensor (B,T,H,W,3C) -> (B,T,H,W,C), through torch's SDPA"""
    B, T, H, W, C3 = qkv.shape
    C = C3 // 3
    hd = C // heads
    x = qkv.float().reshape(B, T, H * W, 3, heads, hd).permute(3, 0, 2, 4, 1, 5)  # (3, B, P, heads, T, hd)
    o = F.scaled_dot_product_attention(x[0], x[1], x[2])  # (B, P, heads, T, hd)
    return o.permute(0, 3, 1, 2, 4).reshape(B, T, H, W, C)


@pytest.mark.parametrize("B,C,heads,T,H,W", [
    (4, 256, 4, 48, 24, 24),   # level-1 block of the benchmark at batch 4 (hd 64)
    (4, 512, 4, 48, 12, 12),   # level-2 / mid block (hd 128)
    (1, 128, 2, 5, 7, 9),      # short depth, odd positions
    (1, 256, 4, 160, 6, 6),    # several query and key tiles: the online softmax
    (2, 192, 4, 48, 6, 6),     # hd 48: a partial 64-channel chunk
    (1, 64, 4, 17, 8, 8),      # hd 16
])
def test_temporal_attention_kernel_vs_fp32_sdpa(dev, B, C, heads, T, H, W):
    from v2v_b200 import ops
    g = torch.Generator().manual_seed(B * 1000 + C + T)
    qkv = torch.randn((B, T, H, W, 3 * C), generator=g).to(dev).half()
    got = ops.temporal_attention(qkv, heads)
    ref = _attention_fp32(qkv, heads)
    # P is rounded to fp16 before the P V product and o is stored in fp16: two roundings of 2^-11 relative each, on
    # values bounded by max|o| (a convex combination of V rows); 2e-3 of max|ref| leaves a factor 2 of headroom
    err = (got.float() - ref).abs().max().item()
    scale = ref.abs().max().item()
    print(f"temporal_attention B{B} C{C} heads{heads} T{T} {H}x{W}: max err {err:.3e} = {err / scale:.2e} of max|ref|")
    assert err <= 2e-3 * scale, (err, scale)
    assert torch.equal(ops.temporal_attention(qkv, heads), got)  # same bits on a second run


def test_temporal_attention_rejects_unsupported_head_dim(dev):
    from v2v_b200 import ops
    qkv = torch.zeros((1, 4, 2, 2, 3 * 64), dtype=torch.float16, device=dev)
    with pytest.raises(RuntimeError, match="head_dim"):
        ops.temporal_attention(qkv, 8)  # hd 8
    with pytest.raises(RuntimeError, match="head_dim"):
        ops.temporal_attention(torch.zeros((1, 4, 2, 2, 3 * 288), dtype=torch.float16, device=dev), 2)  # hd 144


def test_gn_apply_mode2_is_group_norm(dev):
    from v2v_b200 import ops
    g = torch.Generator().manual_seed(21)
    B, C, D, H, W, G = 2, 256, 6, 10, 12, 32
    x = (torch.randn((B, C, D, H, W), generator=g) * 1.7 + 0.3).to(dev)
    gamma = (1 + 0.2 * torch.randn(C, generator=g)).to(dev)
    beta = (0.2 * torch.randn(C, generator=g)).to(dev)
    y = ops.to_cl16(x)
    stats = ops.gn_stats(y, G)
    out, _ = ops.gn_apply(y, stats, gamma, beta, G, mode=2)
    ref = F.group_norm(ops.from_cl16(y), G, gamma, beta, 1e-5)
    got = ops.from_cl16(out)
    assert torch.equal(ops.from_cl16(y), ops.from_cl16(y.clone()))  # input untouched: out of place
    err = (got - ref).abs().max().item()
    assert err <= 2e-3 * ref.abs().max().item(), err


def _op_names(m):
    from v2v_b200 import _lib
    L, h, names, i = _lib.lib(), m._native.handle, [], 0
    while True:
        n = L.b2v_debug_op_name(h, 0, i).decode()
        if not n:
            return names
        names.append(n)
        i += 1


def test_tiny_unet_softmax_mode_vs_oracle_and_mode_switch(dev):
    from v2v_b200.models import UNet3D
    torch.manual_seed(0)
    m = UNet3D(**TINY_UNET).eval().to(dev)
    sd = _sd(m, dev)
    g = torch.Generator().manual_seed(2)
    x = torch.randn((2, 4, 12, 8, 8), generator=g).to(dev)
    c = torch.randn((2, 4, 12, 8, 8), generator=g).to(dev)
    t = torch.tensor([999, 40], device=dev)
    ref_mode = m(x, t, c)
    names = _op_names(m)
    assert not any(n.endswith((".attn.core", ".attn.qkv")) for n in names), names
    m.set_attention_mode("softmax")
    got = m(x, t, c)
    names = _op_names(m)
    assert sum(n.endswith(".attn.core") for n in names) == 4, names  # down1.0, mid, up0.0, up0.1
    with torch.no_grad():
        want = S.unet_forward(sd, TINY_UNET, x, t, c)
        want_ref = R.unet_forward(sd, TINY_UNET, x, t, c)
    err = rel_l2(got, want)
    print(f"tiny U-Net softmax mode: rel-L2 {err:.3e} (reference-mode output differs by {rel_l2(want_ref, want):.3e})")
    assert err <= EPS_TOL, err
    assert rel_l2(want_ref, want) > 10 * EPS_TOL  # the mode changes the model
    assert torch.equal(m(x, t, c), got)
    m.set_attention_mode("reference")
    assert torch.equal(m(x, t, c), ref_mode)


@pytest.mark.parametrize("cfg", [
    # attention at the only level: the last decoder block's attention feeds conv_out's GroupNorm
    dict(latent_dim=4, model_channels=64, num_res_blocks=1, attention_levels=[0], channel_mult=(1,), num_heads=2,
         time_embed_dim=128),
    # 192 / 384 channels: hd 48 / 96, GroupNorm widths that are not powers of two
    dict(latent_dim=4, model_channels=192, num_res_blocks=1, attention_levels=[1], channel_mult=(1, 2), num_heads=4,
         time_embed_dim=128),
], ids=["single_level_attn_before_conv_out", "model_channels_192"])
def test_unet_softmax_mode_extra_configs(dev, cfg):
    from v2v_b200.models import UNet3D
    torch.manual_seed(3)
    m = UNet3D(**cfg).eval().to(dev).set_attention_mode("softmax")
    sd = _sd(m, dev)
    g = torch.Generator().manual_seed(12)
    x = torch.randn((2, 4, 9, 8, 12), generator=g).to(dev)
    c = torch.randn((2, 4, 9, 8, 12), generator=g).to(dev)
    t = torch.tensor([999, 17], device=dev)
    with torch.no_grad():
        ref = S.unet_forward(sd, cfg, x, t, c)
    got = m(x, t, c)
    err = rel_l2(got, ref)
    print(f"U-Net softmax mode {cfg['model_channels']}ch levels {cfg['attention_levels']}: rel-L2 {err:.3e}")
    assert err <= EPS_TOL, err
    assert torch.equal(m(x, t, c), got)


@pytest.fixture(scope="module")
def bench_softmax(dev):
    import yaml
    from v2v_b200.models import VideoToVideoDiffusion
    cfg = yaml.safe_load(open(os.path.join(os.path.dirname(__file__), "golden", "slice_interpolation_full_medium.yaml")))
    cfg = dict(cfg, unet_attention="softmax")
    torch.manual_seed(0)
    m = VideoToVideoDiffusion(cfg).eval().to(dev)
    assert m.unet.attention_mode == "softmax"
    return m, cfg


@pytest.mark.timeout(900)
@pytest.mark.parametrize("batch", [1, 4])
def test_bench_config_unet_softmax_vs_fp32_oracle(dev, bench_softmax, batch):
    m, cfg = bench_softmax
    _, unet_cfg, _ = R.resolve_config(cfg)
    sd = {k[len("unet."):]: v for k, v in m.state_dict().items() if k.startswith("unet.")}
    g = torch.Generator().manual_seed(30 + batch)
    x = torch.randn((batch, 8, 48, 48, 48), generator=g).to(dev)
    c = torch.randn((batch, 8, 48, 48, 48), generator=g).to(dev)
    ts = [[999] * batch, [500] * batch, [0] * batch]
    if batch == 4:
        ts.append([0, 250, 750, 999])  # per-sample timesteps
    for tv in ts:
        t = torch.tensor(tv, device=dev)
        got = m.unet(x, t, c)
        with torch.no_grad():
            ref = S.unet_forward(sd, unet_cfg, x, t, c)
        errs = [rel_l2(got[i], ref[i]) for i in range(batch)]
        print(f"softmax-mode U-Net batch {batch} t={tv}: per-sample rel-L2 {['%.2e' % e for e in errs]}")
        assert max(errs) <= EPS_TOL, (tv, errs)


@pytest.mark.timeout(2400)
def test_generate_ddim50_batch4_softmax_mode_all_gates(dev, bench_softmax):
    """test_full_generate_ddim50_all_gates (batch 4) with both sides in softmax mode:
      1. teacher-forced eps rel-L2 <= 1e-2 at all 51 steps;  2. decode of the reference z_0 >= 60 dB;
      3. |PSNR(new, target) - PSNR(ref, target)| <= 0.05 dB;  4. the same seed gives the same bits."""
    m, cfg = bench_softmax
    sd = _sd(m, dev)
    vae_cfg, unet_cfg, _ = R.resolve_config(cfg)
    batch = 4
    g = torch.Generator().manual_seed(1234)
    v_thick = (torch.rand((batch, 1, 8, 192, 192), generator=g) * 2 - 1).to(dev)
    target = (torch.rand((batch, 1, 48, 192, 192), generator=g) * 2 - 1).to(dev)
    torch.manual_seed(42)
    with torch.no_grad():  # the reference generate() piece by piece, keeping what the teacher-forced gates need
        z_in = R.vae_encode(sd, v_thick, vae_cfg["scaling_factor"], "vae.")
        cond = F.interpolate(z_in, size=(48, z_in.shape[3], z_in.shape[4]), mode="trilinear", align_corners=False)
        torch.randn(tuple(cond.shape), device=dev)  # discarded draw (models/model.py:303)
        buffers = {k[len("diffusion."):]: v for k, v in sd.items() if k.startswith("diffusion.")}
        rec = []
        model = lambda z, t, c: S.unet_forward(sd, unet_cfg, z, t, c, "unet.")  # noqa: E731
        z0 = R.ddim_sample(model, buffers, tuple(cond.shape), cond, 50, dev, record=rec)
        ref = R.vae_decode(sd, z0, vae_cfg["scaling_factor"], "vae.")
    assert len(rec) == 51
    errs = []
    for z_t, t_idx, eps_ref in rec:
        t = torch.full((batch,), t_idx, device=dev, dtype=torch.long)
        errs.append(rel_l2(m.unet(z_t, t, cond), eps_ref))
    print(f"softmax mode, batch 4: teacher-forced eps rel-L2 over 51 steps: max {max(errs):.3e} "
          f"(t={rec[errs.index(max(errs))][1]}), mean {sum(errs) / len(errs):.3e}")
    assert max(errs) <= EPS_TOL, errs
    n = lambda v: (v.clamp(-1, 1) + 1) / 2  # noqa: E731
    p_dec = R.psnr(n(m.vae.decode(z0)), n(ref))
    print(f"softmax mode, batch 4: teacher-forced decode PSNR(new, ref) = {p_dec:.1f} dB")
    assert p_dec >= 60.0, p_dec
    torch.manual_seed(42)
    got = m.generate(v_thick, "ddim", 50, target_depth=48)
    assert got.shape == ref.shape and torch.isfinite(got).all()
    p_new, p_ref, p_direct = R.psnr(n(got), n(target)), R.psnr(n(ref), n(target)), R.psnr(n(got), n(ref))
    print(f"softmax mode, batch 4: generate DDIM-50 PSNR(new,target)={p_new:.4f} PSNR(ref,target)={p_ref:.4f} "
          f"PSNR(new,ref)={p_direct:.2f} dB")
    assert abs(p_new - p_ref) <= 0.05, (p_new, p_ref)
    assert m.last_nan_flag.item() == 0
    torch.manual_seed(42)
    assert torch.equal(m.generate(v_thick, "ddim", 50, target_depth=48), got)
