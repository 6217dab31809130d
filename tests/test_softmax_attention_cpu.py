"""The opt-in softmax temporal attention, on the CPU: the oracle's softmax block against torch's attention, the
identity-augmented projection the U-Net program uses for the residual, and the Python plumbing of the mode."""
import pytest
import torch
import torch.nn.functional as F

from helpers import TINY_UNET, sd_hash
from oracle import ref_port as R
import softmax_oracle as S


def _attn_sd(C, seed):
    g = torch.Generator().manual_seed(seed)
    r = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)  # noqa: E731
    return {"a.norm.weight": 1 + 0.1 * r(C), "a.norm.bias": 0.1 * r(C),
            "a.qkv.weight": r(3 * C, C, 1, 1, 1) / C ** 0.5, "a.qkv.bias": 0.1 * r(3 * C),
            "a.proj_out.weight": r(C, C, 1, 1, 1) / C ** 0.5, "a.proj_out.bias": 0.1 * r(C)}


def _qkv(sd, x, heads):
    """the block's q, k, v as (B*H*W, heads, T, hd), computed independently of the oracle"""
    B, C, T, H, W = x.shape
    h = F.group_norm(x, R.num_groups(C), sd["a.norm.weight"], sd["a.norm.bias"], 1e-5)
    qkv = F.conv3d(h, sd["a.qkv.weight"], sd["a.qkv.bias"])
    hd = C // heads

    def seq(a):
        return a.reshape(B, heads, hd, T, H, W).permute(0, 4, 5, 1, 3, 2).reshape(B * H * W, heads, T, hd)

    return seq(qkv[:, :C]), seq(qkv[:, C:2 * C]), seq(qkv[:, 2 * C:])


def _unseq(o, B, C, T, H, W, heads):
    return o.reshape(B, H, W, heads, T, C // heads).permute(0, 3, 5, 4, 1, 2).reshape(B, C, T, H, W)


@pytest.mark.parametrize("B,C,heads,T,H,W", [(2, 64, 4, 7, 3, 5), (1, 128, 2, 48, 2, 2), (1, 32, 2, 1, 2, 3)])
def test_oracle_softmax_block_equals_sdpa_and_textbook_einsum(B, C, heads, T, H, W):
    sd = _attn_sd(C, seed=C + T)
    x = torch.randn((B, C, T, H, W), generator=torch.Generator().manual_seed(T), dtype=torch.float64)
    got = S.unet_attention_softmax(sd, "a", x, heads)
    q, k, v = _qkv(sd, x, heads)
    # torch's attention on the same q, k, v (default scale 1/sqrt(hd))
    o = F.scaled_dot_product_attention(q, k, v)
    want = F.conv3d(_unseq(o, B, C, T, H, W, heads), sd["a.proj_out.weight"], sd["a.proj_out.bias"]) + x
    assert (got - want).abs().max().item() <= 1e-10
    # the textbook module: the reference's TemporalAttention with its second einsum corrected to 'bhqk,bhkc->bhqc'
    hd = C // heads
    attn = torch.softmax(torch.einsum("bhqc,bhkc->bhqk", q, k) * hd ** -0.5, dim=-1)
    o2 = torch.einsum("bhqk,bhkc->bhqc", attn, v)
    want2 = F.conv3d(_unseq(o2, B, C, T, H, W, heads), sd["a.proj_out.weight"], sd["a.proj_out.bias"]) + x
    assert (got - want2).abs().max().item() <= 1e-10


def test_softmax_block_is_not_the_reference_block():
    C, heads = 64, 4
    sd = _attn_sd(C, seed=3)
    x = torch.randn((1, C, 12, 3, 3), generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    ref = R.unet_attention(sd, "a", x, heads)
    sm = S.unet_attention_softmax(sd, "a", x, heads)
    # relative to the attention branch itself (the residual x is common to both)
    assert ((sm - ref).norm() / (ref - x).norm()).item() > 0.1
    # and the reference block does not depend on q, k: scrambling them leaves it unchanged, but not the softmax block
    sd2 = dict(sd)
    sd2["a.qkv.weight"] = sd["a.qkv.weight"].clone()
    sd2["a.qkv.weight"][:2 * C] *= -3.0
    assert torch.allclose(R.unet_attention(sd2, "a", x, heads), ref, rtol=0, atol=1e-10)
    assert not torch.allclose(S.unet_attention_softmax(sd2, "a", x, heads), sm, rtol=0, atol=1e-3)


def test_softmax_unet_forward_differs_and_agrees_at_one_token():
    """the softmax oracle U-Net is a different model at T > 1; with one depth token the softmax is exactly 1 and both
    contractions give V, so it must reproduce oracle/ref_port.py's unet_forward"""
    from v2v_b200.models import UNet3D
    torch.manual_seed(0)
    m = UNet3D(**TINY_UNET).eval()
    sd = m.state_dict()
    g = torch.Generator().manual_seed(1)
    t = torch.tensor([500])
    for T, same in ((5, False), (1, True)):
        x = torch.randn((1, 4, T, 4, 4), generator=g)
        c = torch.randn((1, 4, T, 4, 4), generator=g)
        with torch.no_grad():
            ref = R.unet_forward(sd, TINY_UNET, x, t, c)
            sm = S.unet_forward(sd, TINY_UNET, x, t, c)
        assert torch.allclose(ref, sm, rtol=0, atol=1e-6) == same, (T, (ref - sm).abs().max().item())


def test_identity_augmented_projection_is_proj_plus_residual():
    """the U-Net program computes proj_out(o) + x as ONE 1x1 conv over cat(o, x) with weight [Wp | I] and bias bp"""
    C = 48
    sd = _attn_sd(C, seed=9)
    g = torch.Generator().manual_seed(10)
    o = torch.randn((2, C, 5, 3, 4), generator=g, dtype=torch.float64)
    x = torch.randn((2, C, 5, 3, 4), generator=g, dtype=torch.float64)
    Wp, bp = sd["a.proj_out.weight"], sd["a.proj_out.bias"]
    Wcat = torch.cat([Wp, torch.eye(C, dtype=torch.float64).view(C, C, 1, 1, 1)], dim=1)
    got = F.conv3d(torch.cat([o, x], dim=1), Wcat, bp)
    want = F.conv3d(o, Wp, bp) + x
    assert (got - want).abs().max().item() <= 1e-12


def test_mirror_attention_mode_plumbing():
    from v2v_b200.models import UNet3D
    torch.manual_seed(0)
    m = UNet3D(**TINY_UNET).eval()
    assert m.attention_mode == "reference"
    h0 = sd_hash(m.state_dict())
    keys = list(m.state_dict())
    assert m.set_attention_mode("softmax") is m and m.attention_mode == "softmax"
    assert sd_hash(m.state_dict()) == h0 and list(m.state_dict()) == keys  # the mode is not a parameter or buffer
    m.set_attention_mode("reference")
    assert m.attention_mode == "reference"
    with pytest.raises(ValueError):
        m.set_attention_mode("flash")
    assert m.attention_mode == "reference"
    # head_dim outside {16, 32, ..., 128}: 64 channels / 8 heads = 8
    bad = UNet3D(**dict(TINY_UNET, attention_levels=[0], channel_mult=(1,), num_heads=8)).eval()
    with pytest.raises(ValueError, match="head_dim"):
        bad.set_attention_mode("softmax")
    assert bad.attention_mode == "reference"
    # 192 channels / 2 heads = 96 at level 0 is fine, but 384 / 2 = 192 at the mid block is not
    wide = UNet3D(latent_dim=4, model_channels=192, num_res_blocks=1, attention_levels=[0], channel_mult=(1, 2),
                  num_heads=2, time_embed_dim=128)
    with pytest.raises(ValueError, match="192"):
        wide.set_attention_mode("softmax")
    UNet3D(latent_dim=4, model_channels=192, num_res_blocks=1, attention_levels=[0], channel_mult=(1, 2), num_heads=4,
           time_embed_dim=128).set_attention_mode("softmax")


def test_facade_reads_unet_attention_from_the_top_level_only():
    from v2v_b200.models import VideoToVideoDiffusion
    base = {"in_channels": 1, "latent_dim": 4, "vae_base_channels": 64, "unet_model_channels": 64,
            "unet_num_res_blocks": 1, "unet_attention_levels": [1], "unet_channel_mult": [1, 2], "unet_num_heads": 2,
            "unet_time_embed_dim": 128}
    assert VideoToVideoDiffusion(base).unet.attention_mode == "reference"
    m = VideoToVideoDiffusion(dict(base, unet_attention="softmax"))
    assert m.unet.attention_mode == "softmax"
    # like every other unet_* key, a value under config['model'] is not read
    nested = dict(base, model={"unet_attention": "softmax"})
    assert VideoToVideoDiffusion(nested).unet.attention_mode == "reference"
    with pytest.raises(ValueError):
        VideoToVideoDiffusion(dict(base, unet_attention="linear"))
    # a checkpoint {'model_state_dict', 'config'} carries the mode in its config
    ckpt = {"model_state_dict": m.state_dict(), "config": m.config}
    m2 = VideoToVideoDiffusion(ckpt["config"])
    m2.load_state_dict(ckpt["model_state_dict"], strict=True)
    assert m2.unet.attention_mode == "softmax" and sd_hash(m2.state_dict()) == sd_hash(m.state_dict())


def test_c_abi_declares_the_attention_entries():
    from v2v_b200 import _lib
    assert "b2v_unet_set_attention" in _lib.SIGNATURES and "b2v_temporal_attention" in _lib.SIGNATURES
    L = _lib.lib()
    assert L.b2v_abi_version() == 2
    assert L.b2v_unet_set_attention(None, 1) != 0 and "null" in _lib.last_error()
