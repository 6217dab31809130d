"""fp32/fp64 restatement of the U-Net with softmax temporal attention: the reference's TemporalAttention
(models/unet3d.py:163-194) with its second contraction corrected to 'bhqk,bhkc->bhqc', i.e. attn @ V.  Everything
else is oracle/ref_port.py's unet_forward, composed from the same helpers; test infrastructure only."""
import torch
import torch.nn.functional as F

from oracle import ref_port as R


def unet_attention_softmax(sd, p, x, heads):
    """x + proj_out(softmax(q k^T / sqrt(hd)) v) over the T depth tokens of each (b, h, w, head)"""
    B, C, T, H, W = x.shape
    hd = C // heads
    qkv = R._conv(sd, p + ".qkv", R._gn(sd, p + ".norm", x, R.num_groups(C)))
    q, k, v = qkv[:, :C], qkv[:, C:2 * C], qkv[:, 2 * C:]

    def seq(a):  # (B, heads*hd, T, H, W) -> (B*H*W, heads, T, hd)
        return a.reshape(B, heads, hd, T, H, W).permute(0, 4, 5, 1, 3, 2).reshape(B * H * W, heads, T, hd)

    q, k, v = seq(q), seq(k), seq(v)
    attn = torch.softmax(torch.matmul(q, k.transpose(-1, -2)) * hd ** -0.5, dim=-1)
    out = torch.matmul(attn, v)  # (N, heads, T, hd)
    out = out.reshape(B, H, W, heads, T, hd).permute(0, 3, 5, 4, 1, 2).reshape(B, C, T, H, W)
    return R._conv(sd, p + ".proj_out", out) + x


def unet_forward(sd, cfg, x, t, c, prefix=""):
    """R.unet_forward with every TemporalAttention in softmax form (same cfg keys)"""
    P = prefix
    mult = tuple(cfg["channel_mult"])
    nl, nres, heads = len(mult), cfg["num_res_blocks"], cfg["num_heads"]
    att = set(cfg["attention_levels"])
    temb = R.time_embedding(sd, P + "time_embed", t, cfg["model_channels"])
    h = R._conv(sd, P + "conv_in", torch.cat([x, c], dim=1), padding=1)
    skips = []
    for lv in range(nl):
        for i in range(nres):
            h = R.unet_resblock(sd, f"{P}down_blocks.{lv}.{i}.0", h, temb)
            if lv in att:
                h = unet_attention_softmax(sd, f"{P}down_blocks.{lv}.{i}.1", h, heads)
        skips.append(h)
        if lv < nl - 1:
            h = R._conv(sd, f"{P}down_samples.{lv}.conv", h, stride=(1, 2, 2), padding=1)
    h = R.unet_resblock(sd, P + "mid_block1", h, temb)
    h = unet_attention_softmax(sd, P + "mid_attn", h, heads)
    h = R.unet_resblock(sd, P + "mid_block2", h, temb)
    for j in range(nl):
        lv = nl - 1 - j
        for i in range(nres + 1):
            if i == 0:
                h = torch.cat([h, skips.pop()], dim=1)
            h = R.unet_resblock(sd, f"{P}up_blocks.{j}.{i}.0", h, temb)
            if lv in att:
                h = unet_attention_softmax(sd, f"{P}up_blocks.{j}.{i}.1", h, heads)
        if j < nl - 1:
            h = F.conv_transpose3d(h, sd[f"{P}up_samples.{j}.conv.weight"], sd[f"{P}up_samples.{j}.conv.bias"],
                                   stride=(1, 2, 2), padding=1)
    C = h.shape[1]
    h = F.silu(R._gn(sd, P + "conv_out.0", h, R.num_groups(C)))
    return R._conv(sd, P + "conv_out.2", h, padding=1)
