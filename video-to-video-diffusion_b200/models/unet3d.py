"""Mirror of the reference `models/unet3d.py` interface: `UNet3D(...)` with identical constructor arguments,
parameter names, creation order (so torch's default initialisers draw the same random numbers) and
`forward(x, t, c)` semantics.  The forward pass itself is one call into libb2v.so (b2v_unet_forward): tcgen05
implicit-GEMM convolutions, fused GroupNorm/SiLU/time-embedding/residual kernels, the reference's (degenerate)
temporal attention or, opt-in, softmax attention over depth, all replayed as a CUDA graph.  See csrc/unet.cu and DESIGN.md.
"""
import torch
import torch.nn as nn

from .. import _lib
from ._native import NativeHandle, ParamsOnly, require_cuda


def _groups(ch):  # reference _get_num_groups (models/unet3d.py:63-68)
    return next(g for g in (32, 16, 8, 4, 2, 1) if ch % g == 0)


class SinusoidalPositionEmbeddings(ParamsOnly):
    def __init__(self, dim):
        super().__init__()
        self.dim = dim


class TimeEmbedding(ParamsOnly):
    def __init__(self, dim, time_dim):
        super().__init__()
        self.time_mlp = nn.Sequential(SinusoidalPositionEmbeddings(dim), nn.Linear(dim, time_dim), nn.SiLU(),
                                      nn.Linear(time_dim, time_dim))


class Conv3DBlock(ParamsOnly):
    def __init__(self, in_channels, out_channels, kernel_size=3, stride=1, padding=1):
        super().__init__()
        self.conv = nn.Conv3d(in_channels, out_channels, kernel_size, stride, padding)
        self.norm = nn.GroupNorm(min(8, out_channels) if out_channels % 8 == 0 else _groups(out_channels), out_channels)
        self.act = nn.SiLU()


class ResBlock3D(ParamsOnly):
    def __init__(self, in_channels, out_channels, time_dim):
        super().__init__()
        self.conv1 = Conv3DBlock(in_channels, out_channels)
        self.time_mlp = nn.Sequential(nn.SiLU(), nn.Linear(time_dim, out_channels))
        self.conv2 = nn.Sequential(nn.Conv3d(out_channels, out_channels, kernel_size=3, padding=1),
                                   nn.GroupNorm(_groups(out_channels), out_channels))
        self.residual_conv = (nn.Conv3d(in_channels, out_channels, kernel_size=1)
                              if in_channels != out_channels else nn.Identity())
        self.act = nn.SiLU()


class TemporalAttention(ParamsOnly):
    def __init__(self, channels, num_heads=4):
        super().__init__()
        assert channels % num_heads == 0, "channels must be divisible by num_heads"
        self.num_heads, self.channels, self.head_dim = num_heads, channels, channels // num_heads
        self.norm = nn.GroupNorm(_groups(channels), channels)
        self.qkv = nn.Conv3d(channels, channels * 3, kernel_size=1)
        self.proj_out = nn.Conv3d(channels, channels, kernel_size=1)


class Downsample3D(ParamsOnly):
    def __init__(self, in_channels, out_channels=None):
        super().__init__()
        self.conv = nn.Conv3d(in_channels, out_channels or in_channels, (3, 4, 4), (1, 2, 2), (1, 1, 1))


class Upsample3D(ParamsOnly):
    def __init__(self, channels):
        super().__init__()
        self.conv = nn.ConvTranspose3d(channels, channels, (3, 4, 4), (1, 2, 2), (1, 1, 1))


ATTENTION_MODES = {"reference": 0, "softmax": 1}  # b2v_unet_set_attention codes


def softmax_head_dim_error(model_channels, channel_mult, attention_levels, num_heads):
    """why softmax attention cannot run for this configuration, or None: every attention level and the mid block need
    head_dim = channels / num_heads to be a multiple of 16 in [16, 128] (the fused attention kernel's tile shapes)"""
    nl = len(channel_mult)
    levels = sorted({int(lv) for lv in attention_levels if 0 <= int(lv) < nl} | {nl - 1})
    for lv in levels:
        C = model_channels * int(channel_mult[lv])
        if num_heads < 1 or C % num_heads:
            return f"{C} channels are not divisible by num_heads = {num_heads}"
        hd = C // num_heads
        if hd % 16 or not 16 <= hd <= 128:
            return (f"head_dim = {C} / {num_heads} = {hd} at {C} channels; softmax attention needs a multiple of 16 "
                    "in [16, 128]")
    return None


class UNet3D(nn.Module):
    """eps = UNet3D(...)(x, t, c) with x, c: (B, latent_dim, T, h, w) fp32 CUDA and t: (B,) int64.

    `attention_mode` selects what TemporalAttention computes: "reference" (default) follows the reference's
    'bhqk,bhvc->bhqc' contraction exactly (its output does not depend on q, k or the softmax); "softmax" is ordinary
    attention over the T depth tokens ('bhqk,bhkc->bhqc'), for checkpoints trained with that contraction.  The mode is
    not stored in the state_dict: set it with `set_attention_mode`."""

    def __init__(self, latent_dim=4, model_channels=128, num_res_blocks=2, attention_levels=[1, 2],
                 channel_mult=(1, 2, 4, 4), num_heads=4, time_embed_dim=512, use_checkpoint=False):
        super().__init__()
        self.latent_dim, self.model_channels, self.num_res_blocks = latent_dim, model_channels, num_res_blocks
        self.attention_levels, self.channel_mult = attention_levels, channel_mult
        self.num_levels, self.use_checkpoint = len(channel_mult), use_checkpoint
        self.num_heads, self.time_embed_dim = num_heads, time_embed_dim
        nl = self.num_levels
        # limits of the B200 kernels (DESIGN.md "known limits"), raised here rather than at the first forward
        if model_channels % 64:
            raise ValueError(f"UNet3D: model_channels = {model_channels} must be a multiple of 64 (64-channel K chunks "
                             "of the implicit-GEMM convolution)")
        if 2 * latent_dim * 3 > 64:
            raise ValueError(f"UNet3D: latent_dim = {latent_dim} too large for the packed conv_in (<= 10)")
        if not 1 <= nl <= 8 or num_res_blocks < 1:
            raise ValueError("UNet3D: 1..8 levels and at least one ResBlock per level")

        def stage(cin, cout, attn):
            layers = [ResBlock3D(cin, cout, time_embed_dim)]
            if attn:
                layers.append(TemporalAttention(cout, num_heads))
            return nn.ModuleList(layers)

        self.time_embed = TimeEmbedding(model_channels, time_embed_dim)
        self.conv_in = nn.Conv3d(latent_dim * 2, model_channels, kernel_size=3, padding=1)
        self.down_blocks, self.down_samples = nn.ModuleList(), nn.ModuleList()
        ch = model_channels
        for lv, m in enumerate(channel_mult):
            blocks = nn.ModuleList()
            for _ in range(num_res_blocks):
                blocks.append(stage(ch, model_channels * m, lv in attention_levels))
                ch = model_channels * m
            self.down_blocks.append(blocks)
            self.down_samples.append(Downsample3D(ch, ch) if lv < nl - 1 else nn.Identity())
        self.mid_block1 = ResBlock3D(ch, ch, time_embed_dim)
        self.mid_attn = TemporalAttention(ch, num_heads)
        self.mid_block2 = ResBlock3D(ch, ch, time_embed_dim)
        self.up_blocks, self.up_samples = nn.ModuleList(), nn.ModuleList()
        for j, m in enumerate(reversed(channel_mult)):
            lv = nl - 1 - j
            blocks = nn.ModuleList()
            for i in range(num_res_blocks + 1):
                cin = ch + model_channels * channel_mult[lv] if i == 0 else ch  # skip concat on the first block
                blocks.append(stage(cin, model_channels * m, lv in attention_levels))
                ch = model_channels * m
            self.up_blocks.append(blocks)
            self.up_samples.append(Upsample3D(ch) if j < nl - 1 else nn.Identity())
        self.conv_out = nn.Sequential(nn.GroupNorm(_groups(ch), ch), nn.SiLU(),
                                      nn.Conv3d(ch, latent_dim, kernel_size=3, padding=1))
        self._native = NativeHandle("unet")
        self.attention_mode = "reference"

    def set_attention_mode(self, mode):
        """"reference" | "softmax"; raises ValueError for another mode or a head_dim the softmax kernel cannot run"""
        if mode not in ATTENTION_MODES:
            raise ValueError(f"UNet3D: unknown attention mode {mode!r} (expected one of {sorted(ATTENTION_MODES)})")
        if mode == "softmax":
            why = softmax_head_dim_error(self.model_channels, self.channel_mult, self.attention_levels, self.num_heads)
            if why:
                raise ValueError(f"UNet3D: softmax attention is not supported here: {why}")
        self.attention_mode = mode
        return self

    # ---- native plumbing
    def _desc(self):
        d = _lib.UNetDesc()
        d.latent_dim, d.model_channels, d.num_res_blocks = self.latent_dim, self.model_channels, self.num_res_blocks
        d.num_levels = self.num_levels
        for i, m in enumerate(self.channel_mult):
            d.channel_mult[i] = int(m)
        d.attention_mask = sum(1 << int(lv) for lv in self.attention_levels if 0 <= int(lv) < self.num_levels)
        d.num_heads, d.time_embed_dim = self.num_heads, self.time_embed_dim
        return d

    def native(self, device):
        """the b2v_unet handle holding this module's current weights on `device`"""
        return self._native.get(self, self._desc(), device, ATTENTION_MODES[self.attention_mode])

    def invalidate_native(self):
        """call after changing weights in a way torch's version counters cannot see (writes through `.data`)"""
        self._native.invalidate()

    @torch.no_grad()
    def forward(self, x, t, c):
        x = require_cuda(x, "UNet3D.forward")
        c = require_cuda(c, "UNet3D.forward").to(x.device)
        t = t.to(device=x.device, dtype=torch.int64).contiguous()
        B, L, T, h, w = x.shape
        if c.shape != x.shape or t.shape != (B,) or L != self.latent_dim:
            raise ValueError(f"UNet3D.forward: x {tuple(x.shape)}, c {tuple(c.shape)}, t {tuple(t.shape)}")
        out = torch.empty_like(x)
        if x.numel() == 0:  # empty batch: nothing to launch
            return out
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().b2v_unet_forward(self.native(x.device), _lib.dptr(x), _lib.dptr(t, torch.int64),
                                                   _lib.dptr(c), _lib.dptr(out), B, T, h, w, _lib.stream()),
                       "unet_forward")
        return out
