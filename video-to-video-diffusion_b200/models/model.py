"""Mirror of the reference `models/model.py` facade: `VideoToVideoDiffusion(config)` resolves the config the way
the reference does (including reading the U-Net keys from the top level of the dict only), exposes `.vae`, `.unet`,
`.diffusion` under the same names so reference checkpoints load, and `generate()` runs
encode -> depth upsample -> DDIM/DDPM (or DPM-Solver++(2M), not in the reference) -> decode entirely on libb2v.so.  Training (`forward`, `save_checkpoint`)
is out of scope of this package.
"""
import ctypes

import numpy as np
import torch
import torch.nn as nn

from .. import _lib, ops
from .diffusion import GaussianDiffusion, ddpm_noise_budget_bytes
from .unet3d import UNet3D
from .vae import VideoVAE


def _guard(x):
    """the reference replaces non-finite values (nan->0, +inf->1, -inf->-1) when any are present; doing it
    unconditionally is identical on finite data and needs no host sync"""
    return torch.nan_to_num(x, nan=0.0, posinf=1.0, neginf=-1.0)


class VideoToVideoDiffusion(nn.Module):
    def __init__(self, config, load_pretrained=False):
        super().__init__()
        pre = config.get("pretrained", {})
        use_pretrained = pre.get("use_pretrained", False) or load_pretrained
        ckpt = config.get("hardware", {}).get("gradient_checkpointing", config.get("gradient_checkpointing", False))
        vae_cfg = pre.get("vae", {}) if use_pretrained else {}
        mc = config.get("model", config)

        def pick(key, default):
            return mc.get(key, config.get(key, default))

        if vae_cfg.get("enabled", False):
            if vae_cfg.get("checkpoint_path"):
                defaults = (1, 128, 8, 1.0)  # custom-VAE defaults (reference models/model.py:59-62)
            elif vae_cfg.get("model_name"):
                VideoVAE.from_pretrained(vae_cfg["model_name"])  # raises NotImplementedError, as the reference does
            else:
                raise ValueError("VAE enabled but neither checkpoint_path nor model_name specified in config")
        else:
            defaults = (3, 64, 4, 0.18215)  # from-scratch defaults (reference models/model.py:87-90)
        self.vae = VideoVAE(in_channels=pick("in_channels", defaults[0]), latent_dim=pick("latent_dim", defaults[2]),
                            base_channels=pick("vae_base_channels", defaults[1]),
                            scaling_factor=pick("vae_scaling_factor", defaults[3]), gradient_checkpointing=ckpt)
        # NB: like the reference, the U-Net / diffusion keys are looked up at the TOP level of `config` only
        self.unet = UNet3D(latent_dim=self.vae.latent_dim, model_channels=config.get("unet_model_channels", 128),
                           num_res_blocks=config.get("unet_num_res_blocks", 2),
                           attention_levels=config.get("unet_attention_levels", [1, 2]),
                           channel_mult=tuple(config.get("unet_channel_mult", [1, 2, 4, 4])),
                           num_heads=config.get("unet_num_heads", 4),
                           time_embed_dim=config.get("unet_time_embed_dim", 512), use_checkpoint=ckpt)
        # not a reference key: "softmax" runs checkpoints trained with the corrected attention contraction
        self.unet.set_attention_mode(config.get("unet_attention", "reference"))
        self.diffusion = GaussianDiffusion(noise_schedule=config.get("noise_schedule", "cosine"),
                                           timesteps=config.get("diffusion_timesteps", 1000),
                                           beta_start=config.get("beta_start", 0.0001),
                                           beta_end=config.get("beta_end", 0.02))
        self.config = config
        self.use_pretrained = use_pretrained

    def encode_videos(self, v_in, v_gt=None):
        z_in = self.vae.encode(v_in)
        return (z_in, self.vae.encode(v_gt)) if v_gt is not None else z_in

    def decode_latent(self, z):
        return self.vae.decode(z)

    def forward(self, v_in, v_gt, mask=None):
        raise NotImplementedError("training forward is out of scope of the B200 sampling package; "
                                  "use the reference implementation for training")

    @torch.no_grad()
    def generate(self, v_in, sampler, num_inference_steps=20, guidance_scale=1.0, target_depth=None):
        """thick slices (B,C,T_in,H,W) -> thin slices (B,C,T_out,H,W), fp32, tanh-bounded.  `guidance_scale` is
        accepted and ignored, exactly like the reference.  Besides the reference's "ddim" / "ddpm", `sampler` may be
        "dpmpp_2m" or "dpmpp_2m_sde" (DPM-Solver++(2M), ODE / SDE: num_inference_steps as for DDIM)."""
        if sampler not in ("ddpm", "ddim", "dpmpp_2m", "dpmpp_2m_sde"):
            raise ValueError(f"Unknown sampler: {sampler}")
        device = v_in.device
        B, C, T_in, H, W = v_in.shape
        T_out = int(target_depth) if target_depth is not None else T_in
        if v_in.numel() == 0:  # empty batch
            return torch.empty((B, C, T_out, H, W), dtype=torch.float32, device=device)
        if not v_in.is_cuda:
            raise RuntimeError(f"generate: input is on {device}; this implementation runs on B200 only (no CPU fallback)")
        if C != self.vae.in_channels or H % 4 or W % 4:
            raise ValueError(f"generate: v_in {tuple(v_in.shape)} needs {self.vae.in_channels} channels and H, W % 4 == 0")
        v_in = v_in.detach().float().contiguous()
        shape = (B, self.vae.latent_dim, T_out, H // 4, W // 4)
        n_lat = int(np.prod(shape))
        n = self.diffusion.timesteps
        if sampler == "ddpm" and n * n_lat * 4 > ddpm_noise_budget_bytes():
            return self._generate_staged(v_in, shape, target_depth)  # per-step noise does not fit: chunked loop
        # RNG order of the reference: a discarded randn(latent_shape) (models/model.py:303), the sampler's initial
        # draw, then (DDPM, DPM-Solver++ SDE) one randn_like per step
        torch.randn(shape, device=device)
        z_init = torch.randn(shape, device=device)
        cfg = _lib.SamplerCfg()
        keep = []  # host tables must outlive the call
        if sampler != "ddpm":
            from ..inference.sampler import _schedule
            ts, acp = _schedule(self.diffusion, num_inference_steps)
            keep += [ts, acp]
            code = {"ddim": 0, "dpmpp_2m": 2, "dpmpp_2m_sde": 3}[sampler]
            cfg.sampler, cfg.n, cfg.n_train, cfg.eta = code, len(ts), acp.numel(), 0.0
            cfg.timesteps = ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
            cfg.alphas_cumprod = ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float))
            if sampler == "dpmpp_2m_sde":
                noise = torch.stack([torch.randn_like(z_init) for _ in range(len(ts))]).contiguous()
                keep.append(noise)
                cfg.noise = noise.data_ptr()
        else:
            rows = self.diffusion.ddpm_coefficients()
            noise = torch.empty((n,) + shape, dtype=torch.float32, device=device)
            for s in range(n):
                noise[s] = torch.randn_like(z_init)
            keep += [rows, noise]
            cfg.sampler, cfg.n = 1, n
            cfg.ddpm_coef = ctypes.cast(rows.data_ptr(), ctypes.POINTER(ctypes.c_float))
            cfg.noise = noise.data_ptr()
        out = torch.empty((B, C, T_out, H, W), dtype=torch.float32, device=device)
        flag = torch.zeros(1, dtype=torch.int32, device=device)
        with torch.cuda.device(device):
            _lib.check(_lib.lib().b2v_generate(self.unet.native(device), self.vae.native(device), ctypes.byref(cfg),
                                               _lib.dptr(v_in), _lib.dptr(z_init), _lib.dptr(out), B, T_in, T_out, H, W,
                                               _lib.dptr(flag, torch.int32), _lib.stream()), "generate")
        self.last_nan_flag = flag  # device tensor: .item() it to learn whether one of the reference's NaN guards fired
        return out

    def _generate_staged(self, v_in, shape, target_depth):
        """generate() as separate C calls (encode / upsample / chunked DDPM loop / decode) for the case where the
        reference-ordered per-step noise of a DDPM run exceeds the staging budget"""
        device = v_in.device
        v_in = torch.nan_to_num(v_in, nan=0.0, posinf=float("inf"), neginf=float("-inf"))
        z_in = _guard(self.vae.encode(v_in))
        cond = _guard(ops.upsample_depth(z_in, int(target_depth))) if target_depth is not None else z_in
        torch.randn(shape, device=device)
        z0 = self.diffusion.p_sample_loop(self.unet, shape, cond, device, progress=True)
        return _guard(self.vae.decode(_guard(z0)))

    def count_parameters(self):
        n = lambda m, trainable=False: sum(p.numel() for p in m.parameters() if p.requires_grad or not trainable)  # noqa: E731
        return {"total": n(self), "trainable": n(self, True), "vae": n(self.vae), "vae_trainable": n(self.vae, True),
                "unet": n(self.unet, True), "diffusion": 0}
