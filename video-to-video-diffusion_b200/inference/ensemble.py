"""Ensemble generation (not in the reference): K samples of each input in one native call (b2v_generate_ensemble), with
the per-voxel mean and standard-deviation maps.  The spread of several samples of the same thick input shows where the
model's thin slices are uncertain, i.e. where plausible-looking structure may be invented.

Member m = k*B + b is sample k of input b (k-major): the B inputs are encoded and depth-upsampled once, the sampler runs
once at batch K*B on the conditioning repeated K times, and the members are decoded in K chunks of B.
"""
import ctypes

import torch

from .. import _lib

SAMPLERS = {"ddim": 0, "ddpm": 1, "dpmpp_2m": 2, "dpmpp_2m_sde": 3, "unipc": 4}


@torch.no_grad()
def generate_ensemble(model, v_in, sampler, num_inference_steps=20, num_samples=4, target_depth=None,
                      return_members=False):
    """thick slices v_in (B, C, T_in, H, W) -> (mean, std), each (B, C, T_out, H, W) fp32, over K = num_samples samples
    per input; std is the unbiased per-voxel standard deviation (like torch.std).  With return_members=True also the
    members (K, B, C, T_out, H, W).  sampler: "ddim" (eta = 0, as generate()), "ddpm", "dpmpp_2m", "dpmpp_2m_sde" or
    "unipc" (UniPC-3, bh2, as generate()).

    RNG order: z_init = torch.randn((K*B, L, T_out, H/4, W/4)); then for "dpmpp_2m_sde" one randn of that shape per step,
    for "ddpm" one seed = torch.randint(0, 2**62, ()) that keys the device Philox generator of the per-step noise.
    Sets model.last_nan_flag (device int32 tensor) like generate()."""
    K = int(num_samples)
    if K < 2:
        raise ValueError(f"generate_ensemble: num_samples must be >= 2 (the std needs two), got {num_samples}")
    if sampler not in SAMPLERS:
        raise ValueError(f"generate_ensemble: unknown sampler {sampler!r} (one of {', '.join(SAMPLERS)})")
    if v_in.dim() != 5:
        raise ValueError(f"generate_ensemble: v_in must be (B, C, T, H, W), got {tuple(v_in.shape)}")
    B, C, T_in, H, W = v_in.shape
    if C != model.vae.in_channels or H % 4 or W % 4:
        raise ValueError(f"generate_ensemble: v_in {tuple(v_in.shape)} needs {model.vae.in_channels} channels and "
                         "H, W % 4 == 0")
    device = v_in.device
    T_out = int(target_depth) if target_depth is not None else T_in
    out_shape = (B, C, T_out, H, W)
    if not v_in.is_cuda:
        raise RuntimeError(f"generate_ensemble: input is on {device}; this implementation runs on B200 only "
                           "(no CPU fallback)")
    members = torch.empty((K,) + out_shape, dtype=torch.float32, device=device) if return_members else None
    mean = torch.empty(out_shape, dtype=torch.float32, device=device)
    std = torch.empty_like(mean)
    if v_in.numel() == 0:
        return (mean, std, members) if return_members else (mean, std)
    v_in = v_in.detach().float().contiguous()
    shape = (K * B, model.vae.latent_dim, T_out, H // 4, W // 4)
    z_init = torch.randn(shape, device=device)
    cfg = _lib.SamplerCfg()
    cfg.sampler = SAMPLERS[sampler]
    keep = []  # host tables and the noise must outlive the call
    if sampler == "ddpm":
        rows = model.diffusion.ddpm_coefficients()
        keep.append(rows)
        cfg.n = model.diffusion.timesteps
        cfg.ddpm_coef = ctypes.cast(rows.data_ptr(), ctypes.POINTER(ctypes.c_float))
        cfg.seed = int(torch.randint(0, 2 ** 62, ()))
    else:
        from .sampler import _schedule
        ts, acp = _schedule(model.diffusion, num_inference_steps)
        keep += [ts, acp]
        cfg.n, cfg.n_train, cfg.eta = len(ts), acp.numel(), 0.0
        cfg.unipc_order, cfg.unipc_variant = 3, 1  # read only for "unipc"
        cfg.timesteps = ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
        cfg.alphas_cumprod = ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float))
        if sampler == "dpmpp_2m_sde":
            noise = torch.stack([torch.randn(shape, device=device) for _ in range(len(ts))]).contiguous()
            keep.append(noise)
            cfg.noise = noise.data_ptr()
    flag = torch.zeros(1, dtype=torch.int32, device=device)
    with torch.cuda.device(device):
        _lib.check(_lib.lib().b2v_generate_ensemble(
            model.unet.native(device), model.vae.native(device), ctypes.byref(cfg), _lib.dptr(v_in), _lib.dptr(z_init),
            K, _lib.dptr(members), _lib.dptr(mean), _lib.dptr(std), B, T_in, T_out, H, W, _lib.dptr(flag, torch.int32),
            _lib.stream()), "generate_ensemble")
    model.last_nan_flag = flag  # device tensor: .item() it to learn whether a NaN/Inf guard fired
    return (mean, std, members) if return_members else (mean, std)
