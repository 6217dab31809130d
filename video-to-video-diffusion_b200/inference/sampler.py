"""Mirror of the reference `inference/sampler.py`: `DDIMSampler` / `DDPMSampler` with the reference's
constructor and `sample(...)` signatures, timestep subset, RNG consumption order and update formulas.
With a native UNet3D the whole DDIM loop is ONE call (b2v_ddim_sample): per step one CUDA-graph replay of the
U-Net plus the fused x0-prediction / clamp / re-noise kernel, no host synchronisation; the reference's five
per-step NaN checks become an on-device flag that is reported once after the loop.
"""
import ctypes
import logging
from typing import Tuple

import numpy as np
import torch

from .. import _lib, ops
from ..models._native import check_sampler_args

logger = logging.getLogger(__name__)


def _is_native(model):
    from ..models.unet3d import UNet3D
    return isinstance(model, UNet3D)


def _gaussian_weight(d, h, w):
    """separable Gaussian blending window, sigma = size / 6 (reference inference/sampler.py:455-479)"""
    def g(n):
        x = torch.arange(n).float() - (n - 1) / 2
        return torch.exp(-(x ** 2) / (2 * (n / 6) ** 2))
    return g(d)[:, None, None] * g(h)[None, :, None] * g(w)[None, None, :]


def _timesteps(n_train, num_inference_steps):
    """every (T // n)-th training step, plus T-1 if the stride missed it, descending: n (+1) evaluations"""
    ts = np.arange(0, n_train, n_train // num_inference_steps)
    if ts[-1] != n_train - 1:
        ts = np.append(ts, n_train - 1)
    return ts[::-1]


def _schedule(diffusion, num_inference_steps):
    """(timesteps, alphas_cumprod) of a DDIM / DPM-Solver++ loop: contiguous int64 array, fp32 CPU tensor"""
    ts = np.ascontiguousarray(_timesteps(diffusion.timesteps, num_inference_steps), dtype=np.int64)
    return ts, diffusion.alphas_cumprod.detach().float().cpu().contiguous()


def _native_sample(smp, entry, shape, conditioning, device, ts, acp, args, draw_noise, takes_noise=True):
    """the whole loop as one call of b2v_<entry> on a native UNet3D; RNG order: z, then one randn_like per step if
    draw_noise.  args are the entry's own arguments between n_train and noise (nan_flag when not takes_noise)."""
    shape, dev = check_sampler_args(smp.model, shape, conditioning, device)  # ValueError before any C call
    z = torch.randn(shape, device=dev)
    cond = conditioning.detach().to(dev, torch.float32).contiguous()
    B, _, T, h, w = shape
    if z.numel() == 0:
        return z
    n = len(ts)
    noise = torch.stack([torch.randn_like(z) for _ in range(n)]).contiguous() if draw_noise else None
    out = torch.empty_like(z)
    flag = torch.zeros(1, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _lib.check(getattr(_lib.lib(), "b2v_" + entry)(
            smp.model.native(dev), _lib.dptr(z), _lib.dptr(cond), _lib.dptr(out), B, T, h, w,
            ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), n,
            ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float)), acp.numel(), *args,
            *((_lib.dptr(noise),) if takes_noise else ()), _lib.dptr(flag, torch.int32), _lib.stream()), entry)
    smp.last_nan_flag = flag  # device tensor; .item() it to learn whether a NaN/Inf guard fired
    return out


def _starts(full, size, stride):
    return sorted(set(list(range(0, full - size + 1, stride)) + [max(0, full - size)]))


class _Stitching:
    """sliding-window inference shared by both samplers (reference inference/sampler.py:63-198, 338-453).
    Like the reference it encodes each thick patch, samples at the patch's own latent depth and decodes, so it
    requires patch depth == target depth (the reference raises a shape error otherwise; so does this)."""

    def _stitch(self, v_full, vae, sample_fn, patch_size, target_patch_size, stride, device):
        B, C, D, H, W = v_full.shape
        (pd, ph, pw), (td, th, tw), (sd_, sh, sw) = patch_size, target_patch_size, stride
        ratio = td / pd
        out = torch.zeros(B, C, int(D * ratio), H, W, device=device)
        wsum = torch.zeros_like(out)
        win = tuple(ops.gaussian_window_1d(n, out.device) for n in (td, th, tw))
        for d0 in _starts(D, pd, sd_):
            for h0 in _starts(H, ph, sh):
                for w0 in _starts(W, pw, sw):
                    z_c = vae.encode(v_full[:, :, d0:d0 + pd, h0:h0 + ph, w0:w0 + pw].contiguous())
                    v = vae.decode(sample_fn(tuple(z_c.shape), z_c))
                    if tuple(v.shape[2:]) != (td, th, tw):  # the reference fails here too (broadcast error, F7)
                        raise RuntimeError(f"decoded patch {tuple(v.shape[2:])} does not match target_patch_size "
                                           f"{(td, th, tw)}; use v2v_b200.inference.volume.generate_volume for "
                                           "thick->thin stitching with the depth upsample")
                    ops.stitch_accumulate(v, out, wsum, int(d0 * ratio), h0, w0, win)
        return ops.stitch_normalize(out, wsum)

    def _create_gaussian_weight(self, d, h, w):
        return _gaussian_weight(d, h, w)


class DDPMSampler(_Stitching):
    def __init__(self, diffusion, model):
        self.diffusion, self.model, self.timesteps = diffusion, model, diffusion.timesteps

    @torch.no_grad()
    def sample(self, shape, conditioning, device, progress=True):
        return self.diffusion.p_sample_loop(self.model, shape, conditioning, device, progress=progress)

    @torch.no_grad()
    def sample_with_stitching(self, v_thick_full, vae, patch_size: Tuple[int, int, int] = (8, 192, 192),
                              target_patch_size: Tuple[int, int, int] = (48, 192, 192),
                              stride: Tuple[int, int, int] = (4, 96, 96), device="cuda", progress=True):
        return self._stitch(v_thick_full, vae, lambda s, c: self.sample(s, c, device, progress=False), patch_size,
                            target_patch_size, stride, device)


class DDIMSampler(_Stitching):
    def __init__(self, diffusion, model):
        self.diffusion, self.model, self.timesteps = diffusion, model, diffusion.timesteps

    def _get_timesteps(self, num_inference_steps):
        return _timesteps(self.timesteps, num_inference_steps)

    @torch.no_grad()
    def sample(self, shape, conditioning, num_inference_steps, device, eta=0.0, progress=True):
        ts, acp = _schedule(self.diffusion, num_inference_steps)
        if not _is_native(self.model):
            dev = torch.device(device)
            z = torch.randn(shape, device=dev)
            return self._sample_generic(z, conditioning.detach().to(dev, torch.float32).contiguous(), ts, acp, eta)
        # the reference draws one randn_like per step when eta > 0; nothing else touches the RNG in between
        return _native_sample(self, "ddim_sample", shape, conditioning, device, ts, acp, (float(eta),), eta > 0)

    def _sample_generic(self, z, cond, ts, acp, eta):
        """any callable model(z, t, c): Python loop, fused update kernel per step"""
        dev = z.device
        for i, t_idx in enumerate(ts):
            t = torch.full((z.shape[0],), int(t_idx), device=dev, dtype=torch.long)
            eps = self.model(z, t, cond).float().contiguous()
            a_t = acp[int(t_idx)]
            a_prev = acp[int(ts[i + 1])] if i < len(ts) - 1 else torch.tensor(1.0)
            coef = torch.zeros(8)
            coef[0] = torch.sqrt(1 - a_t + 1e-8)
            coef[1] = torch.sqrt(a_t + 1e-8) + 1e-8
            coef[2] = torch.sqrt(a_prev + 1e-8)
            coef[3] = torch.sqrt(1 - a_prev + 1e-8)
            noise = None
            if eta > 0:
                coef[4] = eta * torch.sqrt((1 - a_prev + 1e-8) / (1 - a_t + 1e-8) * (1 - a_t / (a_prev + 1e-8)))
                noise = torch.randn_like(z)
            ops.ddim_update(z, eps, coef.to(dev), noise)
        return z

    @torch.no_grad()
    def sample_with_stitching(self, v_thick_full, vae, num_inference_steps: int = 20,
                              patch_size: Tuple[int, int, int] = (8, 192, 192),
                              target_patch_size: Tuple[int, int, int] = (48, 192, 192),
                              stride: Tuple[int, int, int] = (4, 96, 96), device="cuda", eta: float = 0.0,
                              progress=True):
        return self._stitch(v_thick_full, vae,
                            lambda s, c: self.sample(s, c, num_inference_steps, device, eta=eta, progress=False),
                            patch_size, target_patch_size, stride, device)


def dpmpp_coefficients(timesteps, alphas_cumprod, order=2, stochastic=False):
    """the (n, 8) fp32 rows {sigma_t, alpha_t, a, b, w0, w1, c, clip} of a DPM-Solver++(2M) loop over `timesteps`
    (strictly decreasing), computed in fp64 by b2v_dpmpp_coefficients (host only, no device needed)"""
    ts = np.ascontiguousarray(timesteps, dtype=np.int64)
    acp = alphas_cumprod.detach().float().cpu().contiguous()
    rows = torch.empty((len(ts), 8), dtype=torch.float32)
    _lib.check(_lib.lib().b2v_dpmpp_coefficients(
        ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), len(ts), ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float)),
        acp.numel(), int(order), int(bool(stochastic)), ctypes.cast(rows.data_ptr(), ctypes.POINTER(ctypes.c_float))),
        "dpmpp_coefficients")
    return rows


class DPMSolverSampler(_Stitching):
    """DPM-Solver++(2M) (Lu et al. 2022), not in the reference: a second-order multistep solver over the same
    eps-prediction U-Net, one evaluation per step like DDIM, over DDIMSampler's timestep subset (so
    `num_inference_steps` means the same number of evaluations).  stochastic=True is the 2M SDE form.  With a native
    UNet3D the whole loop is one call (b2v_dpmpp_sample); any other callable model runs a Python loop over the same
    update kernel.  RNG order: z = randn(shape), then (SDE only) one randn_like per step."""

    def __init__(self, diffusion, model):
        self.diffusion, self.model, self.timesteps = diffusion, model, diffusion.timesteps

    def _get_timesteps(self, num_inference_steps):
        return _timesteps(self.timesteps, num_inference_steps)

    @torch.no_grad()
    def sample(self, shape, conditioning, num_inference_steps, device, order=2, stochastic=False, progress=True):
        if order not in (1, 2):
            raise ValueError(f"DPMSolverSampler: order must be 1 or 2, got {order}")
        ts, acp = _schedule(self.diffusion, num_inference_steps)
        if _is_native(self.model):
            return _native_sample(self, "dpmpp_sample", shape, conditioning, device, ts, acp,
                                  (int(order), int(stochastic)), stochastic)
        dev = torch.device(device)
        z = torch.randn(shape, device=dev)
        cond = conditioning.detach().to(dev, torch.float32).contiguous()
        if z.numel() == 0:
            return z
        noise = torch.stack([torch.randn_like(z) for _ in range(len(ts))]).contiguous() if stochastic else None
        return self._sample_generic(z, cond, ts, dpmpp_coefficients(ts, acp, order, stochastic).to(dev), noise)

    def _sample_generic(self, z, cond, ts, rows, noise):
        """any callable model(z, t, c): Python loop, the update kernel per step (in place on z)"""
        dev = z.device
        x0_prev = torch.empty_like(z)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        for i, t_idx in enumerate(ts):
            t = torch.full((z.shape[0],), int(t_idx), device=dev, dtype=torch.long)
            eps = self.model(z, t, cond).float().contiguous()
            flag |= ops.dpmpp_update(z, x0_prev, eps, rows[i].contiguous(), None if noise is None else noise[i])
        self.last_nan_flag = flag
        return z

    @torch.no_grad()
    def sample_with_stitching(self, v_thick_full, vae, num_inference_steps: int = 20,
                              patch_size: Tuple[int, int, int] = (8, 192, 192),
                              target_patch_size: Tuple[int, int, int] = (48, 192, 192),
                              stride: Tuple[int, int, int] = (4, 96, 96), device="cuda", order=2, stochastic=False,
                              progress=True):
        return self._stitch(v_thick_full, vae,
                            lambda s, c: self.sample(s, c, num_inference_steps, device, order=order,
                                                     stochastic=stochastic, progress=False),
                            patch_size, target_patch_size, stride, device)


UNIPC_VARIANTS = {"bh1": 0, "bh2": 1}


def unipc_coefficients(timesteps, alphas_cumprod, order=3, variant="bh2"):
    """the (n, 16) fp32 rows {sigma, alpha, g, a_c, c0..c3, a_p, p0..p2, clip, 0, 0, 0} of a UniPC loop over `timesteps`
    (strictly decreasing), computed in fp64 by b2v_unipc_coefficients (host only, no device needed)"""
    if variant not in UNIPC_VARIANTS:
        raise ValueError(f"unipc_coefficients: variant must be 'bh1' or 'bh2', got {variant!r}")
    ts = np.ascontiguousarray(timesteps, dtype=np.int64)
    acp = alphas_cumprod.detach().float().cpu().contiguous()
    rows = torch.empty((len(ts), 16), dtype=torch.float32)
    _lib.check(_lib.lib().b2v_unipc_coefficients(
        ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), len(ts), ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float)),
        acp.numel(), int(order), UNIPC_VARIANTS[variant], ctypes.cast(rows.data_ptr(), ctypes.POINTER(ctypes.c_float))),
        "unipc_coefficients")
    return rows


class UniPCSampler(_Stitching):
    """UniPC (Zhao et al. 2023), not in the reference: a predictor-corrector multistep solver over the same
    eps-prediction U-Net.  The corrector reuses the evaluation the next step needs anyway, so a predictor of order p
    becomes a solver of order p + 1 at one U-Net evaluation per step, like DDIM, over DDIMSampler's timestep subset.
    order 3 with variant "bh2" (the default, and generate(sampler="unipc")) is the choice for guidance-free sampling from
    about 10 steps up; below 10 steps order=1 is more accurate.  With a native UNet3D the whole loop is one call
    (b2v_unipc_sample); any other callable model runs a Python loop over the same update kernel.  RNG order: z =
    randn(shape), nothing else (deterministic solver)."""

    def __init__(self, diffusion, model):
        self.diffusion, self.model, self.timesteps = diffusion, model, diffusion.timesteps

    def _get_timesteps(self, num_inference_steps):
        return _timesteps(self.timesteps, num_inference_steps)

    @torch.no_grad()
    def sample(self, shape, conditioning, num_inference_steps, device, order=3, variant="bh2", progress=True):
        if order not in (1, 2, 3):
            raise ValueError(f"UniPCSampler: order must be 1, 2 or 3, got {order}")
        if variant not in UNIPC_VARIANTS:
            raise ValueError(f"UniPCSampler: variant must be 'bh1' or 'bh2', got {variant!r}")
        ts, acp = _schedule(self.diffusion, num_inference_steps)
        if _is_native(self.model):
            return _native_sample(self, "unipc_sample", shape, conditioning, device, ts, acp,
                                  (int(order), UNIPC_VARIANTS[variant]), False, takes_noise=False)
        dev = torch.device(device)
        z = torch.randn(shape, device=dev)
        cond = conditioning.detach().to(dev, torch.float32).contiguous()
        if z.numel() == 0:
            return z
        return self._sample_generic(z, cond, ts, unipc_coefficients(ts, acp, order, variant).to(dev))

    def _sample_generic(self, z, cond, ts, rows):
        """any callable model(z, t, c): Python loop, the update kernel per step (in place on z)"""
        dev = z.device
        xc = torch.empty_like(z)
        hist = torch.empty((4,) + tuple(z.shape), dtype=torch.float32, device=dev)
        flag = torch.zeros(1, dtype=torch.int32, device=dev)
        for i, t_idx in enumerate(ts):
            t = torch.full((z.shape[0],), int(t_idx), device=dev, dtype=torch.long)
            eps = self.model(z, t, cond).float().contiguous()
            flag |= ops.unipc_update(z, xc, hist, eps, rows[i].contiguous(), i)
        self.last_nan_flag = flag
        return z

    @torch.no_grad()
    def sample_with_stitching(self, v_thick_full, vae, num_inference_steps: int = 20,
                              patch_size: Tuple[int, int, int] = (8, 192, 192),
                              target_patch_size: Tuple[int, int, int] = (48, 192, 192),
                              stride: Tuple[int, int, int] = (4, 96, 96), device="cuda", order=3, variant="bh2",
                              progress=True):
        return self._stitch(v_thick_full, vae,
                            lambda s, c: self.sample(s, c, num_inference_steps, device, order=order, variant=variant,
                                                     progress=False),
                            patch_size, target_patch_size, stride, device)


class EDMSampler:
    def __init__(self, diffusion, model):
        raise NotImplementedError("EDM sampler not yet implemented")  # same as the reference (:482-493)
