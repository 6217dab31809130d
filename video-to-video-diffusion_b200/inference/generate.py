"""Mirror of the tensor-level helper of the reference `inference/generate.py` (generate_batch, :98-155).
The file-level helpers of the reference (mp4 decode/encode through cv2 / PyAV) are data I/O and out of scope.
Besides the reference's "ddim" / "ddpm", sampler_type accepts "dpmpp_2m" and "dpmpp_2m_sde" (DPMSolverSampler)."""
import torch

from .sampler import DDIMSampler, DDPMSampler, DPMSolverSampler


def generate_batch(model, input_videos, sampler_type="ddim", num_inference_steps=20, device="cuda"):
    """encode -> sample at the input's own latent depth -> decode, for a batch (B, C, T, H, W)"""
    model.eval()
    model.to(device)
    input_videos = input_videos.to(device)
    with torch.no_grad():
        z_in = model.vae.encode(input_videos)
    if sampler_type == "ddim":
        z_0 = DDIMSampler(model.diffusion, model.unet).sample(z_in.shape, z_in, num_inference_steps, device,
                                                               progress=True)
    elif sampler_type == "ddpm":
        z_0 = DDPMSampler(model.diffusion, model.unet).sample(z_in.shape, z_in, device, progress=True)
    elif sampler_type in ("dpmpp_2m", "dpmpp_2m_sde"):
        z_0 = DPMSolverSampler(model.diffusion, model.unet).sample(z_in.shape, z_in, num_inference_steps, device,
                                                                    stochastic=sampler_type == "dpmpp_2m_sde",
                                                                    progress=True)
    else:
        raise ValueError(f"Unknown sampler type: {sampler_type}")
    with torch.no_grad():
        return model.vae.decode(z_0)
