"""Full-volume thick->thin inference: the sliding-window stitcher the reference intends
(`sample_with_stitching`, inference/sampler.py:338-453) *with* the depth upsample that only `generate()` has
(models/model.py:284-289) -- the reference's own stitcher raises for 8 -> 48 slices (SURVEY F7, section 8(f).1).

Every window is an independent work item (encode -> trilinear depth upsample -> DDIM/DDPM -> decode), so windows
are batched `batch` at a time on one GPU and sharded across ranks; blending (Gaussian window, sigma = size/6,
normalised by the summed weights) runs in the stitch kernels of libb2v.so.
"""
import torch

from .. import ops
from ..dist import patch_grid, shard_range
from .ensemble import generate_ensemble


def window_starts(D, H, W, patch_size=(8, 192, 192), stride=(4, 96, 96)):
    """window origins in reference order (d outermost, then h, then w)"""
    (pd, ph, pw), (sd, sh, sw) = patch_size, stride
    return [(d0, h0, w0) for d0 in patch_grid(D, pd, sd) for h0 in patch_grid(H, ph, sh) for w0 in patch_grid(W, pw, sw)]


@torch.no_grad()
def generate_volume(model, v_thick_full, sampler="ddim", num_inference_steps=20, patch_size=(8, 192, 192),
                    target_patch_size=(48, 192, 192), stride=(4, 96, 96), batch=4, rank=0, world=1,
                    num_samples=None):
    """v_thick_full (B, C, D_thick, H, W) on the GPU -> (B, C, D_thick * ratio, H, W).
    With world > 1 each rank processes a contiguous shard of the (volume, window) items and returns its PARTIAL
    (accumulator, weight-sum) pair un-normalised so the caller can all-reduce / gather; world == 1 returns the
    normalised volume.
    num_samples = K (an int >= 2): every window batch runs inference.ensemble.generate_ensemble and the result is
    (mean, std) volumes.  The mean is blended like the single-sample volume; the std volume is the weighted blend of
    the per-window std maps with the same Gaussian weights (not the std of a blended sample).  With world > 1 the
    partials are (acc_mean, acc_std, wsum)."""
    Bv, C, D, H, W = v_thick_full.shape
    pd, ph, pw = patch_size
    td, th, tw = target_patch_size
    ratio = td / pd
    dev = v_thick_full.device
    acc = torch.zeros((Bv, C, int(D * ratio), H, W), dtype=torch.float32, device=dev)
    wsum = torch.zeros_like(acc)
    acc_std = None if num_samples is None else torch.zeros_like(acc)
    win = tuple(ops.gaussian_window_1d(n, dev) for n in (td, th, tw))
    items = [(b, s) for b in range(Bv) for s in window_starts(D, H, W, patch_size, stride)]
    lo, hi = shard_range(len(items), rank, world)
    for i in range(lo, hi, batch):
        chunk = items[i:min(i + batch, hi)]
        x = torch.stack([v_thick_full[b, :, d0:d0 + pd, h0:h0 + ph, w0:w0 + pw] for b, (d0, h0, w0) in chunk])
        if num_samples is None:
            v = model.generate(x.contiguous(), sampler, num_inference_steps, target_depth=td)
        else:
            v, sd = generate_ensemble(model, x.contiguous(), sampler, num_inference_steps, num_samples, target_depth=td)
        for j, (b, (d0, h0, w0)) in enumerate(chunk):  # windows of one batch may overlap: accumulate one at a time
            ops.stitch_accumulate(v[j:j + 1], acc[b:b + 1], wsum[b:b + 1], int(d0 * ratio), h0, w0, win)
            if acc_std is not None:  # same weights, already summed into wsum above
                ops.stitch_accumulate(sd[j:j + 1], acc_std[b:b + 1], None, int(d0 * ratio), h0, w0, win)
    if acc_std is None:
        return (acc, wsum) if world > 1 else ops.stitch_normalize(acc, wsum)
    if world > 1:
        return acc, acc_std, wsum
    return ops.stitch_normalize(acc, wsum), ops.stitch_normalize(acc_std, wsum)
