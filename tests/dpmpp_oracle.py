"""DPM-Solver++(2M) restated in torch straight from the paper, independently of libb2v's b2v_dpmpp_coefficients:
Lu et al. 2022, "DPM-Solver++: Fast Solver for Guided Sampling of Diffusion Probabilistic Models", Algorithm 2
(multistep second order, data prediction, lambda / h form) and the 2M SDE update (as in k-diffusion's
sample_dpmpp_2m_sde), for a VP model with eps prediction.  Runs in fp64 or fp32; test infrastructure only.

alpha_t = sqrt(acp_t), sigma_t = sqrt(1 - acp_t), lambda_t = log(alpha_t / sigma_t) from the fp32 table in fp64.
Step i goes from t_i to s = t_{i+1}; the last step goes to the clean sample (alpha = 1, sigma = 0): z' = x0.
"""
import math

import torch


def _schedule(acp, t):
    """(alpha, sigma, lambda) of timestep t in fp64; t = None is the clean sample"""
    if t is None:
        return 1.0, 0.0, math.inf
    a = float(acp[int(t)])
    alpha, sigma = math.sqrt(a), math.sqrt(1.0 - a)
    return alpha, sigma, math.log(alpha / sigma)


def coefficients(timesteps, acp, order=2, sde=False):
    """fp64 rows (sigma_t, alpha_t, a, b, w0, w1, c, clip) with z' = a z + b (w0 x0 + w1 x0_prev) + c xi"""
    ts = [int(t) for t in timesteps]
    n = len(ts)
    rows, h_prev = [], None
    for i, t in enumerate(ts):
        al_t, sg_t, lam_t = _schedule(acp, t)
        if i == n - 1:  # to the clean sample: sigma_s = 0 makes every noise term vanish
            rows.append((sg_t, al_t, 0.0, 1.0, 1.0, 0.0, 0.0, 10.0))
            break
        al_s, sg_s, lam_s = _schedule(acp, ts[i + 1])
        h = lam_s - lam_t
        if sde:
            a = (sg_s / sg_t) * math.exp(-h)
            b = -al_s * math.expm1(-2.0 * h)
            c = sg_s * math.sqrt(-math.expm1(-2.0 * h))
        else:
            a, b, c = sg_s / sg_t, -al_s * math.expm1(-h), 0.0
        if order == 2 and i > 0:
            r = h_prev / h
            w0, w1 = 1.0 + 1.0 / (2.0 * r), -1.0 / (2.0 * r)
        else:
            w0, w1 = 1.0, 0.0
        rows.append((sg_t, al_t, a, b, w0, w1, c, 10.0))
        h_prev = h
    return rows


def _guard(x):
    if torch.isnan(x).any() or torch.isinf(x).any():
        return torch.nan_to_num(x, nan=0.0, posinf=1.0, neginf=-1.0)
    return x


def sample(model, acp, timesteps, z, cond, order=2, sde=False, noise=None, dtype=torch.float32, record=None):
    """the loop from z_init = z (not modified).  model(z, t, c) -> eps with t a (B,) int64 tensor; the update runs in
    `dtype` with the coefficients rounded to it; noise[i] = step i's N(0,1) draw (SDE).  record: optional list that
    receives (z_t, t, eps) per step, for teacher-forced comparisons."""
    rows = coefficients(timesteps, acp, order, sde)
    z = z.to(dtype).clone()
    x0_prev = None
    for i, t in enumerate(timesteps):
        tt = torch.full((z.shape[0],), int(t), device=z.device, dtype=torch.long)
        eps = model(z, tt, cond)
        if record is not None:
            record.append((z.clone(), int(t), eps.clone()))
        sg_t, al_t, a, b, w0, w1, c, clip = (torch.tensor(v, dtype=dtype, device=z.device) for v in rows[i])
        eps = _guard(eps.to(dtype))
        x0 = torch.clamp(_guard((z - sg_t * eps) / al_t), -clip, clip)
        D = x0 if rows[i][5] == 0.0 else w0 * x0 + w1 * x0_prev
        z_new = a * z + b * D
        if rows[i][6] != 0.0:
            z_new = z_new + c * noise[i].to(dtype)
        z = _guard(z_new)
        x0_prev = x0
    return z
