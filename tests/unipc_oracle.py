"""UniPC restated in Python straight from the paper, independently of libb2v's b2v_unipc_coefficients: Zhao et al. 2023,
"UniPC: A Unified Predictor-Corrector Framework for Fast Sampling of Diffusion Models", the multistep UniP-p predictor
and the UniC corrector with B(h) = h (bh1) or e^h - 1 (bh2), data prediction, as in diffusers' UniPCMultistepScheduler
(multistep_uni_p_bh_update / multistep_uni_c_bh_update with predict_x0=True).  Test infrastructure only.

The schedule enters as per-point (alpha, sigma) in fp64, lambda = log(alpha / sigma), so a continuous schedule can drive
it as well as the library's timesteps (`schedule`).  m_i = clamp((z_i - sigma_i eps_i) / alpha_i, +-10) is the data
prediction at the evaluated (uncorrected) state.  Step i: the corrector (i >= 1, the order of the previous predictor)
turns x^c_{i-1} into x^c_i using m_i; the predictor of order k_i takes x^c_i to the next point.

`coefficients` does not expand the formulas: it evaluates the two updates on unit inputs (the updates are linear in
z_i, x^c_{i-1} and m_i .. m_{i-3}) to get each step's row, so the C rows are checked against the formulas themselves.
"""
import math

import numpy as np
import torch

CLIP = 10.0


def schedule(acp, timesteps):
    """(alphas, sigmas) of the timesteps in fp64 from the fp32 table"""
    a = [float(acp[int(t)]) for t in timesteps]
    return [math.sqrt(x) for x in a], [math.sqrt(1.0 - x) for x in a]


def _phi(h, variant, k):
    """phi1 = e^{-h} - 1, B(h) and b_q = h phi_{q+1}(-h) q! / B(h), q = 1..k (the phi_k recursion of the paper)"""
    hh = -h
    phi1 = math.expm1(hh)
    B = hh if variant == "bh1" else math.expm1(hh)
    hphi, fac, b = phi1 / hh - 1.0, 1, []
    for q in range(1, k + 1):
        b.append(hphi * fac / B)
        fac *= q + 1
        hphi = hphi / hh - 1.0 / fac
    return phi1, B, b


def _corrector(i, xc_prev, ms, al, sg, lam, k, variant):
    """UniC-k: x^c_i from x^c_{i-1}; ms[j] = m_{i-j}"""
    h = lam[i] - lam[i - 1]
    phi1, B, b = _phi(h, variant, k)
    rks, D = [], []
    for j in range(1, k):
        rk = (lam[i - 1 - j] - lam[i - 1]) / h
        rks.append(rk)
        D.append((ms[1 + j] - ms[1]) / rk)
    rks.append(1.0)
    R = np.array([[r ** q for r in rks] for q in range(k)])
    rho = [0.5] if k == 1 else np.linalg.solve(R, np.array(b))
    corr = rho[-1] * (ms[0] - ms[1])
    for j in range(k - 1):
        corr = corr + rho[j] * D[j]
    return sg[i] / sg[i - 1] * xc_prev - al[i] * phi1 * ms[1] - al[i] * B * corr


def _predictor(i, xc, ms, al, sg, lam, k, variant):
    """UniP-k: the state at point i+1 from x^c_i; ms[j] = m_{i-j}.  To the clean sample (lambda = inf): m_i"""
    if math.isinf(lam[i + 1]):
        return ms[0]
    h = lam[i + 1] - lam[i]
    phi1, B, b = _phi(h, variant, k)
    rks, D = [], []
    for j in range(1, k):
        rk = (lam[i - j] - lam[i]) / h
        rks.append(rk)
        D.append((ms[j] - ms[0]) / rk)
    z = sg[i + 1] / sg[i] * xc - al[i + 1] * phi1 * ms[0]
    if k > 1:
        R = np.array([[r ** q for r in rks] for q in range(k - 1)])
        rho = [0.5] if k == 2 else np.linalg.solve(R, np.array(b[:-1]))
        pred = rho[0] * D[0]
        for j in range(1, k - 1):
            pred = pred + rho[j] * D[j]
        z = z - al[i + 1] * B * pred
    return z


def _points(al, sg, clean):
    """alpha, sigma, lambda lists over the evaluation points, plus the clean sample when `clean`"""
    al, sg = [float(a) for a in al], [float(s) for s in sg]
    lam = [math.log(a / s) for a, s in zip(al, sg)]
    return (al + [1.0], sg + [0.0], lam + [math.inf]) if clean else (al, sg, lam)


def predictor_order(i, order, n):
    """k_i = min(p, i+1, n-i): lower order in the warm-up and on the last steps of an n-evaluation loop"""
    return min(order, i + 1, n - i)


def coefficients(al, sg, order=3, variant="bh2"):
    """fp64 rows (sigma, alpha, g, a_c, c0..c3, a_p, p0..p2, clip, 0, 0, 0) of an n-point loop whose last step goes to
    the clean sample: x^c = g z + a_c x^c_prev + sum_j c_j m_{i-j};  z' = a_p x^c + sum_j p_j m_{i-j}"""
    n = len(al)
    A, S, lam = _points(al, sg, True)
    rows = np.zeros((n, 16))
    unit = lambda j, size: [1.0 if q == j else 0.0 for q in range(size)]  # noqa: E731
    for i in range(n):
        r = rows[i]
        r[0], r[1], r[12] = S[i], A[i], CLIP
        if i == 0:
            r[2] = 1.0  # x^c_0 = z_0
        else:
            k = predictor_order(i - 1, order, n)
            r[3] = _corrector(i, 1.0, [0.0] * 4, A, S, lam, k, variant)
            for j in range(4):
                r[4 + j] = _corrector(i, 0.0, unit(j, 4), A, S, lam, k, variant)
        k = predictor_order(i, order, n)
        r[8] = _predictor(i, 1.0, [0.0] * 3, A, S, lam, k, variant)
        for j in range(3):
            r[9 + j] = _predictor(i, 0.0, unit(j, 3), A, S, lam, k, variant)
    return rows


def _guard(x):
    if torch.isnan(x).any() or torch.isinf(x).any():
        return torch.nan_to_num(x, nan=0.0, posinf=1.0, neginf=-1.0)
    return x


def sample(model, al, sg, z, order=3, variant="bh2", corrector=True, clean=True, dtype=torch.float64, record=None):
    """the loop from z (not modified); model(z, i) -> eps at evaluation point i.  clean=True: n steps, the last one to
    the clean sample, predictor orders min(p, i+1, n-i), returns that sample.  clean=False: n-1 steps between the
    points, orders min(p, i+1), returns the corrected state at the last point (what a convergence study measures).
    corrector=False keeps x^c_i = z_i (UniP alone).  record: optional list of (z_i, i, eps_i) per evaluation."""
    n = len(al)
    A, S, lam = _points(al, sg, clean)
    z = z.to(dtype).clone()
    ms, xc, k_prev = [], None, None
    for i in range(n):
        eps = model(z, i)
        if record is not None:
            record.append((z.clone(), i, eps.clone()))
        eps = _guard(eps.to(dtype))
        m = torch.clamp(_guard((z - S[i] * eps) / A[i]), -CLIP, CLIP)
        ms = [m] + ms[:3]
        xc = z if (i == 0 or not corrector) else _corrector(i, xc, ms, A, S, lam, k_prev, variant)
        if not clean and i == n - 1:
            return xc
        k_prev = predictor_order(i, order, n) if clean else min(order, i + 1)
        z = _guard(_predictor(i, xc, ms, A, S, lam, k_prev, variant))
    return z


def sample_timesteps(model, acp, timesteps, z, cond, order=3, variant="bh2", dtype=torch.float32, record=None):
    """sample() over the library's timesteps with model(z, t, c), t a (B,) int64 tensor; record gets (z_t, t, eps)"""
    al, sg = schedule(acp, timesteps)
    ts = [int(t) for t in timesteps]
    rec = [] if record is not None else None

    def eps_fn(zz, i):
        return model(zz, torch.full((zz.shape[0],), ts[i], device=zz.device, dtype=torch.long), cond)

    out = sample(eps_fn, al, sg, z, order, variant, dtype=dtype, record=rec)
    if record is not None:
        record.extend((zz, ts[i], e) for zz, i, e in rec)
    return out
