"""Op-level wrappers over the C ABI (building blocks + parity tests).  Activations are NDHWC fp16 ("cl16")."""
import ctypes

import torch

from . import _lib

KIND_K3, KIND_K1, KIND_DOWN, KIND_UPT = 0, 1, 2, 3
STAT_SCALE = float(1 << 20)  # GroupNorm statistics cross the C ABI as int64 Q43.20 fixed point (include/b2v.h)


def stats_to_float(stats):
    """int64 (B, G, 2) fixed-point (sum, sumsq) -> float64"""
    return stats.to(torch.float64) / STAT_SCALE


def stats_from_float(stats):
    """(B, G, 2) floating (sum, sumsq) -> the int64 fixed-point form the kernels read"""
    return torch.round(stats.to(torch.float64) * STAT_SCALE).to(torch.int64).contiguous()


def to_cl16(x, cpad=None):
    """(B,C,D,H,W) fp32 CUDA -> (B,D,H,W,Cpad) fp16"""
    B, C, D, H, W = x.shape
    cpad = cpad or C
    out = torch.empty((B, D, H, W, cpad), dtype=torch.float16, device=x.device)
    _lib.check(_lib.lib().b2v_nc32_to_cl16(_lib.dptr(x.contiguous()), _lib.dptr(out, torch.float16), B, C, cpad,
                                           D * H * W, _lib.stream()), "nc32_to_cl16")
    return out


def from_cl16(x, C=None):
    """(B,D,H,W,Cpad) fp16 -> (B,C,D,H,W) fp32"""
    B, D, H, W, cpad = x.shape
    C = C or cpad
    out = torch.empty((B, C, D, H, W), dtype=torch.float32, device=x.device)
    _lib.check(_lib.lib().b2v_cl16_to_nc32(_lib.dptr(x, torch.float16), _lib.dptr(out), B, C, cpad, D * H * W,
                                           _lib.stream()), "cl16_to_nc32")
    return out


class Conv:
    """One convolution layer on the tcgen05 implicit-GEMM kernel, built from torch-layout weights."""

    def __init__(self, kind, weight, bias, cin0, cin1, cout):
        self.kind, self.cin0, self.cin1, self.cout = kind, cin0, cin1, cout
        w = weight.detach().to("cpu", torch.float32).contiguous()
        b = None if bias is None else bias.detach().to("cpu", torch.float32).contiguous()
        h = ctypes.c_void_p()
        _lib.check(_lib.lib().b2v_conv_create(ctypes.byref(h), kind, _lib.hptr(w), None if b is None else _lib.hptr(b),
                                              cin0, cin1, cout), "conv_create")
        self._h = h

    def __call__(self, x0, x1=None, out_fp32=False, groups=0, tanh=False):
        """x0/x1: cl16 (B,D,H,W,C).  Returns (out, stats): out cl16 or NCDHW fp32; stats (B,groups,2) or None."""
        B, D, H, W, _ = x0.shape
        oH, oW = (H // 2, W // 2) if self.kind == KIND_DOWN else (2 * H, 2 * W) if self.kind == KIND_UPT else (H, W)
        if out_fp32:
            out = torch.empty((B, self.cout, D, oH, oW), dtype=torch.float32, device=x0.device)
        else:
            out = torch.empty((B, D, oH, oW, self.cout), dtype=torch.float16, device=x0.device)
        stats = torch.zeros((B, groups, 2), dtype=torch.int64, device=x0.device) if groups else None
        _lib.check(_lib.lib().b2v_conv_forward(
            self._h, _lib.dptr(x0, torch.float16), _lib.dptr(x1, torch.float16),
            _lib.dptr(out, torch.float32 if out_fp32 else torch.float16), int(out_fp32), _lib.dptr(stats, torch.int64),
            groups,
            int(tanh), B, D, H, W, _lib.stream()), "conv_forward")
        return out, stats

    def __del__(self):
        try:
            if self._h:
                _lib.lib().b2v_conv_destroy(self._h)
                self._h = None
        except Exception:
            pass


def gn_apply(y, stats, gamma, beta, groups, temb=None, res=None, mode=0, groups_out=0):
    """y: cl16 (B,D,H,W,C).  mode 0: silu(gn(y)) + temb ; mode 1: silu(gn(y) + res) ; mode 2: gn(y).
    Returns (out, stats_out)."""
    B, D, H, W, C = y.shape
    out = torch.empty_like(y)
    so = torch.zeros((B, groups_out, 2), dtype=torch.int64, device=y.device) if groups_out else None
    _lib.check(_lib.lib().b2v_gn_apply(
        _lib.dptr(y, torch.float16), _lib.dptr(out, torch.float16), _lib.dptr(stats, torch.int64), _lib.dptr(gamma),
        _lib.dptr(beta), _lib.dptr(temb), _lib.dptr(res, torch.float16), B, D * H * W, C, groups, mode,
        _lib.dptr(so, torch.int64), groups_out, _lib.stream()), "gn_apply")
    return out, so


def res_attn_tail(y, res, stats_in, gamma2, beta2, groups2, gamma_a, beta_a, groups_a, wpv, bias):
    """Fused ResBlock tail + TemporalAttention: returns silu(GN(y)+res) + Wpv.sum_t GN_a(.) + bias (cl16, new tensor).
    wpv: fp32 (C, C) folded projection [co][c]; bias: fp32 (C,)."""
    B, D, H, W, C = y.shape
    out = y.clone()
    wt = wpv.t().contiguous().to(torch.float16)
    sm = torch.zeros((B, groups_a, 2), dtype=torch.int64, device=y.device)
    ws = torch.empty(B * 5 * H * W * C, dtype=torch.float32, device=y.device)
    _lib.check(_lib.lib().b2v_res_attn_tail(
        _lib.dptr(out, torch.float16), _lib.dptr(res, torch.float16), _lib.dptr(stats_in, torch.int64), _lib.dptr(gamma2),
        _lib.dptr(beta2), groups2, _lib.dptr(gamma_a), _lib.dptr(beta_a), groups_a, _lib.dptr(wt, torch.float16),
        _lib.dptr(bias), _lib.dptr(sm, torch.int64), _lib.dptr(ws), ws.numel(), B, D, H * W, C, _lib.stream()), "res_attn_tail")
    return out


def temporal_attention(qkv, heads):
    """softmax attention over depth: qkv cl16 (B,T,H,W,3C) (the qkv 1x1 conv output) -> o cl16 (B,T,H,W,C),
    o[..., h*hd:(h+1)*hd] = softmax(q k^T / sqrt(hd)) v over the T tokens of each position and head h"""
    B, T, H, W, C3 = qkv.shape
    if C3 % 3:
        raise ValueError(f"temporal_attention: last dim {C3} is not 3C")
    C = C3 // 3
    out = torch.empty((B, T, H, W, C), dtype=torch.float16, device=qkv.device)
    if out.numel() == 0:
        return out
    with torch.cuda.device(qkv.device):
        _lib.check(_lib.lib().b2v_temporal_attention(_lib.dptr(qkv, torch.float16), _lib.dptr(out, torch.float16), B, T,
                                                     H * W, C, int(heads), _lib.stream()), "temporal_attention")
    return out


def gn_stats(x, groups):
    B, D, H, W, C = x.shape
    st = torch.zeros((B, groups, 2), dtype=torch.int64, device=x.device)
    _lib.check(_lib.lib().b2v_gn_stats(_lib.dptr(x, torch.float16), B, D * H * W, C, groups, _lib.dptr(st, torch.int64),
                                       _lib.stream()), "gn_stats")
    return st


def ddim_update(z, eps, coef, noise=None):
    """in-place DDIM update of z (fp32); coef: device fp32[8].  Returns the NaN flag tensor."""
    flag = torch.zeros(1, dtype=torch.int32, device=z.device)
    _lib.check(_lib.lib().b2v_ddim_update(_lib.dptr(z), _lib.dptr(eps), _lib.dptr(noise), _lib.dptr(coef), z.numel(),
                                          _lib.dptr(flag, torch.int32), _lib.stream()), "ddim_update")
    return flag


def dpmpp_update(z, x0_prev, eps, coef, noise=None):
    """in-place DPM-Solver++(2M) step on z and x0_prev (fp32); coef: device fp32[8], one b2v_dpmpp_coefficients row;
    noise: this step's N(0,1) draw (read when coef[6] != 0).  Returns the NaN flag tensor."""
    flag = torch.zeros(1, dtype=torch.int32, device=z.device)
    _lib.check(_lib.lib().b2v_dpmpp_update(_lib.dptr(z), _lib.dptr(x0_prev), _lib.dptr(eps), _lib.dptr(noise),
                                           _lib.dptr(coef), z.numel(), _lib.dptr(flag, torch.int32), _lib.stream()),
               "dpmpp_update")
    return flag


def ddpm_update(z, eps, noise, coef_row):
    """in-place DDPM ancestral update of z (fp32); coef_row: 8 host floats (GaussianDiffusion.ddpm_coefficients()[t])"""
    coef = (ctypes.c_float * 8)(*[float(v) for v in coef_row])
    _lib.check(_lib.lib().b2v_ddpm_update(_lib.dptr(z), _lib.dptr(eps), _lib.dptr(noise), coef, z.numel(),
                                          _lib.stream()), "ddpm_update")
    return z


def upsample_depth(z, depth):
    """F.interpolate(z, (depth, h, w), mode='trilinear', align_corners=False) for unchanged h, w"""
    B, C, D, H, W = z.shape
    out = torch.empty((B, C, depth, H, W), dtype=torch.float32, device=z.device)
    if out.numel() == 0:
        return out
    _lib.check(_lib.lib().b2v_upsample_depth(_lib.dptr(z.contiguous()), _lib.dptr(out), B * C, D, depth, H * W,
                                             _lib.stream()), "upsample_depth")
    return out


def gaussian_window_1d(n, device):
    """1-D factor of the reference's blending window (inference/sampler.py:455-479): exp(-x^2 / (2 (n/6)^2))"""
    x = torch.arange(n).float() - (n - 1) / 2
    return torch.exp(-(x ** 2) / (2 * (n / 6) ** 2)).to(device).contiguous()


def stitch_accumulate(patch, acc, wsum, d0, h0, w0, win=None):
    """acc[..., d0:d0+pd, h0:h0+ph, w0:w0+pw] += patch * window ; wsum likewise (in place, fp32 NCDHW)"""
    B, C, pd, ph, pw = patch.shape
    _, _, D, H, W = acc.shape
    gd, gh, gw = win if win is not None else (gaussian_window_1d(pd, patch.device), gaussian_window_1d(ph, patch.device),
                                              gaussian_window_1d(pw, patch.device))
    _lib.check(_lib.lib().b2v_stitch_accumulate(_lib.dptr(patch.contiguous()), _lib.dptr(acc), _lib.dptr(wsum),
                                                _lib.dptr(gd), _lib.dptr(gh), _lib.dptr(gw), B * C, pd, ph, pw, D, H, W,
                                                int(d0), int(h0), int(w0), _lib.stream()), "stitch_accumulate")


def stitch_normalize(acc, wsum):
    _lib.check(_lib.lib().b2v_stitch_normalize(_lib.dptr(acc), _lib.dptr(wsum), acc.numel(), _lib.stream()),
               "stitch_normalize")
    return acc


def philox_normal(n, seed, step, device):
    """the N(0,1) draws b2v_ddpm_sample generates on the device for loop step `step` when no noise is supplied"""
    out = torch.empty(n, dtype=torch.float32, device=device)
    with torch.cuda.device(device):
        _lib.check(_lib.lib().b2v_philox_normal(_lib.dptr(out), int(seed), int(step), n, _lib.stream()), "philox_normal")
    return out


def q_sample(z0, t, noise, sqrt_ac, sqrt_1m_ac):
    """forward diffusion z_t = sqrt_ac[t] z_0 + sqrt_1m_ac[t] noise (reference models/diffusion.py:81-107)"""
    B = z0.shape[0]
    zt = torch.empty_like(z0)
    if z0.numel():
        _lib.check(_lib.lib().b2v_q_sample(_lib.dptr(z0), _lib.dptr(noise), _lib.dptr(t, torch.int64), _lib.dptr(sqrt_ac),
                                           _lib.dptr(sqrt_1m_ac), _lib.dptr(zt), B, z0.numel() // B, _lib.stream()),
                   "q_sample")
    return zt


def eps_mse(eps_pred, noise, mask=None):
    """per sample (sum mask*(eps_pred-noise)^2, sum mask) -> (B, 2) fp32; mask (B, C, T) or None"""
    B, C, T, H, W = eps_pred.shape
    out = torch.zeros((B, 2), dtype=torch.float32, device=eps_pred.device)
    if eps_pred.numel() == 0:
        return out
    L = _lib.lib()
    ws = torch.empty(int(L.b2v_eps_mse_ws_bytes(B)) // 8, dtype=torch.float64, device=eps_pred.device)
    _lib.check(L.b2v_eps_mse(_lib.dptr(eps_pred), _lib.dptr(noise), _lib.dptr(mask), _lib.dptr(out),
                             _lib.dptr(ws, torch.float64), ws.numel() * 8, B, C * T * H * W, H * W, _lib.stream()),
               "eps_mse")
    return out
