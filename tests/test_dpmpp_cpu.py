"""DPM-Solver++(2M) without a GPU: the oracle's order of accuracy on Gaussian data (exact solution known), the host
coefficient rows of b2v_dpmpp_coefficients against the oracle and their identities, argument rejection."""
import ctypes
import inspect
import math

import numpy as np
import pytest
import torch

import dpmpp_oracle as O


def _acp(schedule):
    from v2v_b200.models import GaussianDiffusion
    return GaussianDiffusion(noise_schedule=schedule).alphas_cumprod.float()


# ------------------------------------------------------------------------------------- 1. order of accuracy
MU, S = 0.3, 0.7  # data ~ N(MU, S^2) per element


def _gauss_eps(acp64):
    """exact eps prediction for N(MU, S^2) data: sigma (z - alpha MU) / (alpha^2 S^2 + sigma^2)"""
    def model(z, t, c):
        a = acp64[t].view(-1, *([1] * (z.dim() - 1)))
        al, sg = a.sqrt(), (1 - a).sqrt()
        return sg * (z - al * MU) / (al ** 2 * S ** 2 + sg ** 2)
    return model


def _final_errors(schedule, order, Ns, t_start=960):
    acp = _acp(schedule)
    acp64 = acp.double()
    model = _gauss_eps(acp64)
    g = torch.Generator().manual_seed(0)
    aT, a0 = float(acp64[t_start]), float(acp64[0])
    (alT, sgT), (al0, sg0) = (math.sqrt(aT), math.sqrt(1 - aT)), (math.sqrt(a0), math.sqrt(1 - a0))
    zT = (torch.randn(100000, generator=g, dtype=torch.float64) * math.sqrt(alT ** 2 * S ** 2 + sgT ** 2) + alT * MU)
    zT = zT.view(1, -1)
    # the probability-flow ODE keeps (z - alpha MU) / sqrt(alpha^2 S^2 + sigma^2) constant: exact z at t = 0, then the
    # exact denoiser on it (the loop's last step applies the denoiser at t = 0)
    z0 = al0 * MU + math.sqrt(al0 ** 2 * S ** 2 + sg0 ** 2) * (zT - alT * MU) / math.sqrt(alT ** 2 * S ** 2 + sgT ** 2)
    ref = (z0 - sg0 * model(z0, torch.zeros(1, dtype=torch.long), None)) / al0
    errs = []
    for N in Ns:
        ts = np.linspace(t_start, 0, N + 1)
        assert np.all(ts == np.round(ts))
        got = O.sample(model, acp, ts.astype(np.int64), zT, None, order=order, dtype=torch.float64)
        errs.append(((got - ref) ** 2).mean().sqrt().item())
    return errs


@pytest.mark.parametrize("schedule,Ns", [("cosine", (10, 20, 40)), ("linear", (20, 40, 80))])
def test_oracle_order_of_accuracy_on_gaussian_data(schedule, Ns):
    e2 = _final_errors(schedule, 2, Ns)
    e1 = _final_errors(schedule, 1, Ns)
    r2 = [e2[k] / e2[k + 1] for k in range(len(Ns) - 1)]
    r1 = [e1[k] / e1[k + 1] for k in range(len(Ns) - 1)]
    print(f"{schedule} N={Ns}: order-2 errors {['%.3e' % e for e in e2]} ratios {['%.2f' % r for r in r2]}; "
          f"order-1 errors {['%.3e' % e for e in e1]} ratios {['%.2f' % r for r in r1]}")
    assert all(r >= 3.0 for r in r2), r2
    assert all(1.6 <= r <= 2.6 for r in r1), r1


# ------------------------------------------------------------------------------------- 2./3. coefficient rows
def _rows_native(ts, acp, order, sde):
    from v2v_b200.inference.sampler import dpmpp_coefficients
    return dpmpp_coefficients(ts, acp, order, sde).numpy()


def _timesteps(n):
    if n == 51:  # DDIM-50's subset
        return _ddim(50)
    return np.round(np.linspace(999, 0, n)).astype(np.int64) if n > 1 else np.array([999], dtype=np.int64)


def _ddim(steps):
    from v2v_b200.inference import DDIMSampler
    from v2v_b200.models import GaussianDiffusion
    return np.ascontiguousarray(DDIMSampler(GaussianDiffusion(), None)._get_timesteps(steps), dtype=np.int64)


def _ulp_diff(a, b):
    ia = np.asarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    ib = np.asarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    # map the sign-magnitude bit patterns to a monotone integer line
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return np.abs(ia - ib)


CASES = [(s, n, o, sde) for s in ("cosine", "linear") for n in (1, 2, 3, 11, 21, 51) for o in (1, 2) for sde in (0, 1)]


@pytest.mark.parametrize("schedule,n,order,sde", CASES)
def test_rows_equal_oracle_and_identities(schedule, n, order, sde):
    acp = _acp(schedule)
    ts = _timesteps(n)
    assert len(ts) == n and np.all(np.diff(ts) < 0)
    got = _rows_native(ts, acp, order, sde)
    want64 = np.array(O.coefficients(ts, acp, order, bool(sde)), dtype=np.float64)
    want = want64.astype(np.float32)
    d = _ulp_diff(got, want)
    assert d.max() <= 2, (d.max(), np.argwhere(d > 2)[:4].tolist())
    r = got.astype(np.float64)
    # w0 + w1 = 1 and a alpha_t + b = alpha_s (the update is exact for a point mass at the prediction)
    assert np.allclose(r[:, 4] + r[:, 5], 1.0, rtol=0, atol=1e-6)
    al_s = np.array([math.sqrt(float(acp[t])) for t in ts[1:]] + [1.0])
    sg_s = np.array([math.sqrt(1 - float(acp[t])) for t in ts[1:]] + [0.0])
    assert np.allclose(r[:, 2] * r[:, 1] + r[:, 3], al_s, rtol=0, atol=2e-6)
    if sde:  # a^2 sigma_t^2 + c^2 = sigma_s^2: the marginal variance of point-mass data is kept
        assert np.allclose(r[:, 2] ** 2 * r[:, 0] ** 2 + r[:, 6] ** 2, sg_s ** 2, rtol=0, atol=2e-6)
    else:
        assert np.all(r[:, 6] == 0)
    assert r[-1, 2:].tolist() == [0.0, 1.0, 1.0, 0.0, 0.0, 10.0]
    assert np.all(r[:, 7] == 10.0)
    # order 2 only between the first and the last step
    assert r[0, 5] == 0.0
    if order == 1:
        assert np.all(r[:, 5] == 0.0)
    elif n > 2:
        assert np.all(r[1:-1, 5] != 0.0)


def test_rows_at_t999_cosine_use_the_exact_schedule():
    """no DDIM-style +1e-8 terms: cosine acp_999 = 2.43e-10, alpha_999 = 1.56e-5"""
    acp = _acp("cosine")
    r = _rows_native(np.array([999, 980], dtype=np.int64), acp, 2, 0)
    assert abs(r[0, 1] - math.sqrt(float(acp[999]))) <= 1e-7 * r[0, 1]
    assert 1.5e-5 < r[0, 1] < 1.6e-5


# ------------------------------------------------------------------------------------- 4. rejections
def _call(ts, n, acp, n_train, order, sde, rows=True):
    from v2v_b200 import _lib
    L = _lib.lib()
    keep = None if ts is None else np.ascontiguousarray(ts, dtype=np.int64)  # alive for the call
    ts_p = None if keep is None else keep.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    acp_p = None if acp is None else ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float))
    out = torch.zeros((max(n, 1), 8))
    out_p = ctypes.cast(out.data_ptr(), ctypes.POINTER(ctypes.c_float)) if rows else None
    return L.b2v_dpmpp_coefficients(ts_p, n, acp_p, n_train, order, sde, out_p), _lib.last_error()


def test_coefficients_reject_invalid_arguments():
    acp = _acp("cosine").contiguous()
    ok = np.array([999, 500, 0])
    assert _call(ok, 3, acp, 1000, 2, 0)[0] == 0
    bad = {
        "n = 0": _call(ok, 0, acp, 1000, 2, 0),
        "n > 4096": _call(np.arange(4097)[::-1], 4097, acp, 1000, 2, 0),
        "order 0": _call(ok, 3, acp, 1000, 0, 0),
        "order 3": _call(ok, 3, acp, 1000, 3, 0),
        "sde 2": _call(ok, 3, acp, 1000, 2, 2),
        "increasing": _call(np.array([0, 500, 999]), 3, acp, 1000, 2, 0),
        "repeated": _call(np.array([999, 500, 500]), 3, acp, 1000, 2, 0),
        "t = n_train": _call(np.array([1000, 500, 0]), 3, acp, 1000, 2, 0),
        "t < 0": _call(np.array([999, 500, -1]), 3, acp, 1000, 2, 0),
        "null timesteps": _call(None, 3, acp, 1000, 2, 0),
        "null alphas_cumprod": _call(ok, 3, None, 1000, 2, 0),
        "null rows": _call(ok, 3, acp, 1000, 2, 0, rows=False),
    }
    for what, (rc, msg) in bad.items():
        assert rc != 0, what
        assert msg.startswith("dpmpp_coefficients:"), (what, msg)


def test_sampler_signature_and_order_validation():
    from v2v_b200.inference import DPMSolverSampler
    from v2v_b200.models import GaussianDiffusion
    params = list(inspect.signature(DPMSolverSampler.sample).parameters.items())
    assert [k for k, _ in params] == ["self", "shape", "conditioning", "num_inference_steps", "device", "order",
                                      "stochastic", "progress"]
    assert dict(params)["order"].default == 2 and dict(params)["stochastic"].default is False
    smp = DPMSolverSampler(GaussianDiffusion(), lambda z, t, c: z)
    assert smp._get_timesteps(20).tolist()[:3] == [999, 950, 900] and len(smp._get_timesteps(20)) == 21
    for order in (0, 3):
        with pytest.raises(ValueError, match="order"):
            smp.sample((1, 4, 2, 4, 4), torch.zeros(1, 4, 2, 4, 4), 5, "cpu", order=order)


def test_generate_rejects_unknown_sampler_names():
    from v2v_b200.models import VideoToVideoDiffusion
    cfg = {"in_channels": 1, "latent_dim": 4, "vae_base_channels": 64, "unet_model_channels": 64,
           "unet_num_res_blocks": 1, "unet_attention_levels": [1], "unet_channel_mult": [1, 2], "unet_num_heads": 2,
           "unet_time_embed_dim": 128}
    m = VideoToVideoDiffusion(cfg)
    for name in ("euler", "dpmpp_3m", "dpmpp_2s"):
        with pytest.raises(ValueError, match="Unknown sampler"):
            m.generate(torch.zeros(1, 1, 2, 16, 16), name)
