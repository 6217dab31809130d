"""UniPC without a GPU: the oracle's order of accuracy on Gaussian data (exact solution known), its reduction to
DPM-Solver++(2M), its error at the library's timesteps against dpmpp_2m, the host coefficient rows of
b2v_unipc_coefficients against the oracle and their identities, and argument rejection (C entries and Python names)."""
import ctypes
import inspect
import math

import numpy as np
import pytest
import torch

import dpmpp_oracle as DO
import unipc_oracle as O

MU, S = 0.3, 0.7  # data ~ N(MU, S^2) per element


def _acp(schedule):
    from v2v_b200.models import GaussianDiffusion
    return GaussianDiffusion(noise_schedule=schedule).alphas_cumprod.float()


def _library_timesteps(N):
    from v2v_b200.inference import DDIMSampler
    from v2v_b200.models import GaussianDiffusion
    return np.ascontiguousarray(DDIMSampler(GaussianDiffusion(), None)._get_timesteps(N), dtype=np.int64)


# ------------------------------------------------------------------------------------- 1. order of accuracy
def _vp(lam):
    """continuous VP schedule: alpha^2 + sigma^2 = 1, lambda = log(alpha / sigma)"""
    a = 1.0 / math.sqrt(1.0 + math.exp(-2.0 * lam))
    return a, a * math.exp(-lam)


def _exact_z(zT, aT, sT, a, s):
    """the probability-flow ODE keeps (z - alpha MU) / sqrt(alpha^2 S^2 + sigma^2) constant for N(MU, S^2) data"""
    return a * MU + math.sqrt(a * a * S * S + s * s) * (zT - aT * MU) / math.sqrt(aT * aT * S * S + sT * sT)


def _gauss_eps(a, s):
    """exact eps prediction for N(MU, S^2) data at (alpha, sigma)"""
    return lambda z: s * (z - a * MU) / (a * a * S * S + s * s)


MIN_ORDER = {1: 1.8, 2: 2.7, 3: 3.0}


@pytest.mark.parametrize("variant", ["bh1", "bh2"])
@pytest.mark.parametrize("order", [1, 2, 3])
def test_oracle_order_of_accuracy_on_gaussian_data(order, variant):
    """uniform lambda steps on [-3, 3]; the corrected state at the last point against the exact solution"""
    lT, l0 = -3.0, 3.0
    aT, sT = _vp(lT)
    g = torch.Generator().manual_seed(0)
    zT = torch.randn(20000, generator=g, dtype=torch.float64) * math.sqrt(aT * aT * S * S + sT * sT) + aT * MU
    ref = _exact_z(zT, aT, sT, *_vp(l0))
    errs = []
    for N in (16, 32, 64):
        ab = [_vp(lam) for lam in np.linspace(lT, l0, N + 1)]
        al, sg = [a for a, _ in ab], [s for _, s in ab]
        got = O.sample(lambda z, i: _gauss_eps(al[i], sg[i])(z), al, sg, zT, order, variant, clean=False)
        errs.append(((got - ref) ** 2).mean().sqrt().item())
    orders = [math.log2(errs[k] / errs[k + 1]) for k in range(2)]
    print(f"UniPC-{order} {variant}: errors {['%.3e' % e for e in errs]}, observed orders "
          f"{['%.2f' % o for o in orders]}")
    assert orders[-1] >= MIN_ORDER[order], orders


# ------------------------------------------------------------------------------------- 2. DPM-Solver++ and dpmpp_2m
def _library_setup(schedule="cosine", n_el=100000):
    acp = _acp(schedule)
    acp64 = acp.double()

    def model(z, t, c):
        a = acp64[t].view(-1, 1)
        al, sg = a.sqrt(), (1 - a).sqrt()
        return sg * (z - al * MU) / (al ** 2 * S ** 2 + sg ** 2)

    g = torch.Generator().manual_seed(0)
    aT, a0 = float(acp64[999]), float(acp64[0])
    (alT, sgT), (al0, sg0) = (math.sqrt(aT), math.sqrt(1 - aT)), (math.sqrt(a0), math.sqrt(1 - a0))
    zT = (torch.randn(n_el, generator=g, dtype=torch.float64) * math.sqrt(alT ** 2 * S ** 2 + sgT ** 2) + alT * MU)
    zT = zT.view(1, -1)
    z0 = _exact_z(zT, alT, sgT, al0, sg0)
    ref = (z0 - sg0 * model(z0, torch.zeros(1, dtype=torch.long), None)) / al0  # the loop ends with the t = 0 denoiser
    return acp, model, zT, ref


def _unipc(model, acp, ts, z, order, variant, corrector=True):
    al, sg = O.schedule(acp, ts)
    tt = [torch.full((1,), int(t), dtype=torch.long) for t in ts]
    return O.sample(lambda zz, i: model(zz, tt[i], None), al, sg, z, order, variant, corrector=corrector)


@pytest.mark.parametrize("order", [1, 2])
def test_oracle_without_corrector_is_dpmpp(order):
    acp, model, zT, _ = _library_setup(n_el=2000)
    for N in (5, 10, 20):
        ts = _library_timesteps(N)
        got = _unipc(model, acp, ts, zT, order, "bh2", corrector=False)
        want = DO.sample(model, acp, ts, zT, None, order=order, dtype=torch.float64)
        assert torch.allclose(got, want, rtol=0, atol=1e-12), (N, (got - want).abs().max().item())


def test_unipc3_bh2_beats_dpmpp_2m_at_library_timesteps():
    acp, model, zT, ref = _library_setup()
    err = lambda x: ((x - ref) ** 2).mean().sqrt().item()  # noqa: E731
    for N in (10, 15, 20, 25):
        ts = _library_timesteps(N)
        e_dpm = err(DO.sample(model, acp, ts, zT, None, order=2, dtype=torch.float64))
        e_uni = err(_unipc(model, acp, ts, zT, 3, "bh2"))
        print(f"N = {N}: dpmpp_2m {e_dpm:.3e}, UniPC-3 bh2 {e_uni:.3e} ({e_dpm / e_uni:.2f}x)")
        assert e_uni < e_dpm, (N, e_uni, e_dpm)


# ------------------------------------------------------------------------------------- 3. coefficient rows
def _rows_native(ts, acp, order, variant):
    from v2v_b200.inference.sampler import unipc_coefficients
    return unipc_coefficients(ts, acp, order, variant).numpy()


def _timesteps(n):
    if n == 51:  # DDIM-50's subset
        return _library_timesteps(50)
    return np.round(np.linspace(999, 0, n)).astype(np.int64) if n > 1 else np.array([999], dtype=np.int64)


def _ulp_diff(a, b):
    ia = np.asarray(a, dtype=np.float32).view(np.int32).astype(np.int64)
    ib = np.asarray(b, dtype=np.float32).view(np.int32).astype(np.int64)
    ia = np.where(ia < 0, -(ia & 0x7FFFFFFF), ia)
    ib = np.where(ib < 0, -(ib & 0x7FFFFFFF), ib)
    return np.abs(ia - ib)


CASES = [(s, n, o, v) for s in ("cosine", "linear") for n in (1, 2, 3, 4, 11, 21, 51) for o in (1, 2, 3)
         for v in ("bh1", "bh2")]


@pytest.mark.parametrize("schedule,n,order,variant", CASES)
def test_rows_equal_oracle_and_identities(schedule, n, order, variant):
    from v2v_b200.inference.sampler import dpmpp_coefficients
    acp = _acp(schedule)
    ts = _timesteps(n)
    assert len(ts) == n and np.all(np.diff(ts) < 0)
    got = _rows_native(ts, acp, order, variant)
    want = O.coefficients(*O.schedule(acp, ts), order, variant)
    d = _ulp_diff(got, want.astype(np.float32))
    assert d.max() <= 2, (d.max(), np.argwhere(d > 2)[:4].tolist())
    r = got.astype(np.float64)
    al, sg = O.schedule(acp, ts)
    lam = [math.log(a / s) for a, s in zip(al, sg)]
    # step 0: x^c_0 = z_0;  the last step: z' = m_{n-1};  clip 10 and three zero pads everywhere
    assert r[0, 2:8].tolist() == [1.0, 0.0, 0.0, 0.0, 0.0, 0.0]
    assert r[-1, 8:12].tolist() == [0.0, 1.0, 0.0, 0.0]
    assert np.all(r[:, 12] == 10.0) and np.all(r[:, 13:] == 0.0)
    assert np.all(r[1:, 2] == 0.0)  # the corrector does not read z after step 0
    # row sums: constant data predictions are transported exactly
    for i in range(1, n):
        assert abs(r[i, 4:8].sum() + al[i] * math.expm1(-(lam[i] - lam[i - 1]))) <= 4e-6 * max(1.0, al[i]), i
    for i in range(n - 1):
        assert abs(r[i, 9:12].sum() + al[i + 1] * math.expm1(-(lam[i + 1] - lam[i]))) <= 4e-6, i
    # the predictor uses no more history than its order k_i = min(p, i+1, n-i); the corrector no more than k_{i-1}
    for i in range(n):
        k = O.predictor_order(i, order, n)
        assert np.all(r[i, 9 + k:12] == 0.0) and (i == n - 1 or np.all(r[i, 9:9 + k] != 0.0)), i
        if i >= 1:
            kc = O.predictor_order(i - 1, order, n)
            assert np.all(r[i, 5 + kc:8] == 0.0) and np.all(r[i, 4:5 + kc] != 0.0), i
    if order == 1:  # the UniP-1 predictor is the first-order DPM-Solver++ step
        d1 = dpmpp_coefficients(ts, acp, 1, False).numpy()
        assert np.array_equal(got[:, 8], d1[:, 2]) and np.array_equal(got[:, 9], d1[:, 3])
        assert np.array_equal(got[:, :2], d1[:, :2])


# ------------------------------------------------------------------------------------- 4. rejections
def _call(ts, n, acp, n_train, order, variant, rows=True):
    from v2v_b200 import _lib
    L = _lib.lib()
    keep = None if ts is None else np.ascontiguousarray(ts, dtype=np.int64)  # alive for the call
    ts_p = None if keep is None else keep.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    acp_p = None if acp is None else ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float))
    out = torch.zeros((max(n, 1), 16))
    out_p = ctypes.cast(out.data_ptr(), ctypes.POINTER(ctypes.c_float)) if rows else None
    return L.b2v_unipc_coefficients(ts_p, n, acp_p, n_train, order, variant, out_p), _lib.last_error()


def test_coefficients_reject_invalid_arguments():
    acp = _acp("cosine").contiguous()
    ok = np.array([999, 500, 0])
    for order in (1, 2, 3):
        for variant in (0, 1):
            assert _call(ok, 3, acp, 1000, order, variant)[0] == 0
    bad_acp = acp.clone()
    bad_acp[500] = 1.0
    zero_acp = acp.clone()
    zero_acp[0] = 0.0
    bad = {
        "n = 0": _call(ok, 0, acp, 1000, 3, 1),
        "n > 4096": _call(np.arange(4097)[::-1], 4097, acp, 1000, 3, 1),
        "order 0": _call(ok, 3, acp, 1000, 0, 1),
        "order 4": _call(ok, 3, acp, 1000, 4, 1),
        "variant -1": _call(ok, 3, acp, 1000, 3, -1),
        "variant 2": _call(ok, 3, acp, 1000, 3, 2),
        "increasing": _call(np.array([0, 500, 999]), 3, acp, 1000, 3, 1),
        "repeated": _call(np.array([999, 500, 500]), 3, acp, 1000, 3, 1),
        "t = n_train": _call(np.array([1000, 500, 0]), 3, acp, 1000, 3, 1),
        "t < 0": _call(np.array([999, 500, -1]), 3, acp, 1000, 3, 1),
        "alphas_cumprod = 1": _call(ok, 3, bad_acp, 1000, 3, 1),
        "alphas_cumprod = 0": _call(ok, 3, zero_acp, 1000, 3, 1),
        "null timesteps": _call(None, 3, acp, 1000, 3, 1),
        "null alphas_cumprod": _call(ok, 3, None, 1000, 3, 1),
        "null rows": _call(ok, 3, acp, 1000, 3, 1, rows=False),
    }
    for what, (rc, msg) in bad.items():
        assert rc != 0, what
        assert msg.startswith("unipc_coefficients:"), (what, msg)


def test_generate_entries_reject_bad_unipc_configurations_before_any_device_call():
    """sampler code 4 with bad fields or tables fails in the argument checks (stand-in pointers, never dereferenced)"""
    from v2v_b200 import _lib
    L = _lib.lib()
    acp = _acp("cosine").contiguous()
    p = ctypes.c_void_p(1)
    for kw, phrase in ((dict(order=0), "order"), (dict(order=4), "order"), (dict(variant=2), "variant"),
                       (dict(ts=np.array([500, 999, 0])), "decreasing"), (dict(ts=np.array([999, 500, 1000])), "range"),
                       (dict(ts=np.arange(4097)[::-1]), "4096"), (dict(code=5), "4 = unipc")):
        ts = np.ascontiguousarray(kw.get("ts", np.array([999, 500, 0])), dtype=np.int64)
        cfg = _lib.SamplerCfg()
        cfg.sampler, cfg.n, cfg.n_train = kw.get("code", 4), len(ts), acp.numel()
        cfg.timesteps = ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
        cfg.alphas_cumprod = ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float))
        cfg.unipc_order, cfg.unipc_variant = kw.get("order", 3), kw.get("variant", 1)
        assert L.b2v_generate(p, p, ctypes.byref(cfg), p, p, p, 1, 2, 6, 16, 16, None, None) != 0, kw
        assert phrase in _lib.last_error(), (kw, _lib.last_error())
        assert L.b2v_generate_ensemble(p, p, ctypes.byref(cfg), p, p, 2, None, p, p, 1, 2, 6, 16, 16, None, None) != 0
        assert phrase in _lib.last_error(), (kw, _lib.last_error())
    assert L.b2v_unipc_update(None, p, p, p, p, 0, 8, None, None) != 0 and "null argument" in _lib.last_error()
    assert L.b2v_unipc_update(p, p, p, p, p, -1, 8, None, None) != 0 and "negative step" in _lib.last_error()
    assert L.b2v_unipc_sample(None, p, p, p, 1, 2, 4, 4, None, 3, None, 1000, 3, 1, None, None) != 0
    assert "null handle" in _lib.last_error()


CFG = {"in_channels": 1, "latent_dim": 4, "vae_base_channels": 64, "unet_model_channels": 64, "unet_num_res_blocks": 1,
       "unet_attention_levels": [1], "unet_channel_mult": [1, 2], "unet_num_heads": 2, "unet_time_embed_dim": 128}


def test_sampler_signature_and_validation_before_any_c_call(monkeypatch):
    from v2v_b200 import _lib
    from v2v_b200.inference import UniPCSampler
    from v2v_b200.models import GaussianDiffusion
    params = list(inspect.signature(UniPCSampler.sample).parameters.items())
    assert [k for k, _ in params] == ["self", "shape", "conditioning", "num_inference_steps", "device", "order",
                                      "variant", "progress"]
    assert dict(params)["order"].default == 3 and dict(params)["variant"].default == "bh2"
    assert "variant" in inspect.signature(UniPCSampler.sample_with_stitching).parameters
    smp = UniPCSampler(GaussianDiffusion(), lambda z, t, c: z)
    assert smp._get_timesteps(20).tolist()[:3] == [999, 950, 900] and len(smp._get_timesteps(20)) == 21

    def no_c_call():
        raise AssertionError("a C call was made")
    monkeypatch.setattr(_lib, "lib", no_c_call)
    for kw, match in ((dict(order=0), "order"), (dict(order=4), "order"), (dict(variant="bh3"), "variant")):
        with pytest.raises(ValueError, match=match):
            smp.sample((1, 4, 2, 4, 4), torch.zeros(1, 4, 2, 4, 4), 5, "cpu", **kw)
    from v2v_b200.inference.sampler import unipc_coefficients
    with pytest.raises(ValueError, match="variant"):
        unipc_coefficients([999, 0], GaussianDiffusion().alphas_cumprod, 3, "bh0")


def test_unipc_name_is_accepted_and_unknown_names_still_raise(monkeypatch):
    """"unipc" passes the name checks of generate / generate_batch / generate_ensemble and reaches the device check"""
    from v2v_b200.inference import ensemble
    from v2v_b200.inference.generate import generate_batch
    from v2v_b200.models import VideoToVideoDiffusion
    m = VideoToVideoDiffusion(CFG)
    v = torch.zeros(1, 1, 2, 16, 16)
    with pytest.raises(RuntimeError, match="B200 only"):
        m.generate(v, "unipc")
    with pytest.raises(RuntimeError, match="B200 only"):
        ensemble.generate_ensemble(m, v, "unipc", num_samples=2)
    for name in ("unipc_3", "UniPC", "unipc_bh1", "euler"):
        with pytest.raises(ValueError, match="Unknown sampler"):
            m.generate(v, name)
        with pytest.raises(ValueError, match="unknown sampler"):
            ensemble.generate_ensemble(m, v, name, num_samples=2)
    class Reached(Exception):
        pass

    def fake_sample(self, *a, **k):
        raise Reached()
    from v2v_b200.inference import sampler as S
    monkeypatch.setattr(S.UniPCSampler, "sample", fake_sample)
    monkeypatch.setattr(m.vae, "encode", lambda x: torch.zeros(1, 4, 2, 4, 4))
    with pytest.raises(Reached):
        generate_batch(m, v, sampler_type="unipc", device="cpu")
    with pytest.raises(ValueError, match="Unknown sampler type"):
        generate_batch(m, v, sampler_type="unipc2", device="cpu")
