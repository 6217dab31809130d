"""Ensemble generation, host side: argument errors of generate_ensemble / ops.ensemble_stats before any C call, and
the argument checks of b2v_generate_ensemble / b2v_ensemble_stats, which come before any device call (so they answer
on a machine without a GPU too)."""
import ctypes
import inspect

import numpy as np
import pytest
import torch

CFG = {"in_channels": 1, "latent_dim": 4, "vae_base_channels": 64, "unet_model_channels": 64, "unet_num_res_blocks": 1,
       "unet_attention_levels": [1], "unet_channel_mult": [1, 2], "unet_num_heads": 2, "unet_time_embed_dim": 128}


def test_generate_ensemble_argument_errors_before_any_c_call(monkeypatch):
    from v2v_b200 import _lib
    from v2v_b200.inference import ensemble
    from v2v_b200.models import VideoToVideoDiffusion
    m = VideoToVideoDiffusion(CFG)

    def no_c_call():
        raise AssertionError("a C call was made")
    monkeypatch.setattr(_lib, "lib", no_c_call)
    v = torch.zeros(1, 1, 2, 16, 16)
    for kw, match in ((dict(num_samples=1), "num_samples"), (dict(num_samples=0), "num_samples"),
                      (dict(sampler="euler"), "unknown sampler"), (dict(v_in=torch.zeros(1, 2, 2, 16, 16)), "channels"),
                      (dict(v_in=torch.zeros(1, 1, 2, 18, 16)), "H, W"), (dict(v_in=torch.zeros(1, 1, 2, 16, 14)), "H, W"),
                      (dict(v_in=torch.zeros(1, 1, 16, 16)), "B, C, T, H, W")):
        args = dict(model=m, v_in=v, sampler="dpmpp_2m", num_samples=2)
        args.update(kw)
        with pytest.raises(ValueError, match=match):
            ensemble.generate_ensemble(**args)
    with pytest.raises(RuntimeError, match="B200 only"):
        ensemble.generate_ensemble(m, v, "ddim", num_samples=2)
    from v2v_b200 import ops
    with pytest.raises(ValueError, match="K >= 2"):
        ops.ensemble_stats(torch.zeros(1, 8))


def test_signatures():
    from v2v_b200.inference.ensemble import generate_ensemble
    from v2v_b200.inference.volume import generate_volume
    params = inspect.signature(generate_ensemble).parameters
    assert list(params) == ["model", "v_in", "sampler", "num_inference_steps", "num_samples", "target_depth",
                            "return_members"]
    assert params["num_inference_steps"].default == 20 and params["num_samples"].default == 4
    assert params["return_members"].default is False
    assert inspect.signature(generate_volume).parameters["num_samples"].default is None


def _ensemble(L, cfg, K=2, u=1, v=1, mean=1, std=1, B=1, H=16, sampler=2, ts=None, acp=None, noise=None):
    """b2v_generate_ensemble with stand-in (never dereferenced) device pointers: every case here fails validation"""
    keep = []
    ts = np.array([999, 500, 0], dtype=np.int64) if ts is None else ts
    acp = torch.linspace(0.999, 0.01, 1000).contiguous() if acp is None else acp
    keep += [ts, acp]
    cfg.sampler, cfg.n, cfg.n_train = sampler, len(ts), acp.numel()
    cfg.timesteps = ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    cfg.alphas_cumprod = ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float))
    cfg.noise = noise
    p = lambda x: None if x is None else ctypes.c_void_p(x)  # noqa: E731
    return L.b2v_generate_ensemble(p(u), p(v), ctypes.byref(cfg), p(1), p(1), K, None, p(mean), p(std), B, 2, 6, H, 16,
                                   None, None)


def test_c_entry_rejects_bad_arguments_before_any_device_call():
    from v2v_b200 import _lib
    L = _lib.lib()
    cfg = _lib.SamplerCfg()
    for kw, phrase in ((dict(u=None), "null argument"), (dict(v=None), "null argument"),
                       (dict(mean=None), "null argument"), (dict(std=None), "null argument"),
                       (dict(K=1), "K >= 2"), (dict(K=0), "K >= 2"), (dict(H=18), "bad shape"),
                       (dict(B=-1), "bad shape"), (dict(sampler=7), "unknown sampler"),
                       (dict(sampler=3), "noise"), (dict(ts=np.array([500, 999, 0], dtype=np.int64)), "decreasing")):
        assert _ensemble(L, cfg, **kw) != 0, kw
        msg = _lib.last_error()
        assert msg.startswith("generate_ensemble:") or msg.startswith("dpmpp_coefficients:"), (kw, msg)
        assert phrase in msg, (kw, msg)
    assert L.b2v_generate_ensemble(None, None, None, None, None, 2, None, None, None, 1, 2, 6, 16, 16, None, None) != 0
    assert "null argument" in _lib.last_error()
    p = ctypes.c_void_p(1)
    assert L.b2v_ensemble_stats(None, p, p, 2, 8, None) != 0 and "null argument" in _lib.last_error()
    assert L.b2v_ensemble_stats(p, p, p, 1, 8, None) != 0 and "K >= 2" in _lib.last_error()
