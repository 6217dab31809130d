"""ctypes binding of libb2v.so -- the C ABI declared in include/b2v.h.

This is the only place Python touches native code.  There is deliberately no fallback: if the shared library is
missing or no sm_100 device is present every call raises.  torch is used for device memory and streams only.
"""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_float, c_int, c_int64, c_longlong, c_size_t, c_uint64, c_void_p

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libb2v.so")
_lib = None


class UNetDesc(ctypes.Structure):
    _fields_ = [
        ("latent_dim", c_int),
        ("model_channels", c_int),
        ("num_res_blocks", c_int),
        ("num_levels", c_int),
        ("channel_mult", c_int * 8),
        ("attention_mask", c_int),
        ("num_heads", c_int),
        ("time_embed_dim", c_int),
    ]


class VAEDesc(ctypes.Structure):
    _fields_ = [("in_channels", c_int), ("latent_dim", c_int), ("base_channels", c_int), ("scaling_factor", c_float)]


class SamplerCfg(ctypes.Structure):
    """b2v_sampler_cfg: the schedule tables b2v_generate runs its sampler with (host pointers; noise is a device pointer)"""
    _fields_ = [("sampler", c_int), ("n", c_int), ("timesteps", POINTER(c_int64)), ("alphas_cumprod", POINTER(c_float)),
                ("n_train", c_int), ("eta", c_float), ("ddpm_coef", POINTER(c_float)), ("noise", c_void_p),
                ("seed", c_uint64), ("unipc_order", c_int), ("unipc_variant", c_int)]


# name -> (restype, argtypes); mirrors include/b2v.h one to one
_P = c_void_p
SIGNATURES = {
    "b2v_last_error": (c_char_p, []),
    "b2v_abi_version": (c_int, []),
    "b2v_launch_count": (c_longlong, []),
    "b2v_unet_create": (c_int, [POINTER(_P), POINTER(UNetDesc)]),
    "b2v_unet_destroy": (None, [_P]),
    "b2v_unet_load_weight": (c_int, [_P, c_char_p, _P, POINTER(c_int64), c_int]),
    "b2v_unet_set_attention": (c_int, [_P, c_int]),
    "b2v_unet_finalize": (c_int, [_P]),
    "b2v_unet_forward": (c_int, [_P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    "b2v_ddim_sample": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, POINTER(c_int64), c_int, POINTER(c_float),
                                c_int, c_float, _P, _P, _P]),
    "b2v_dpmpp_coefficients": (c_int, [POINTER(c_int64), c_int, POINTER(c_float), c_int, c_int, c_int, POINTER(c_float)]),
    "b2v_dpmpp_sample": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, POINTER(c_int64), c_int, POINTER(c_float),
                                 c_int, c_int, c_int, _P, _P, _P]),
    "b2v_dpmpp_update": (c_int, [_P, _P, _P, _P, _P, c_longlong, _P, _P]),
    "b2v_unipc_coefficients": (c_int, [POINTER(c_int64), c_int, POINTER(c_float), c_int, c_int, c_int, POINTER(c_float)]),
    "b2v_unipc_sample": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, POINTER(c_int64), c_int, POINTER(c_float),
                                 c_int, c_int, c_int, _P, _P]),
    "b2v_unipc_update": (c_int, [_P, _P, _P, _P, _P, c_int, c_longlong, _P, _P]),
    "b2v_sampler_begin": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    "b2v_ddpm_step": (c_int, [_P, c_int64, POINTER(c_float), _P, _P]),
    "b2v_sampler_end": (c_int, [_P, _P, _P]),
    "b2v_ddpm_sample": (c_int, [_P, _P, _P, _P, c_int, c_int, c_int, c_int, POINTER(c_float), c_int, _P, c_uint64, _P]),
    "b2v_ddpm_run": (c_int, [_P, POINTER(c_float), c_int, c_int, c_int, _P, c_uint64, _P]),
    "b2v_ddim_timesteps": (c_int, [c_int, c_int, POINTER(c_int64), c_int]),
    "b2v_philox_normal": (c_int, [_P, c_uint64, c_int, c_longlong, _P]),
    "b2v_generate": (c_int, [_P, _P, POINTER(SamplerCfg), _P, _P, _P, c_int, c_int, c_int, c_int, c_int, _P, _P]),
    "b2v_generate_ensemble": (c_int, [_P, _P, POINTER(SamplerCfg), _P, _P, c_int, _P, _P, _P, c_int, c_int, c_int, c_int,
                                      c_int, _P, _P]),
    "b2v_ensemble_stats": (c_int, [_P, _P, _P, c_int, c_longlong, _P]),
    "b2v_q_sample": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_longlong, _P]),
    "b2v_eps_mse_ws_bytes": (c_size_t, [c_int]),
    "b2v_eps_mse": (c_int, [_P, _P, _P, _P, _P, c_size_t, c_int, c_longlong, c_longlong, _P]),
    "b2v_vae_create": (c_int, [POINTER(_P), POINTER(VAEDesc)]),
    "b2v_vae_destroy": (None, [_P]),
    "b2v_vae_load_weight": (c_int, [_P, c_char_p, _P, POINTER(c_int64), c_int]),
    "b2v_vae_finalize": (c_int, [_P]),
    "b2v_vae_encode": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    "b2v_vae_decode": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, _P]),
    "b2v_upsample_depth": (c_int, [_P, _P, c_int, c_int, c_int, c_int, _P]),
    "b2v_stitch_accumulate": (c_int, [_P, _P, _P, _P, _P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int,
                                      c_int, c_int, _P]),
    "b2v_stitch_normalize": (c_int, [_P, _P, c_longlong, _P]),
    "b2v_video_metrics": (c_int, [_P, _P, _P, c_int, c_int, c_int, c_int, c_float, _P]),
    "b2v_extract_patch": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_int, c_float,
                                  c_float, c_float, c_float, _P]),
    "b2v_unet_profile": (c_int, [_P, c_int, c_char_p, c_size_t, _P]),
    "b2v_vae_profile": (c_int, [_P, c_int, c_int, c_char_p, c_size_t, _P]),
    "b2v_debug_op_output": (c_longlong, [_P, c_int, c_int, c_int, _P, c_size_t, _P]),
    "b2v_debug_op_name": (c_char_p, [_P, c_int, c_int]),
    "b2v_conv_create": (c_int, [POINTER(_P), c_int, _P, _P, c_int, c_int, c_int]),
    "b2v_conv_destroy": (None, [_P]),
    "b2v_conv_forward": (c_int, [_P, _P, _P, _P, c_int, _P, c_int, c_int, c_int, c_int, c_int, c_int, _P]),
    "b2v_nc32_to_cl16": (c_int, [_P, _P, c_int, c_int, c_int, c_longlong, _P]),
    "b2v_cl16_to_nc32": (c_int, [_P, _P, c_int, c_int, c_int, c_longlong, _P]),
    "b2v_gn_apply": (c_int, [_P, _P, _P, _P, _P, _P, _P, c_int, c_longlong, c_int, c_int, c_int, _P, c_int, _P]),
    "b2v_res_attn_tail": (c_int, [_P, _P, _P, _P, _P, c_int, _P, _P, c_int, _P, _P, _P, _P, c_longlong, c_int, c_int,
                                  c_int, c_int, _P]),
    "b2v_temporal_attention": (c_int, [_P, _P, c_int, c_int, c_int, c_int, c_int, _P]),
    "b2v_gn_stats": (c_int, [_P, c_int, c_longlong, c_int, c_int, _P, _P]),
    "b2v_ddim_update": (c_int, [_P, _P, _P, _P, c_longlong, _P, _P]),
    "b2v_ddpm_update": (c_int, [_P, _P, _P, POINTER(c_float), c_longlong, _P]),
}


def lib():
    """Load libb2v.so (once).  Raises if it has not been built -- there is no Python/torch fallback path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or `make -C video-to-video-diffusion_b200/csrc`). There is no fallback implementation.")
        handle = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(handle, name)
            fn.restype = res
            fn.argtypes = args
        if handle.b2v_abi_version() != 2:
            raise RuntimeError("libb2v.so ABI version mismatch; rebuild it")
        _lib = handle
    return _lib


def last_error():
    return lib().b2v_last_error().decode("utf-8", "replace")


def check(rc, what):
    if rc != 0:
        raise RuntimeError(f"{what}: {last_error()}")


def dptr(t, dtype=torch.float32):
    """device pointer of a contiguous CUDA tensor (or None)"""
    if t is None:
        return None
    if not t.is_cuda:
        raise RuntimeError("libb2v needs CUDA tensors (no CPU fallback)")
    if t.dtype != dtype:
        raise TypeError(f"expected {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise ValueError("tensor must be contiguous")
    return c_void_p(t.data_ptr())


def hptr(t):
    """host pointer of a contiguous fp32 CPU tensor"""
    assert not t.is_cuda and t.dtype == torch.float32 and t.is_contiguous()
    return c_void_p(t.data_ptr())


def stream():
    return c_void_p(torch.cuda.current_stream().cuda_stream)


def launch_count():
    return int(lib().b2v_launch_count())
