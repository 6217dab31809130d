"""The U-Net's channel limit on the B200: the GroupNorm kernels run one thread per 8-channel vector of a row in blocks
of at most 256 threads, so no level may have more than 2048 channels.  UNet3D rejects such a model at construction
(tests/test_host_cpu.py); the native library rejects it in b2v_unet_finalize, before any weight is read."""
import ctypes

import pytest

pytestmark = pytest.mark.gpu


def _finalize_without_weights(model_channels, channel_mult):
    from v2v_b200 import _lib
    L = _lib.lib()
    d = _lib.UNetDesc()
    d.latent_dim, d.model_channels, d.num_res_blocks = 4, model_channels, 1
    d.num_levels = len(channel_mult)
    for i, m in enumerate(channel_mult):
        d.channel_mult[i] = m
    d.attention_mask, d.num_heads, d.time_embed_dim = 0b10, 4, 512
    h = ctypes.c_void_p()
    _lib.check(L.b2v_unet_create(ctypes.byref(h), ctypes.byref(d)), "create")
    try:
        return L.b2v_unet_finalize(h), _lib.last_error()
    finally:
        L.b2v_unet_destroy(h)


def test_finalize_rejects_levels_above_2048_channels(cuda_dev):
    from v2v_b200 import _lib
    n0 = _lib.launch_count()
    rc, err = _finalize_without_weights(1088, (1, 2))  # level 1: 2176 channels
    assert rc == -1 and "2048" in err, (rc, err)
    assert _lib.launch_count() == n0
    # at the limit the descriptor is accepted: finalize goes on to the weights, of which there are none
    rc, err = _finalize_without_weights(1024, (1, 2))
    assert rc == -1 and "missing state_dict key" in err, (rc, err)
