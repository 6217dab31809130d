"""Ensemble generation on the GPU: generate_ensemble / b2v_generate_ensemble against the staged composition of the
existing ops (bitwise), the statistics kernel against torch fp64, the NaN flag, argument rejection, and the
ensemble mode of generate_volume."""
import ctypes
import os

import numpy as np
import pytest
import torch

from helpers import golden

pytestmark = pytest.mark.gpu


def _tiny_model(dev):
    from v2v_b200.models import VideoToVideoDiffusion
    g = golden("generate_tiny.pt")
    torch.manual_seed(g["seed"])
    return VideoToVideoDiffusion(g["config"]).eval().to(dev), g


def _staged(m, v, sampler, steps, K, depth, seed):
    """generate_ensemble restated with the existing ops, in the same RNG order"""
    from v2v_b200 import ops
    from v2v_b200.inference import DDIMSampler, DPMSolverSampler
    dev = v.device
    B = v.shape[0]
    cond = ops.upsample_depth(m.vae.encode(v), depth).repeat(K, 1, 1, 1, 1).contiguous()
    shape = tuple(cond.shape)
    torch.manual_seed(seed)
    if sampler == "ddim":
        z0 = DDIMSampler(m.diffusion, m.unet).sample(shape, cond, steps, dev, progress=False)
    elif sampler == "ddpm":
        torch.randn(shape, device=dev)
        dseed = int(torch.randint(0, 2 ** 62, ()))
        torch.manual_seed(seed)
        z0 = m.diffusion.p_sample_loop(m.unet, shape, cond, dev, progress=False, device_rng_seed=dseed)
    else:
        z0 = DPMSolverSampler(m.diffusion, m.unet).sample(shape, cond, steps, dev,
                                                          stochastic=sampler == "dpmpp_2m_sde", progress=False)
    return torch.stack([m.vae.decode(z0[k * B:(k + 1) * B].contiguous()) for k in range(K)])


def _check_stats(mean, std, members):
    ref = members.double()
    assert (mean.double() - ref.mean(0)).abs().max().item() <= 1e-6
    assert (std.double() - ref.std(0)).abs().max().item() <= 1e-6


@pytest.mark.parametrize("sampler", ["ddim", "dpmpp_2m", "dpmpp_2m_sde", "ddpm"])
def test_one_call_equals_staged_composition(cuda_dev, sampler):
    from v2v_b200.inference.ensemble import generate_ensemble
    m, _ = _tiny_model(cuda_dev)
    gen = torch.Generator().manual_seed(13)
    v = (torch.rand((2, 1, 8, 32, 32), generator=gen) * 2 - 1).to(cuda_dev)
    K = 3
    torch.manual_seed(6)
    mean, std, members = generate_ensemble(m, v, sampler, 20, K, target_depth=48, return_members=True)
    assert members.shape == (K, 2, 1, 48, 32, 32) and mean.shape == std.shape == (2, 1, 48, 32, 32)
    assert torch.isfinite(members).all() and m.last_nan_flag.item() == 0
    assert torch.equal(members, _staged(m, v, sampler, 20, K, 48, 6))
    _check_stats(mean, std, members)
    assert std.max().item() > 0  # the members differ
    torch.manual_seed(6)
    mean2, std2, members2 = generate_ensemble(m, v, sampler, 20, K, target_depth=48, return_members=True)
    assert torch.equal(members2, members) and torch.equal(mean2, mean) and torch.equal(std2, std)
    torch.manual_seed(6)
    mean3, std3 = generate_ensemble(m, v, sampler, 20, K, target_depth=48)  # members in the object's scratch
    assert torch.equal(mean3, mean) and torch.equal(std3, std)


def _cfg_ddim(m, steps, keep):
    from v2v_b200 import _lib
    from v2v_b200.inference.sampler import _schedule
    ts, acp = _schedule(m.diffusion, steps)
    keep += [ts, acp]
    cfg = _lib.SamplerCfg()
    cfg.sampler, cfg.n, cfg.n_train, cfg.eta = 0, len(ts), acp.numel(), 0.0
    cfg.timesteps = ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    cfg.alphas_cumprod = ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float))
    return cfg


def test_identical_members_have_zero_std(cuda_dev):
    from v2v_b200 import _lib
    m, _ = _tiny_model(cuda_dev)
    gen = torch.Generator().manual_seed(21)
    v = (torch.rand((1, 1, 4, 16, 16), generator=gen) * 2 - 1).to(cuda_dev)
    K = 3
    keep = []
    cfg = _cfg_ddim(m, 8, keep)
    z_init = torch.randn((1, 4, 12, 4, 4), generator=gen).to(cuda_dev).repeat(K, 1, 1, 1, 1).contiguous()
    members = torch.empty((K, 1, 1, 12, 16, 16), device=cuda_dev)
    mean, std = torch.empty((1, 1, 12, 16, 16), device=cuda_dev), torch.empty((1, 1, 12, 16, 16), device=cuda_dev)
    _lib.check(_lib.lib().b2v_generate_ensemble(
        m.unet.native(cuda_dev), m.vae.native(cuda_dev), ctypes.byref(cfg), _lib.dptr(v), _lib.dptr(z_init), K,
        _lib.dptr(members), _lib.dptr(mean), _lib.dptr(std), 1, 4, 12, 16, 16, None, _lib.stream()), "generate_ensemble")
    torch.cuda.synchronize()
    assert std.abs().max().item() <= 1e-6
    assert torch.equal(mean, members[0])


@pytest.mark.parametrize("K", [2, 3, 8])
@pytest.mark.parametrize("n", [1001, 4 * 12345])
def test_ensemble_stats_matches_torch_fp64(cuda_dev, K, n):
    from v2v_b200 import ops
    g = torch.Generator().manual_seed(K * 7 + n)
    x = (torch.randn((K, n), generator=g) * 0.5 + 0.1).to(cuda_dev)
    mean, std = ops.ensemble_stats(x)
    assert mean.shape == std.shape == (n,)
    _check_stats(mean, std, x)
    m2, s2 = ops.ensemble_stats(x)
    assert torch.equal(m2, mean) and torch.equal(s2, std)
    # an odd-sized view at an unaligned offset takes the element-wise path and gives the same values
    y = torch.empty(K * n + 1, device=cuda_dev)[1:].view(K, n)
    y.copy_(x)
    m3, s3 = ops.ensemble_stats(y)
    assert torch.equal(m3, mean) and torch.equal(s3, std)


def test_full_shape_dpmpp10_k4(cuda_dev):
    import yaml
    from v2v_b200.inference.ensemble import generate_ensemble
    from v2v_b200.models import VideoToVideoDiffusion
    cfg = yaml.safe_load(open(os.path.join(os.path.dirname(__file__), "golden", "slice_interpolation_full_medium.yaml")))
    torch.manual_seed(0)
    m = VideoToVideoDiffusion(cfg).eval().to(cuda_dev)
    g = torch.Generator().manual_seed(1234)
    v = (torch.rand((1, 1, 8, 192, 192), generator=g) * 2 - 1).to(cuda_dev)
    torch.manual_seed(42)
    mean, std, members = generate_ensemble(m, v, "dpmpp_2m", 10, 4, target_depth=48, return_members=True)
    assert members.shape == (4, 1, 1, 48, 192, 192)
    assert torch.equal(members, _staged(m, v, "dpmpp_2m", 10, 4, 48, 42))
    assert torch.isfinite(mean).all() and torch.isfinite(std).all()
    assert mean.abs().max().item() <= 1.0 and std.min().item() >= 0.0
    assert m.last_nan_flag.item() == 0
    _check_stats(mean, std, members)
    print(f"full shape, K = 4, dpmpp_2m-10: mean std {std.mean().item():.4f}, max std {std.max().item():.4f}")


def test_nan_flag_like_generate(cuda_dev):
    from v2v_b200.inference.ensemble import generate_ensemble
    m, _ = _tiny_model(cuda_dev)
    gen = torch.Generator().manual_seed(3)
    v = (torch.rand((1, 1, 4, 16, 16), generator=gen) * 2 - 1).to(cuda_dev)
    for poison in (False, True):
        x = v.clone()
        if poison:
            x[0, 0, 1, 5, 7] = float("nan")
        m.generate(x, "dpmpp_2m", 5, target_depth=12)
        want = m.last_nan_flag.item()
        mean, std = generate_ensemble(m, x, "dpmpp_2m", 5, 2, target_depth=12)
        assert m.last_nan_flag.item() == want == int(poison)
        assert torch.isfinite(mean).all() and torch.isfinite(std).all()


def test_invalid_arguments_launch_nothing(cuda_dev):
    from v2v_b200 import _lib
    m, _ = _tiny_model(cuda_dev)
    L = _lib.lib()
    u, vh = m.unet.native(cuda_dev), m.vae.native(cuda_dev)
    v_in = torch.zeros((1, 1, 2, 16, 16), device=cuda_dev)
    z = torch.zeros((2, 4, 6, 4, 4), device=cuda_dev)
    mean = torch.empty((1, 1, 6, 16, 16), device=cuda_dev)
    std = torch.empty_like(mean)
    acp = m.diffusion.alphas_cumprod.detach().float().cpu().contiguous()
    good = np.array([999, 500, 0], dtype=np.int64)
    unsorted = np.array([500, 999, 0], dtype=np.int64)
    cfg = _lib.SamplerCfg()
    cfg.n, cfg.n_train = 3, acp.numel()
    cfg.alphas_cumprod = ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float))

    def call(code=2, K=2, ts=good, mn=mean, sd=std, H=16):
        cfg.sampler = code
        cfg.timesteps = ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
        return L.b2v_generate_ensemble(u, vh, ctypes.byref(cfg), _lib.dptr(v_in), _lib.dptr(z), K, None,
                                       _lib.dptr(mn), _lib.dptr(sd), 1, 2, 6, H, 16, None, _lib.stream())

    torch.cuda.synchronize()
    n0 = _lib.launch_count()
    for what, kw, phrase in (("K = 1", dict(K=1), "K >= 2"),
                             ("null mean", dict(mn=None), "null argument"),
                             ("null std", dict(sd=None), "null argument"),
                             ("unknown sampler", dict(code=7), "unknown sampler"),
                             ("sde without noise", dict(code=3), "noise"),
                             ("unsorted timesteps", dict(ts=unsorted), "decreasing"),
                             ("H % 4", dict(H=18), "bad shape")):
        assert call(**kw) != 0, what
        assert phrase in _lib.last_error(), (what, _lib.last_error())
    assert L.b2v_ensemble_stats(_lib.dptr(z), _lib.dptr(mean), _lib.dptr(std), 1, 16, _lib.stream()) != 0
    assert "K >= 2" in _lib.last_error()
    assert _lib.launch_count() == n0


def test_generate_volume_ensemble(cuda_dev):
    from v2v_b200 import ops
    from v2v_b200.inference.ensemble import generate_ensemble
    from v2v_b200.inference.volume import generate_volume, window_starts
    m, _ = _tiny_model(cuda_dev)
    gen = torch.Generator().manual_seed(19)
    vol = (torch.rand((1, 1, 4, 32, 32), generator=gen) * 2 - 1).to(cuda_dev)
    kw = dict(patch_size=(2, 16, 16), target_patch_size=(6, 16, 16), stride=(2, 8, 8), batch=3)
    torch.manual_seed(9)
    mean, std = generate_volume(m, vol, "dpmpp_2m", 4, num_samples=2, **kw)
    assert mean.shape == std.shape == (1, 1, 12, 32, 32)
    assert torch.isfinite(mean).all() and mean.abs().max() <= 1.0 and std.min() >= 0 and std.max() > 0

    def compose(fn):
        """the per-window composition: windows in reference order, `batch` at a time, Gaussian-blended"""
        items = window_starts(4, 32, 32, kw["patch_size"], kw["stride"])
        acc = [torch.zeros((1, 1, 12, 32, 32), device=cuda_dev) for _ in range(2)]
        wsum = [torch.zeros_like(acc[0]) for _ in range(2)]
        win = tuple(ops.gaussian_window_1d(n, cuda_dev) for n in (6, 16, 16))
        for i in range(0, len(items), 3):
            chunk = items[i:i + 3]
            x = torch.stack([vol[0, :, d0:d0 + 2, h0:h0 + 16, w0:w0 + 16] for d0, h0, w0 in chunk]).contiguous()
            outs = fn(x)
            for j, (d0, h0, w0) in enumerate(chunk):
                for o, a, w in zip(outs, acc, wsum):
                    ops.stitch_accumulate(o[j:j + 1], a, w, d0 * 3, h0, w0, win)
        return [ops.stitch_normalize(a, w) for a, w in zip(acc[:len(outs)], wsum)]

    torch.manual_seed(9)
    ref_mean, ref_std = compose(lambda x: generate_ensemble(m, x, "dpmpp_2m", 4, 2, target_depth=6))
    assert torch.equal(mean, ref_mean) and torch.equal(std, ref_std)
    # two ranks (run one after the other: the same RNG stream as one rank, since batch 3 splits 18 windows evenly)
    torch.manual_seed(9)
    parts = [generate_volume(m, vol, "dpmpp_2m", 4, num_samples=2, rank=r, world=2, **kw) for r in range(2)]
    wsum = parts[0][2] + parts[1][2]
    for i, single in ((0, mean), (1, std)):
        merged = ops.stitch_normalize(parts[0][i] + parts[1][i], wsum)
        assert (merged - single).abs().max().item() <= 2e-6
    # num_samples=None: the single-sample volume, unchanged
    torch.manual_seed(9)
    one = generate_volume(m, vol, "dpmpp_2m", 4, **kw)
    torch.manual_seed(9)
    (ref_one,) = compose(lambda x: (m.generate(x, "dpmpp_2m", 4, target_depth=6),))
    assert torch.equal(one, ref_one)
