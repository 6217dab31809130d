"""UniPC on the B200: the update kernel bit for bit against the fp32 eager chain on its vector and element-wise paths,
the whole-loop C entry against the step-wise loop, the DDIM gates of DESIGN.md section 2 at the benchmark shape against
the fp32 oracle trajectory (tests/unipc_oracle.py over oracle/ref_port.py's U-Net), softmax attention mode, generate()
and generate_ensemble() against their staged composition, the wrappers, and argument errors that launch nothing."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import unipc_oracle as O
from helpers import TINY_UNET, golden, rel_l2, tiny_unet
from oracle import ref_port as R

pytestmark = pytest.mark.gpu
EPS_TOL = 1e-2


def _sd(m, dev):
    return {k: v.to(dev) for k, v in m.state_dict().items()}


def _acp():
    from v2v_b200.models import GaussianDiffusion
    return GaussianDiffusion("cosine", 1000).alphas_cumprod.float()


def _rows(ts, order=3, variant="bh2"):
    from v2v_b200.inference.sampler import unipc_coefficients
    return unipc_coefficients(np.asarray(ts, dtype=np.int64), _acp(), order, variant)


def _guard(x):
    return torch.nan_to_num(x, nan=0.0, posinf=1.0, neginf=-1.0)


def _eager_chain(z, xcp, hist, eps, row, step):
    """the kernel's stated fp32 operation order as torch eager ops (fp32 0-dim coefficients); zero weights skipped"""
    r = row.to(z.device)
    e = _guard(eps)
    m = torch.clamp(_guard((z - r[0] * e) / r[1]), -r[12], r[12])
    ms = [m] + [hist[(step - j) % 4] for j in (1, 2, 3)]

    def acc(terms):
        a = torch.zeros_like(z)
        for w, v in terms:
            if float(row[w]) != 0.0:
                a = a + r[w] * v
        return a

    x = _guard(acc([(2, z), (3, xcp), (4, ms[0]), (5, ms[1]), (6, ms[2]), (7, ms[3])]))
    zn = _guard(acc([(8, x), (9, ms[0]), (10, ms[1]), (11, ms[2])]))
    return zn, x, m


def _check_update(shape, offset, dev, g):
    """every row kind of a UniPC-3 loop: z, xc, the written slot bitwise, the other slots untouched; injected NaN/Inf
    guarded and flagged; NaN-filled unread slots and x^c_prev do not leak.  offset > 0 misaligns every pointer."""
    from v2v_b200 import ops
    ts = [999, 980, 960, 700, 500, 300, 0]
    rows = {"bh2": _rows(ts, 3, "bh2"), "bh1": _rows(ts, 3, "bh1"), "o1": _rows(ts, 1, "bh2")}
    cases = [("bh2", 0), ("bh2", 1), ("bh2", 2), ("bh2", 3), ("bh2", 5), ("bh2", 6), ("bh1", 3), ("bh1", 4),
             ("o1", 1), ("o1", 6)]
    n = int(np.prod(shape))

    def buf(k):  # k tensors of `shape` at `offset` floats into a fresh allocation
        t = torch.empty(offset + k * n, device=dev)[offset:].view((k,) + shape) if k > 1 else \
            torch.empty(offset + n, device=dev)[offset:].view(shape)
        return t

    for name, step in cases:
        row = rows[name][step]
        z, eps, xcp, hist = buf(1), buf(1), buf(1), buf(4)
        z.copy_(torch.randn(shape, generator=g) * 3)
        eps.copy_(torch.randn(shape, generator=g))
        xcp.copy_(torch.randn(shape, generator=g))
        hist.copy_(torch.randn((4,) + shape, generator=g))
        for inject in (False, True):
            if inject:  # non-finite eps / z: guarded like ddim_update, and flagged
                eps.view(-1)[:3] = torch.tensor([float("nan"), float("inf"), -float("inf")])
                z.view(-1)[5:8] = torch.tensor([float("nan"), float("inf"), -float("inf")])
            want_z, want_x, want_m = _eager_chain(z, xcp, hist, eps, row, step)
            z1, x1, h1 = buf(1), buf(1), buf(4)
            z1.copy_(z)
            x1.copy_(xcp)
            h1.copy_(hist)
            flag = ops.unipc_update(z1, x1, h1, eps, row.to(dev), step)
            assert torch.equal(z1, want_z) and torch.equal(x1, want_x), (name, step, inject, offset)
            assert torch.equal(h1[step % 4], want_m), (name, step, inject)
            for s in range(4):
                if s != step % 4:
                    assert torch.equal(h1[s], hist[s]), (name, step, s)
            assert flag.item() == int(inject) and torch.isfinite(z1).all(), (name, step, inject)
        if step == 0:  # t = 999: alpha = 1.6e-5, the +-10 clamp fires
            assert (want_m.abs() == 10.0).any()
        # weights that are zero: their operands are not read (all NaN must not matter)
        z2, x2, h2 = buf(1), buf(1), buf(4)
        z2.copy_(z)
        x2.copy_(xcp if float(row[3]) != 0.0 else torch.full(shape, float("nan"), device=dev))
        h2.copy_(hist)
        for j, weights in ((1, (5, 10)), (2, (6, 11)), (3, (7,))):
            if all(float(row[w]) == 0.0 for w in weights):
                h2[(step - j) % 4] = float("nan")
        want_z, want_x, want_m = _eager_chain(z, x2, h2, eps, row, step)
        assert torch.isfinite(want_z).all() and torch.isfinite(want_x).all()
        flag = ops.unipc_update(z2, x2, h2, eps, row.to(dev), step)
        assert torch.equal(z2, want_z) and torch.equal(x2, want_x) and torch.equal(h2[step % 4], want_m), (name, step)
        assert flag.item() == 1  # the injected values above are still in eps / z


@pytest.mark.parametrize("path", ["vector", "elementwise_n_odd", "elementwise_misaligned"])
def test_update_kernel_bit_exact_guards_and_unread_slots(cuda_dev, path):
    g = torch.Generator().manual_seed(3)
    shape, offset = {"vector": ((2, 4, 6, 8, 8), 0), "elementwise_n_odd": ((3, 1, 5, 7, 7), 0),
                     "elementwise_misaligned": ((2, 4, 6, 8, 8), 1)}[path]
    _check_update(shape, offset, cuda_dev, g)


def test_update_rejects_bad_history_shape(cuda_dev):
    from v2v_b200 import ops
    z = torch.zeros((2, 8), device=cuda_dev)
    with pytest.raises(ValueError, match="hist"):
        ops.unipc_update(z, z.clone(), torch.zeros((3, 2, 8), device=cuda_dev), z.clone(),
                         torch.zeros(16, device=cuda_dev), 0)


@pytest.mark.parametrize("variant", ["bh1", "bh2"])
@pytest.mark.parametrize("order", [1, 2, 3])
def test_whole_loop_equals_stepwise_loop(cuda_dev, order, variant):
    from v2v_b200 import _lib, ops
    from v2v_b200.inference import UniPCSampler
    from v2v_b200.models import GaussianDiffusion
    m = tiny_unet(0).to(cuda_dev)
    diff = GaussianDiffusion("cosine", 1000)
    ts = np.ascontiguousarray(UniPCSampler(diff, m)._get_timesteps(5), dtype=np.int64)
    assert ts.tolist() == [999, 800, 600, 400, 200, 0]
    n = len(ts)
    cond = golden("ddim_tiny.pt")["cond"].to(cuda_dev)
    shape = (1, 4, 4, 8, 8)
    g = torch.Generator().manual_seed(21)
    z_init = torch.randn(shape, generator=g).to(cuda_dev)
    z_keep = z_init.clone()
    acp = diff.alphas_cumprod.float().contiguous()
    L, h = _lib.lib(), m.native(cuda_dev)
    var = {"bh1": 0, "bh2": 1}[variant]

    def whole():
        out, flag = torch.empty_like(z_init), torch.zeros(1, dtype=torch.int32, device=cuda_dev)
        _lib.check(L.b2v_unipc_sample(h, _lib.dptr(z_init), _lib.dptr(cond), _lib.dptr(out), *shape[:1], *shape[2:],
                                      ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), n,
                                      ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float)), acp.numel(), order,
                                      var, _lib.dptr(flag, torch.int32), _lib.stream()), "unipc_sample")
        return out, flag

    a, flag = whole()
    b, _ = whole()
    assert torch.equal(a, b) and flag.item() == 0
    assert torch.equal(z_init, z_keep)
    rows = _rows(ts, order, variant).to(cuda_dev)

    def stepwise(z0):
        z, xc, hist = z0.clone(), torch.empty_like(z0), torch.empty((4,) + shape, device=cuda_dev)
        for i, t in enumerate(ts):
            eps = m(z, torch.tensor([int(t)], device=cuda_dev), cond)
            ops.unipc_update(z, xc, hist, eps, rows[i].contiguous(), i)
        return z

    assert torch.equal(a, stepwise(z_init))
    # the oracle's loop over the fp32 U-Net, free-running through the t = 999 clamp: a loose sanity bound only
    sd = _sd(m, cuda_dev)
    with torch.no_grad():
        ref = O.sample_timesteps(lambda zz, tt, cc: R.unet_forward(sd, TINY_UNET, zz, tt, cc), acp, ts, z_init, cond,
                                 order, variant)
    print(f"tiny U-Net, UniPC-{order} {variant} 6 steps: rel-L2 vs fp32 oracle {rel_l2(a, ref):.2e}")
    assert rel_l2(a, ref) < 0.2
    # the sampler class: same RNG order (z only), same call; any callable model: the Python loop over the same kernel
    torch.manual_seed(4)
    s1 = UniPCSampler(diff, m).sample(shape, cond, 5, cuda_dev, order=order, variant=variant, progress=False)
    torch.manual_seed(4)
    assert torch.equal(s1, stepwise(torch.randn(shape, device=cuda_dev)))
    torch.manual_seed(4)
    s2 = UniPCSampler(diff, lambda zz_, tt, cc: m(zz_, tt, cc)).sample(shape, cond, 5, cuda_dev, order=order,
                                                                      variant=variant, progress=False)
    assert torch.equal(s2, s1)


# ------------------------------------------------------------------------------------- benchmark shape
@pytest.fixture(scope="module")
def bench_model(cuda_dev):
    import yaml
    from v2v_b200.models import VideoToVideoDiffusion
    cfg = yaml.safe_load(open(os.path.join(os.path.dirname(__file__), "golden", "slice_interpolation_full_medium.yaml")))
    torch.manual_seed(0)
    m = VideoToVideoDiffusion(cfg).eval().to(cuda_dev)
    return m, cfg


@pytest.mark.timeout(2400)
def test_generate_unipc20_batch4_all_gates(cuda_dev, bench_model):
    """BASELINE configs[1] (batch 4, 8 -> 48 slices at 192^2) with 20 steps = 21 U-Net evaluations of UniPC-3/bh2, the
    DDIM gates of DESIGN.md section 2 against the fp32 oracle trajectory (tests/unipc_oracle.py over oracle/ref_port.py):
      1. teacher-forced eps rel-L2 <= 1e-2 at every one of the 21 steps;  2. decode of the oracle z_0 >= 60 dB;
      3. |PSNR(new, target) - PSNR(ref, target)| <= 0.05 dB;  4. a second run with the same seed gives the same bits."""
    from v2v_b200.inference import UniPCSampler
    m, cfg = bench_model
    sd = _sd(m, cuda_dev)
    vae_cfg, unet_cfg, _ = R.resolve_config(cfg)
    batch, steps = 4, 20
    g = torch.Generator().manual_seed(1234)
    v_thick = (torch.rand((batch, 1, 8, 192, 192), generator=g) * 2 - 1).to(cuda_dev)
    target = (torch.rand((batch, 1, 48, 192, 192), generator=g) * 2 - 1).to(cuda_dev)
    ts = UniPCSampler(m.diffusion, m.unet)._get_timesteps(steps)
    acp = m.diffusion.alphas_cumprod.detach().float().cpu()
    torch.manual_seed(42)
    with torch.no_grad():  # generate() restated piece by piece, in the same RNG order
        z_in = R.vae_encode(sd, v_thick, vae_cfg["scaling_factor"], "vae.")
        cond = F.interpolate(z_in, size=(48, z_in.shape[3], z_in.shape[4]), mode="trilinear", align_corners=False)
        shape = tuple(cond.shape)
        torch.randn(shape, device=cuda_dev)  # discarded draw (models/model.py:303)
        z_init = torch.randn(shape, device=cuda_dev)
        rec = []
        model = lambda z, t, c: R.unet_forward(sd, unet_cfg, z, t, c, "unet.")  # noqa: E731
        z0 = O.sample_timesteps(model, acp, ts, z_init, cond, 3, "bh2", record=rec)
        ref = R.vae_decode(sd, z0, vae_cfg["scaling_factor"], "vae.")
    assert len(rec) == 21 and rec[0][1] == 999 and rec[-1][1] == 0
    errs = []
    for z_t, t_idx, eps_ref in rec:
        errs.append(rel_l2(m.unet(z_t, torch.full((batch,), t_idx, device=cuda_dev, dtype=torch.long), cond), eps_ref))
    del rec
    print(f"unipc-20, batch 4: teacher-forced eps rel-L2 over 21 steps: max {max(errs):.3e} "
          f"(t={ts[errs.index(max(errs))]}), mean {sum(errs) / len(errs):.3e}")
    assert max(errs) <= EPS_TOL, errs
    n = lambda v: (v.clamp(-1, 1) + 1) / 2  # noqa: E731
    p_dec = R.psnr(n(m.vae.decode(z0)), n(ref))
    print(f"unipc-20, batch 4: teacher-forced decode PSNR(new, ref) = {p_dec:.1f} dB")
    assert p_dec >= 60.0, p_dec
    torch.manual_seed(42)
    got = m.generate(v_thick, "unipc", steps, target_depth=48)
    assert got.shape == ref.shape == (batch, 1, 48, 192, 192) and torch.isfinite(got).all()
    p_new, p_ref, p_direct = R.psnr(n(got), n(target)), R.psnr(n(ref), n(target)), R.psnr(n(got), n(ref))
    print(f"unipc-20, batch 4: generate PSNR(new,target)={p_new:.4f} PSNR(ref,target)={p_ref:.4f} "
          f"PSNR(new,ref)={p_direct:.2f} dB")
    assert abs(p_new - p_ref) <= 0.05, (p_new, p_ref)
    assert m.last_nan_flag.item() == 0
    torch.manual_seed(42)
    assert torch.equal(m.generate(v_thick, "unipc", steps, target_depth=48), got)


def test_softmax_mode_teacher_forced_against_softmax_oracle(cuda_dev):
    import softmax_oracle as S
    from v2v_b200.inference import UniPCSampler
    from v2v_b200.models import GaussianDiffusion, UNet3D
    torch.manual_seed(0)
    m = UNet3D(**TINY_UNET).eval().to(cuda_dev).set_attention_mode("softmax")
    sd = _sd(m, cuda_dev)
    diff = GaussianDiffusion("cosine", 1000)
    ts = UniPCSampler(diff, m)._get_timesteps(10)
    g = torch.Generator().manual_seed(8)
    shape = (2, 4, 12, 8, 8)
    cond = torch.randn(shape, generator=g).to(cuda_dev)
    z_init = torch.randn(shape, generator=g).to(cuda_dev)
    rec = []
    with torch.no_grad():
        ref = O.sample_timesteps(lambda z, t, c: S.unet_forward(sd, TINY_UNET, z, t, c), diff.alphas_cumprod.float(), ts,
                                 z_init, cond, record=rec)
    errs = [rel_l2(m(z_t, torch.full((2,), t, device=cuda_dev, dtype=torch.long), cond), e) for z_t, t, e in rec]
    print(f"softmax mode, tiny U-Net, UniPC-3 bh2 11 steps teacher-forced: max eps rel-L2 {max(errs):.3e}")
    assert max(errs) <= EPS_TOL, errs
    torch.manual_seed(1)
    out = UniPCSampler(diff, m).sample(shape, cond, 10, cuda_dev, progress=False)
    assert torch.isfinite(out).all()
    torch.manual_seed(1)
    z_same = torch.randn(shape, device=cuda_dev)  # the sampler's initial draw
    with torch.no_grad():
        ref = O.sample_timesteps(lambda z, t, c: S.unet_forward(sd, TINY_UNET, z, t, c), diff.alphas_cumprod.float(), ts,
                                 z_same, cond)
    print(f"softmax mode, UniPC-3 bh2 11 steps free-running: rel-L2 vs the softmax oracle {rel_l2(out, ref):.2e}")
    assert rel_l2(out, ref) < 0.2


# ------------------------------------------------------------------------------------- generate() and wrappers
def _tiny_model(dev, **extra):
    from v2v_b200.models import VideoToVideoDiffusion
    g = golden("generate_tiny.pt")
    torch.manual_seed(g["seed"])
    return VideoToVideoDiffusion(dict(g["config"], **extra)).eval().to(dev), g


def test_generate_equals_staged_composition(cuda_dev):
    from v2v_b200 import ops
    from v2v_b200.inference import UniPCSampler
    m, _ = _tiny_model(cuda_dev)
    gen = torch.Generator().manual_seed(13)
    v = (torch.rand((2, 1, 8, 32, 32), generator=gen) * 2 - 1).to(cuda_dev)
    torch.manual_seed(6)
    got = m.generate(v, "unipc", 20, target_depth=48)
    assert got.shape == (2, 1, 48, 32, 32) and torch.isfinite(got).all() and m.last_nan_flag.item() == 0
    torch.manual_seed(6)
    cond = ops.upsample_depth(m.vae.encode(v), 48)
    torch.randn(tuple(cond.shape), device=cuda_dev)  # the reference's discarded draw
    z0 = UniPCSampler(m.diffusion, m.unet).sample(tuple(cond.shape), cond, 20, cuda_dev, progress=False)
    assert torch.equal(got, m.vae.decode(z0))
    torch.manual_seed(6)
    assert torch.equal(m.generate(v, "unipc", 20, target_depth=48), got)
    # the DPM-Solver++ program of the same shape is unaffected by a UniPC run on it (and the other way round)
    torch.manual_seed(6)
    d1 = m.generate(v, "dpmpp_2m", 20, target_depth=48)
    torch.manual_seed(6)
    assert torch.equal(m.generate(v, "unipc", 20, target_depth=48), got)
    torch.manual_seed(6)
    assert torch.equal(m.generate(v, "dpmpp_2m", 20, target_depth=48), d1)


def test_generate_ensemble_equals_staged_composition(cuda_dev):
    from v2v_b200 import ops
    from v2v_b200.inference import UniPCSampler
    from v2v_b200.inference.ensemble import generate_ensemble
    m, _ = _tiny_model(cuda_dev)
    gen = torch.Generator().manual_seed(13)
    v = (torch.rand((2, 1, 8, 32, 32), generator=gen) * 2 - 1).to(cuda_dev)
    K = 3
    torch.manual_seed(6)
    mean, std, members = generate_ensemble(m, v, "unipc", 20, K, target_depth=48, return_members=True)
    assert members.shape == (K, 2, 1, 48, 32, 32) and torch.isfinite(members).all() and m.last_nan_flag.item() == 0
    cond = ops.upsample_depth(m.vae.encode(v), 48).repeat(K, 1, 1, 1, 1).contiguous()
    torch.manual_seed(6)
    z0 = UniPCSampler(m.diffusion, m.unet).sample(tuple(cond.shape), cond, 20, cuda_dev, progress=False)
    staged = torch.stack([m.vae.decode(z0[k * 2:(k + 1) * 2].contiguous()) for k in range(K)])
    assert torch.equal(members, staged)
    ref = members.double()
    assert (mean.double() - ref.mean(0)).abs().max().item() <= 1e-6
    assert (std.double() - ref.std(0)).abs().max().item() <= 1e-6 and std.max().item() > 0


def test_generate_batch_and_generate_volume(cuda_dev):
    from v2v_b200.inference import UniPCSampler
    from v2v_b200.inference.generate import generate_batch
    from v2v_b200.inference.volume import generate_volume
    m, _ = _tiny_model(cuda_dev)
    gen = torch.Generator().manual_seed(17)
    vids = torch.rand((2, 1, 3, 16, 24), generator=gen) * 2 - 1
    torch.manual_seed(8)
    got = generate_batch(m, vids, sampler_type="unipc", num_inference_steps=6, device=cuda_dev)
    assert got.shape == (2, 1, 3, 16, 24) and torch.isfinite(got).all()
    torch.manual_seed(8)
    z_in = m.vae.encode(vids.to(cuda_dev))
    z0 = UniPCSampler(m.diffusion, m.unet).sample(z_in.shape, z_in, 6, cuda_dev, progress=False)
    assert torch.equal(got, m.vae.decode(z0))
    vol = (torch.rand((1, 1, 4, 32, 32), generator=gen) * 2 - 1).to(cuda_dev)
    torch.manual_seed(9)
    full = generate_volume(m, vol, "unipc", 4, patch_size=(2, 16, 16), target_patch_size=(6, 16, 16),
                           stride=(2, 8, 8), batch=4)
    assert full.shape == (1, 1, 12, 32, 32) and torch.isfinite(full).all() and full.abs().max() <= 1.0


def test_invalid_arguments_launch_nothing(cuda_dev):
    from v2v_b200 import _lib, ops
    from v2v_b200.inference import UniPCSampler
    m, g = _tiny_model(cuda_dev)
    L = _lib.lib()
    u, vh = m.unet.native(cuda_dev), m.vae.native(cuda_dev)
    shape = (1, 4, 6, 4, 4)
    z = torch.randn(shape, device=cuda_dev)
    out = torch.empty_like(z)
    acp = m.diffusion.alphas_cumprod.detach().float().cpu().contiguous()
    acp_p = ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float))
    good = np.array([999, 500, 0], dtype=np.int64)
    unsorted = np.array([500, 999, 0], dtype=np.int64)
    torch.cuda.synchronize()
    n0 = _lib.launch_count()

    def sample(ts, order, variant):
        return L.b2v_unipc_sample(u, _lib.dptr(z), _lib.dptr(z), _lib.dptr(out), 1, 6, 4, 4,
                                  ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), len(ts), acp_p, acp.numel(), order,
                                  variant, None, _lib.stream())

    for what, args, phrase in (("order 4", (good, 4, 1), "order"), ("order 0", (good, 0, 1), "order"),
                               ("variant 2", (good, 3, 2), "variant"),
                               ("unsorted timesteps", (unsorted, 3, 1), "decreasing")):
        assert sample(*args) != 0, what
        assert phrase in _lib.last_error(), (what, _lib.last_error())
    for kw in (dict(order=4), dict(variant="bh3")):
        with pytest.raises(ValueError):
            UniPCSampler(m.diffusion, m.unet).sample(shape, z, 5, cuda_dev, **kw)
    p = _lib.dptr(z)
    assert L.b2v_unipc_update(p, p, None, p, p, 0, z.numel(), None, _lib.stream()) != 0
    assert L.b2v_unipc_update(p, p, p, p, p, -1, z.numel(), None, _lib.stream()) != 0
    with pytest.raises(ValueError):
        ops.unipc_update(z, z.clone(), torch.zeros((4, 1), device=cuda_dev), z, torch.zeros(16, device=cuda_dev), 0)
    v_in = g["v_in"].to(cuda_dev).contiguous()
    cfg = _lib.SamplerCfg()
    cfg.sampler, cfg.n, cfg.n_train = 4, len(good), acp.numel()
    cfg.timesteps = good.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    cfg.alphas_cumprod = acp_p
    vout = torch.empty((1, 1, 6, 16, 16), device=cuda_dev)

    def generate(order, variant, code=4):
        cfg.sampler, cfg.unipc_order, cfg.unipc_variant = code, order, variant
        return L.b2v_generate(u, vh, ctypes.byref(cfg), _lib.dptr(v_in), _lib.dptr(z), _lib.dptr(vout), 1, 2, 6, 16, 16,
                              None, _lib.stream())

    assert generate(3, 1, code=5) != 0 and "4 = unipc" in _lib.last_error()
    assert generate(0, 1) != 0 and "order" in _lib.last_error()
    assert generate(3, 5) != 0 and "variant" in _lib.last_error()
    cfg.timesteps = unsorted.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    assert generate(3, 1) != 0 and "decreasing" in _lib.last_error()
    assert _lib.launch_count() == n0
