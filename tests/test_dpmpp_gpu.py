"""DPM-Solver++(2M) on the B200: the update kernel bit for bit against the fp32 eager chain, its first-order identity with
DDIM, the whole-loop C entry against the step-wise loop, the DDIM gates of DESIGN.md section 2 at the benchmark shape
against the fp32 oracle trajectory (tests/dpmpp_oracle.py over oracle/ref_port.py's U-Net), softmax attention mode,
generate() and its wrappers, and argument errors that launch nothing."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

import dpmpp_oracle as O
from helpers import TINY_UNET, golden, rel_l2, tiny_unet
from oracle import ref_port as R

pytestmark = pytest.mark.gpu
EPS_TOL = 1e-2


def _sd(m, dev):
    return {k: v.to(dev) for k, v in m.state_dict().items()}


def _acp():
    from v2v_b200.models import GaussianDiffusion
    return GaussianDiffusion("cosine", 1000).alphas_cumprod.float()


def _rows(ts, order=2, sde=False):
    from v2v_b200.inference.sampler import dpmpp_coefficients
    return dpmpp_coefficients(np.asarray(ts, dtype=np.int64), _acp(), order, sde)


def _guard(x):
    return torch.nan_to_num(x, nan=0.0, posinf=1.0, neginf=-1.0)


def _eager_chain(z, x0_prev, eps, row, noise):
    """the kernel's stated fp32 operation order as torch eager ops (fp32 0-dim coefficients)"""
    r = row.to(z.device)
    e = _guard(eps)
    x0 = torch.clamp(_guard((z - r[0] * e) / r[1]), -r[7], r[7])
    D = x0 if float(row[5]) == 0.0 else r[4] * x0 + r[5] * x0_prev
    zn = r[2] * z + r[3] * D
    if float(row[6]) != 0.0:
        zn = zn + r[6] * noise
    return _guard(zn), x0


def test_update_kernel_bit_exact_guards_and_unread_x0_prev(cuda_dev):
    from v2v_b200 import ops
    g = torch.Generator().manual_seed(3)
    shape = (2, 4, 6, 8, 8)
    ts = [999, 980, 960, 500, 0]
    cases = {"order1_first": _rows(ts, 2)[0], "order2": _rows(ts, 2)[2], "order1_row": _rows(ts, 1)[3],
             "sde_order2": _rows(ts, 2, True)[2], "sde_first": _rows(ts, 2, True)[0], "last": _rows(ts, 2)[4]}
    assert float(cases["order2"][5]) != 0.0 and float(cases["sde_order2"][6]) != 0.0
    for name, row in cases.items():
        z = (torch.randn(shape, generator=g) * 3).to(cuda_dev)
        eps = torch.randn(shape, generator=g).to(cuda_dev)
        x0p = torch.randn(shape, generator=g).to(cuda_dev)
        nz = torch.randn(shape, generator=g).to(cuda_dev)
        want_z, want_x0 = _eager_chain(z, x0p, eps, row, nz)
        z1, x1 = z.clone(), x0p.clone()
        flag = ops.dpmpp_update(z1, x1, eps, row.to(cuda_dev), nz)
        assert torch.equal(z1, want_z) and torch.equal(x1, want_x0), (name, (z1 - want_z).abs().max().item())
        assert flag.item() == 0, name
        if name in ("order1_first", "sde_first"):  # t = 999: alpha_t = 1.6e-5, the +-10 clamp fires
            assert (want_x0.abs() == 10.0).any(), name
        # non-finite eps / z: guarded like ddim_update, and flagged
        eb, zb = eps.clone(), z.clone()
        eb.view(-1)[:3] = torch.tensor([float("nan"), float("inf"), -float("inf")])
        zb.view(-1)[5:8] = torch.tensor([float("nan"), float("inf"), -float("inf")])
        want_z, want_x0 = _eager_chain(zb, x0p, eb, row, nz)
        z1, x1 = zb.clone(), x0p.clone()
        flag = ops.dpmpp_update(z1, x1, eb, row.to(cuda_dev), nz)
        assert torch.equal(z1, want_z) and torch.equal(x1, want_x0), name
        assert flag.item() == 1 and torch.isfinite(z1).all(), name
        # w1 == 0: x0_prev is not read (all NaN must not matter); c == 0: noise is not read
        if float(row[5]) == 0.0:
            z2, nanp = z.clone(), torch.full(shape, float("nan"), device=cuda_dev)
            flag = ops.dpmpp_update(z2, nanp, eps, row.to(cuda_dev), None if float(row[6]) == 0.0 else nz)
            want_z, want_x0 = _eager_chain(z, None, eps, row, nz)
            assert torch.equal(z2, want_z) and torch.equal(nanp, want_x0) and flag.item() == 0, name


def test_first_order_step_equals_ddim(cuda_dev):
    """order 1, ODE, t = 500 -> 480: algebraically the DDIM (eta 0) step; only DDIM's +1e-8 terms differ"""
    from v2v_b200 import ops
    acp = _acp()
    row = _rows([500, 480, 0], 1)[0]
    g = torch.Generator().manual_seed(5)
    z = torch.randn((2, 4, 8, 16, 16), generator=g).to(cuda_dev)
    eps = torch.randn((2, 4, 8, 16, 16), generator=g).to(cuda_dev)
    a_t, a_prev = acp[500], acp[480]
    coef = torch.zeros(8)
    coef[0], coef[1] = torch.sqrt(1 - a_t + 1e-8), torch.sqrt(a_t + 1e-8) + 1e-8
    coef[2], coef[3] = torch.sqrt(a_prev + 1e-8), torch.sqrt(1 - a_prev + 1e-8)
    zd = z.clone()
    ops.ddim_update(zd, eps, coef.to(cuda_dev))
    zp, x0p = z.clone(), torch.empty_like(z)
    ops.dpmpp_update(zp, x0p, eps, row.to(cuda_dev))
    assert (x0p.abs() < 10).all()  # the clamp does not fire here
    err = rel_l2(zp, zd)
    print(f"order-1 DPM-Solver++ vs DDIM step t=500->480: rel-L2 {err:.2e}")
    assert err <= 1e-6, err


@pytest.mark.parametrize("sde", [0, 1], ids=["ode", "sde"])
def test_whole_loop_equals_stepwise_loop(cuda_dev, sde):
    from v2v_b200 import _lib, ops
    from v2v_b200.inference import DPMSolverSampler
    from v2v_b200.models import GaussianDiffusion
    m = tiny_unet(0).to(cuda_dev)
    diff = GaussianDiffusion("cosine", 1000)
    ts = np.ascontiguousarray(DPMSolverSampler(diff, m)._get_timesteps(5), dtype=np.int64)
    assert ts.tolist() == [999, 800, 600, 400, 200, 0]
    n = len(ts)
    cond = golden("ddim_tiny.pt")["cond"].to(cuda_dev)
    shape = (1, 4, 4, 8, 8)
    g = torch.Generator().manual_seed(21)
    z_init = torch.randn(shape, generator=g).to(cuda_dev)
    z_keep = z_init.clone()
    noise = torch.randn((n,) + shape, generator=g).to(cuda_dev) if sde else None
    acp = diff.alphas_cumprod.float().contiguous()
    L, h = _lib.lib(), m.native(cuda_dev)

    def whole():
        out, flag = torch.empty_like(z_init), torch.zeros(1, dtype=torch.int32, device=cuda_dev)
        _lib.check(L.b2v_dpmpp_sample(h, _lib.dptr(z_init), _lib.dptr(cond), _lib.dptr(out), *shape[:1], *shape[2:],
                                      ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), n,
                                      ctypes.cast(acp.data_ptr(), ctypes.POINTER(ctypes.c_float)), acp.numel(), 2, sde,
                                      _lib.dptr(noise), _lib.dptr(flag, torch.int32), _lib.stream()), "dpmpp_sample")
        return out, flag

    a, flag = whole()
    b, _ = whole()
    assert torch.equal(a, b) and flag.item() == 0
    assert torch.equal(z_init, z_keep)
    rows = _rows(ts, 2, bool(sde)).to(cuda_dev)
    z, x0p = z_init.clone(), torch.empty_like(z_init)
    for i, t in enumerate(ts):
        eps = m(z, torch.tensor([int(t)], device=cuda_dev), cond)
        ops.dpmpp_update(z, x0p, eps, rows[i].contiguous(), noise[i] if sde else None)
    assert torch.equal(a, z)
    # the oracle's loop over the fp32 U-Net, free-running through the t = 999 clamp: a loose sanity bound only
    sd = _sd(m, cuda_dev)
    with torch.no_grad():
        ref = O.sample(lambda zz, tt, cc: R.unet_forward(sd, TINY_UNET, zz, tt, cc), acp, ts, z_init, cond, 2,
                       bool(sde), noise)
    print(f"tiny U-Net, DPM-Solver++(2M) {'SDE' if sde else 'ODE'} 6 steps: rel-L2 vs fp32 oracle {rel_l2(a, ref):.2e}")
    assert rel_l2(a, ref) < 0.2
    # the sampler class: same RNG order (z, then the per-step draws), same call
    torch.manual_seed(4)
    s1 = DPMSolverSampler(diff, m).sample(shape, cond, 5, cuda_dev, stochastic=bool(sde), progress=False)
    torch.manual_seed(4)
    zz = torch.randn(shape, device=cuda_dev)
    nn_ = torch.stack([torch.randn_like(zz) for _ in range(n)]) if sde else None
    z, x0p = zz.clone(), torch.empty_like(zz)
    for i, t in enumerate(ts):
        ops.dpmpp_update(z, x0p, m(z, torch.tensor([int(t)], device=cuda_dev), cond), rows[i].contiguous(),
                         nn_[i] if sde else None)
    assert torch.equal(s1, z)
    # any callable model: the Python loop over the same kernel
    torch.manual_seed(4)
    s2 = DPMSolverSampler(diff, lambda zz_, tt, cc: m(zz_, tt, cc)).sample(shape, cond, 5, cuda_dev,
                                                                          stochastic=bool(sde), progress=False)
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
@pytest.mark.parametrize("sampler", ["dpmpp_2m", "dpmpp_2m_sde"])
def test_generate_dpmpp20_batch4_all_gates(cuda_dev, bench_model, sampler):
    """BASELINE configs[1] (batch 4, 8 -> 48 slices at 192^2) with 20 steps = 21 U-Net evaluations, the DDIM gates of
    DESIGN.md section 2 against the fp32 oracle trajectory (tests/dpmpp_oracle.py over oracle/ref_port.py's U-Net):
      1. teacher-forced eps rel-L2 <= 1e-2 at every one of the 21 steps;  2. decode of the oracle z_0 >= 60 dB;
      3. |PSNR(new, target) - PSNR(ref, target)| <= 0.05 dB;  4. a second run with the same seed gives the same bits."""
    from v2v_b200.inference import DPMSolverSampler
    m, cfg = bench_model
    sd = _sd(m, cuda_dev)
    vae_cfg, unet_cfg, _ = R.resolve_config(cfg)
    sde = sampler == "dpmpp_2m_sde"
    batch, steps = 4, 20
    g = torch.Generator().manual_seed(1234)
    v_thick = (torch.rand((batch, 1, 8, 192, 192), generator=g) * 2 - 1).to(cuda_dev)
    target = (torch.rand((batch, 1, 48, 192, 192), generator=g) * 2 - 1).to(cuda_dev)
    ts = DPMSolverSampler(m.diffusion, m.unet)._get_timesteps(steps)
    acp = m.diffusion.alphas_cumprod.detach().float().cpu()
    torch.manual_seed(42)
    with torch.no_grad():  # generate() restated piece by piece, in the same RNG order
        z_in = R.vae_encode(sd, v_thick, vae_cfg["scaling_factor"], "vae.")
        cond = F.interpolate(z_in, size=(48, z_in.shape[3], z_in.shape[4]), mode="trilinear", align_corners=False)
        shape = tuple(cond.shape)
        torch.randn(shape, device=cuda_dev)  # discarded draw (models/model.py:303)
        z_init = torch.randn(shape, device=cuda_dev)
        noise = torch.stack([torch.randn_like(z_init) for _ in range(len(ts))]) if sde else None
        rec = []
        model = lambda z, t, c: R.unet_forward(sd, unet_cfg, z, t, c, "unet.")  # noqa: E731
        z0 = O.sample(model, acp, ts, z_init, cond, 2, sde, noise, record=rec)
        ref = R.vae_decode(sd, z0, vae_cfg["scaling_factor"], "vae.")
        del noise
    assert len(rec) == 21 and rec[0][1] == 999 and rec[-1][1] == 0
    errs = []
    for z_t, t_idx, eps_ref in rec:
        errs.append(rel_l2(m.unet(z_t, torch.full((batch,), t_idx, device=cuda_dev, dtype=torch.long), cond), eps_ref))
    del rec
    print(f"{sampler}-20, batch 4: teacher-forced eps rel-L2 over 21 steps: max {max(errs):.3e} "
          f"(t={ts[errs.index(max(errs))]}), mean {sum(errs) / len(errs):.3e}")
    assert max(errs) <= EPS_TOL, errs
    n = lambda v: (v.clamp(-1, 1) + 1) / 2  # noqa: E731
    p_dec = R.psnr(n(m.vae.decode(z0)), n(ref))
    print(f"{sampler}-20, batch 4: teacher-forced decode PSNR(new, ref) = {p_dec:.1f} dB")
    assert p_dec >= 60.0, p_dec
    torch.manual_seed(42)
    got = m.generate(v_thick, sampler, steps, target_depth=48)
    assert got.shape == ref.shape == (batch, 1, 48, 192, 192) and torch.isfinite(got).all()
    p_new, p_ref, p_direct = R.psnr(n(got), n(target)), R.psnr(n(ref), n(target)), R.psnr(n(got), n(ref))
    print(f"{sampler}-20, batch 4: generate PSNR(new,target)={p_new:.4f} PSNR(ref,target)={p_ref:.4f} "
          f"PSNR(new,ref)={p_direct:.2f} dB")
    assert abs(p_new - p_ref) <= 0.05, (p_new, p_ref)
    assert m.last_nan_flag.item() == 0
    torch.manual_seed(42)
    assert torch.equal(m.generate(v_thick, sampler, steps, target_depth=48), got)


def test_softmax_mode_teacher_forced_against_softmax_oracle(cuda_dev):
    import softmax_oracle as S
    from v2v_b200.inference import DPMSolverSampler
    from v2v_b200.models import GaussianDiffusion, UNet3D
    torch.manual_seed(0)
    m = UNet3D(**TINY_UNET).eval().to(cuda_dev).set_attention_mode("softmax")
    sd = _sd(m, cuda_dev)
    diff = GaussianDiffusion("cosine", 1000)
    ts = DPMSolverSampler(diff, m)._get_timesteps(10)
    g = torch.Generator().manual_seed(8)
    shape = (2, 4, 12, 8, 8)
    cond = torch.randn(shape, generator=g).to(cuda_dev)
    z_init = torch.randn(shape, generator=g).to(cuda_dev)
    rec = []
    with torch.no_grad():
        O.sample(lambda z, t, c: S.unet_forward(sd, TINY_UNET, z, t, c), diff.alphas_cumprod.float(), ts, z_init, cond,
                 record=rec)
    errs = [rel_l2(m(z_t, torch.full((2,), t, device=cuda_dev, dtype=torch.long), cond), e) for z_t, t, e in rec]
    print(f"softmax mode, tiny U-Net, DPM-Solver++(2M) 11 steps teacher-forced: max eps rel-L2 {max(errs):.3e}")
    assert max(errs) <= EPS_TOL, errs
    torch.manual_seed(1)
    out = DPMSolverSampler(diff, m).sample(shape, cond, 10, cuda_dev, stochastic=True, progress=False)
    assert torch.isfinite(out).all()


# ------------------------------------------------------------------------------------- generate() and wrappers
def _tiny_model(dev, **extra):
    from v2v_b200.models import VideoToVideoDiffusion
    g = golden("generate_tiny.pt")
    torch.manual_seed(g["seed"])
    return VideoToVideoDiffusion(dict(g["config"], **extra)).eval().to(dev), g


@pytest.mark.parametrize("sampler", ["dpmpp_2m", "dpmpp_2m_sde"])
def test_generate_equals_staged_composition(cuda_dev, sampler):
    from v2v_b200 import ops
    from v2v_b200.inference import DPMSolverSampler
    m, _ = _tiny_model(cuda_dev)
    gen = torch.Generator().manual_seed(13)
    v = (torch.rand((2, 1, 8, 32, 32), generator=gen) * 2 - 1).to(cuda_dev)
    torch.manual_seed(6)
    got = m.generate(v, sampler, 20, target_depth=48)
    assert got.shape == (2, 1, 48, 32, 32) and torch.isfinite(got).all() and m.last_nan_flag.item() == 0
    torch.manual_seed(6)
    cond = ops.upsample_depth(m.vae.encode(v), 48)
    torch.randn(tuple(cond.shape), device=cuda_dev)  # the reference's discarded draw
    z0 = DPMSolverSampler(m.diffusion, m.unet).sample(tuple(cond.shape), cond, 20, cuda_dev,
                                                      stochastic=sampler == "dpmpp_2m_sde", progress=False)
    assert torch.equal(got, m.vae.decode(z0))
    torch.manual_seed(6)
    assert torch.equal(m.generate(v, sampler, 20, target_depth=48), got)


def test_generate_batch_and_generate_volume(cuda_dev):
    from v2v_b200.inference import DPMSolverSampler
    from v2v_b200.inference.generate import generate_batch
    from v2v_b200.inference.volume import generate_volume
    m, _ = _tiny_model(cuda_dev)
    gen = torch.Generator().manual_seed(17)
    vids = torch.rand((2, 1, 3, 16, 24), generator=gen) * 2 - 1
    for name in ("dpmpp_2m", "dpmpp_2m_sde"):
        torch.manual_seed(8)
        got = generate_batch(m, vids, sampler_type=name, num_inference_steps=6, device=cuda_dev)
        assert got.shape == (2, 1, 3, 16, 24) and torch.isfinite(got).all()
        torch.manual_seed(8)
        z_in = m.vae.encode(vids.to(cuda_dev))
        z0 = DPMSolverSampler(m.diffusion, m.unet).sample(z_in.shape, z_in, 6, cuda_dev, stochastic=name.endswith("sde"),
                                                          progress=False)
        assert torch.equal(got, m.vae.decode(z0)), name
    with pytest.raises(ValueError):
        generate_batch(m, vids, sampler_type="euler", device=cuda_dev)
    vol = (torch.rand((1, 1, 4, 32, 32), generator=gen) * 2 - 1).to(cuda_dev)
    torch.manual_seed(9)
    full = generate_volume(m, vol, "dpmpp_2m", 4, patch_size=(2, 16, 16), target_patch_size=(6, 16, 16),
                           stride=(2, 8, 8), batch=4)
    assert full.shape == (1, 1, 12, 32, 32) and torch.isfinite(full).all() and full.abs().max() <= 1.0


def test_invalid_arguments_launch_nothing(cuda_dev):
    from v2v_b200 import _lib
    from v2v_b200.inference import DPMSolverSampler
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

    def sample(ts, order, sde, noise):
        return L.b2v_dpmpp_sample(u, _lib.dptr(z), _lib.dptr(z), _lib.dptr(out), 1, 6, 4, 4,
                                  ts.ctypes.data_as(ctypes.POINTER(ctypes.c_int64)), len(ts), acp_p, acp.numel(), order,
                                  sde, noise, None, _lib.stream())

    for what, args, phrase in (("sde without noise", (good, 2, 1, None), "noise"),
                               ("order 3", (good, 3, 0, None), "order"),
                               ("unsorted timesteps", (unsorted, 2, 0, None), "decreasing")):
        assert sample(*args) != 0, what
        assert phrase in _lib.last_error(), (what, _lib.last_error())
    with pytest.raises(ValueError):
        DPMSolverSampler(m.diffusion, m.unet).sample(shape, z, 5, cuda_dev, order=3)
    v_in = g["v_in"].to(cuda_dev).contiguous()
    cfg = _lib.SamplerCfg()
    cfg.n, cfg.n_train = len(good), acp.numel()
    cfg.timesteps = good.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    cfg.alphas_cumprod = acp_p
    vout = torch.empty((1, 1, 6, 16, 16), device=cuda_dev)

    def generate(code):
        cfg.sampler = code
        return L.b2v_generate(u, vh, ctypes.byref(cfg), _lib.dptr(v_in), _lib.dptr(z), _lib.dptr(vout), 1, 2, 6, 16, 16,
                              None, _lib.stream())

    assert generate(7) != 0 and "unknown sampler" in _lib.last_error()
    assert generate(3) != 0 and "noise" in _lib.last_error()
    cfg.timesteps = unsorted.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))
    assert generate(2) != 0 and "decreasing" in _lib.last_error()
    assert _lib.launch_count() == n0
