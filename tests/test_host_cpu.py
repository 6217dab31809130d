"""CPU suite, part 2: host-side logic of the drop-in mirror, the C-ABI surface, and the multi-rank plumbing
(world_size-2 gloo).  No compute call is made through libb2v here (there is no GPU)."""
import ctypes
import os
import re
import socket

import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_c_abi_exports_every_declared_symbol():
    from v2v_b200 import _lib
    hdr = open(os.path.join(ROOT, "include", "b2v.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    declared = set(re.findall(r"\b(b2v_[a-z0-9_]+)\s*\(", hdr))
    assert len(declared) >= 30
    handle = ctypes.CDLL(_lib.LIB_PATH)
    missing = [s for s in sorted(declared) if not hasattr(handle, s)]
    assert not missing, missing
    assert set(_lib.SIGNATURES) == declared  # the ctypes binding covers the whole header, and nothing else
    L = _lib.lib()
    assert L.b2v_abi_version() == 2
    # a freshly loaded library has launched nothing; checked in a new process, since GPU tests run earlier in this one
    # launch kernels through the same handle
    import subprocess
    import sys
    probe = (f"import sys; sys.path.insert(0, {ROOT!r}); from v2v_b200 import _lib; L = _lib.lib(); "
             "print(L.b2v_abi_version(), L.b2v_launch_count())")
    r = subprocess.run([sys.executable, "-c", probe], capture_output=True, text=True)
    assert r.stdout.split() == ["2", "0"], (r.stdout, r.stderr)


def test_c_abi_has_no_torch_or_cpu_fallback_dependency():
    import subprocess
    from v2v_b200 import _lib
    needed = subprocess.run(["objdump", "-p", _lib.LIB_PATH], capture_output=True, text=True).stdout
    libs = re.findall(r"NEEDED\s+(\S+)", needed)
    assert not any("torch" in l or "c10" in l or "cudnn" in l or "cublas" in l for l in libs), libs


def test_create_fails_loudly_without_a_gpu():
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from v2v_b200 import _lib
    h = ctypes.c_void_p()
    d = _lib.UNetDesc()
    d.num_levels, d.num_res_blocks = 2, 1
    assert _lib.lib().b2v_unet_create(ctypes.byref(h), ctypes.byref(d)) != 0
    assert "no CUDA device" in _lib.last_error() or "sm_100a" in _lib.last_error()
    from helpers import tiny_unet, tiny_vae
    with pytest.raises(RuntimeError):
        tiny_unet()(torch.zeros(1, 4, 4, 8, 8), torch.zeros(1, dtype=torch.long), torch.zeros(1, 4, 4, 8, 8))
    with pytest.raises(RuntimeError):
        tiny_vae().decode(torch.zeros(1, 4, 2, 4, 4))


def test_mirror_surface_matches_reference_signatures():
    import inspect
    from v2v_b200.inference import DDIMSampler, DDPMSampler
    from v2v_b200.inference.generate import generate_batch
    from v2v_b200.models import GaussianDiffusion, UNet3D, VideoToVideoDiffusion, VideoVAE
    sig = lambda f: list(inspect.signature(f).parameters)  # noqa: E731
    assert sig(UNet3D.__init__)[1:] == ["latent_dim", "model_channels", "num_res_blocks", "attention_levels",
                                        "channel_mult", "num_heads", "time_embed_dim", "use_checkpoint"]
    assert sig(UNet3D.forward)[1:] == ["x", "t", "c"]
    assert sig(VideoVAE.__init__)[1:] == ["in_channels", "latent_dim", "base_channels", "scaling_factor",
                                          "gradient_checkpointing"]
    assert sig(GaussianDiffusion.__init__)[1:] == ["noise_schedule", "timesteps", "beta_start", "beta_end"]
    assert sig(DDIMSampler.sample)[1:] == ["shape", "conditioning", "num_inference_steps", "device", "eta", "progress"]
    assert sig(DDPMSampler.sample)[1:] == ["shape", "conditioning", "device", "progress"]
    assert sig(VideoToVideoDiffusion.generate)[1:] == ["v_in", "sampler", "num_inference_steps", "guidance_scale",
                                                       "target_depth"]
    assert sig(generate_batch) == ["model", "input_videos", "sampler_type", "num_inference_steps", "device"]
    assert sig(DDIMSampler.sample_with_stitching)[1:4] == ["v_thick_full", "vae", "num_inference_steps"]
    vae = VideoVAE(1, 8, 64, 1.0)
    assert vae.get_latent_shape((2, 1, 48, 192, 192)) == (2, 8, 48, 48, 48)
    with pytest.raises(NotImplementedError):
        VideoVAE.from_pretrained("x")


def test_reference_checkpoint_format_loads():
    """a reference checkpoint is {'model_state_dict': ..., 'config': ...} (models/model.py:362-365)"""
    from helpers import golden, sd_hash
    from v2v_b200.models import VideoToVideoDiffusion
    g = golden("generate_tiny.pt")
    torch.manual_seed(g["seed"])
    src = VideoToVideoDiffusion(g["config"])
    ckpt = {"model_state_dict": src.state_dict(), "config": g["config"]}
    torch.manual_seed(123)
    dst = VideoToVideoDiffusion(ckpt["config"])
    assert sd_hash(dst.state_dict()) != g["sd_hash"]
    dst.load_state_dict(ckpt["model_state_dict"], strict=True)
    assert sd_hash(dst.state_dict()) == g["sd_hash"]
    assert {k.split(".")[0] for k in dst.state_dict()} == {"vae", "unet", "diffusion"}
    import copy
    copy.deepcopy(dst)  # the native handle must not be shared by copies


def test_ddim_timesteps_and_ddpm_coefficients():
    from helpers import golden
    from v2v_b200.inference import DDIMSampler
    from v2v_b200.models import GaussianDiffusion
    g = golden("schedule.pt")
    d = GaussianDiffusion("cosine", 1000)
    s = DDIMSampler(d, None)
    for n, key in ((50, "ts50"), (20, "ts20"), (7, "ts7")):
        assert s._get_timesteps(n).tolist() == g[key].tolist()
    assert torch.equal(d.alphas_cumprod, g["alphas_cumprod"])
    rows = d.ddpm_coefficients()
    assert rows.shape == (1000, 8) and rows[0, 4] == 0 and rows[1:, 4].min() == 1
    assert torch.allclose(rows[:, 5], torch.exp(0.5 * g["posterior_log_variance_clipped"]))
    with pytest.raises(ValueError):
        GaussianDiffusion("sigmoid")


def test_work_sharding_and_patch_grid():
    from v2v_b200.dist import patch_grid, shard_range, volume_work_items
    assert patch_grid(512, 192, 96) == [0, 96, 192, 288, 320]  # SURVEY 8(d): 25 patches per 512^2 slab
    assert patch_grid(192, 192, 96) == [0]
    items = volume_work_items(64, 512, 512)
    assert len(items) == 1600
    for world in (1, 2, 4, 8, 3):
        spans = [shard_range(len(items), r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == len(items)
        assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
        assert max(b - a for a, b in spans) - min(b - a for a, b in spans) <= 1
    assert [shard_range(32, r, 8) for r in range(8)][3] == (12, 16)  # config 4: batch 32 -> 4 per GPU
    assert shard_range(0, 0, 2) == (0, 0)  # empty input


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _gather_worker(rank, world, port, ragged):
    import torch.distributed as dist
    from v2v_b200.dist import gather_slabs, shard_range
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        n_items = 5 if ragged else 4
        full = torch.arange(n_items * 2 * 3, dtype=torch.float32).reshape(n_items, 1, 2, 3, 1)
        lo, hi = shard_range(n_items, rank, world)
        counts = [shard_range(n_items, r, world)[1] - shard_range(n_items, r, world)[0] for r in range(world)]
        out = gather_slabs(full[lo:hi].clone(), counts if ragged else None)
        assert torch.equal(out, full), (rank, out.shape)
    finally:
        dist.destroy_process_group()


def _async_gather_worker(rank, world, port):
    import torch.distributed as dist
    from v2v_b200.dist import SlabGatherer
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        g = SlabGatherer(depth=2)
        outs = []
        for step in range(5):  # more batches than buffers: results are consumed before their buffer is reused
            local = torch.full((2, 1, 2, 3, 1), float(10 * step + rank))
            out = g.gather(local)
            outs.append((step, out))
            if step % 2 == 1:
                g.finish()
                for st, o in outs:
                    assert torch.equal(o[:2], torch.full((2, 1, 2, 3, 1), float(10 * st)))
                    assert torch.equal(o[2:], torch.full((2, 1, 2, 3, 1), float(10 * st + 1)))
                outs = []
        g.finish()
        assert not g.pending
    finally:
        dist.destroy_process_group()


def test_async_slab_gatherer_world2_gloo():
    """bench.py's N > 1 path: one asynchronous all-gather per batch into rotating buffers, completed by finish()"""
    import sys
    sys.path.insert(0, ROOT)
    mp.spawn(_async_gather_worker, args=(2, _free_port()), nprocs=2, join=True)


@pytest.mark.parametrize("ragged", [False, True])
def test_gather_of_decoded_slabs_world2_gloo(ragged):
    """the N>1 data path: each rank decodes its shard, one all-gather rebuilds the single-GPU result"""
    import sys
    sys.path.insert(0, ROOT)
    mp.spawn(_gather_worker, args=(2, _free_port(), ragged), nprocs=2, join=True)


def test_c_ddim_timesteps_matches_reference_subset():
    """b2v_ddim_timesteps is host-only integer logic (inference/sampler.py:221-239): checked against the golden lists"""
    from helpers import golden
    from v2v_b200 import _lib
    g = golden("schedule.pt")
    L = _lib.lib()
    buf = (ctypes.c_int64 * 64)()
    for n, key in ((50, "ts50"), (20, "ts20"), (7, "ts7")):
        cnt = L.b2v_ddim_timesteps(1000, n, buf, 64)
        assert cnt == len(g[key]) and list(buf[:cnt]) == g[key].tolist()
    assert L.b2v_ddim_timesteps(1000, 50, buf, 10) < 0 and "too small" in _lib.last_error()
    assert L.b2v_ddim_timesteps(1000, 0, buf, 64) < 0


def test_sampler_entry_points_validate_shapes_before_the_c_call():
    """ADVICE r1: a conditioning tensor that was not depth-upsampled (or a wrong channel count) must raise like the
    reference's torch.cat does, not reach the pointer-based C ABI"""
    from helpers import tiny_unet
    from v2v_b200.inference import DDIMSampler, DDPMSampler
    from v2v_b200.models import GaussianDiffusion
    m = tiny_unet()
    d = GaussianDiffusion("cosine", 20)
    shape = (1, 4, 6, 4, 4)
    with pytest.raises(ValueError, match="conditioning has shape"):
        DDIMSampler(d, m).sample(shape, torch.zeros(1, 4, 2, 4, 4), 5, "cuda")
    with pytest.raises(ValueError, match="latent_dim"):
        DDIMSampler(d, m).sample((1, 3, 6, 4, 4), torch.zeros(1, 3, 6, 4, 4), 5, "cuda")
    with pytest.raises(ValueError, match="conditioning has shape"):
        DDPMSampler(d, m).sample(shape, torch.zeros(2, 4, 6, 4, 4), "cuda")
    with pytest.raises(ValueError):
        d.p_sample_loop(m, (1, 4, 6, 4), torch.zeros(1, 4, 6, 4), "cuda")


def test_unsupported_configs_fail_at_construction():
    from v2v_b200.models import UNet3D, VideoVAE
    with pytest.raises(ValueError, match="multiple of 64"):
        UNet3D(latent_dim=4, model_channels=96)
    with pytest.raises(ValueError, match="latent_dim"):
        UNet3D(latent_dim=12, model_channels=64, channel_mult=(1,), attention_levels=[])
    with pytest.raises(ValueError, match="multiple of 64"):
        VideoVAE(1, 4, 32, 1.0)
    UNet3D(latent_dim=4, model_channels=192, channel_mult=(1, 2), num_res_blocks=1, attention_levels=[1])  # 24 ch / group


def test_native_handle_tracks_parameter_identity_and_versions():
    """ADVICE r1: a sum of version counters misses replaced / re-assigned tensors"""
    from helpers import tiny_unet
    from v2v_b200.models._native import _weights_version, normalize_device
    m = tiny_unet()
    v0 = _weights_version(m)
    with torch.no_grad():
        m.conv_in.weight.add_(1.0)  # in-place update: version counter
    v1 = _weights_version(m)
    m.conv_in.weight = torch.nn.Parameter(m.conv_in.weight.detach().clone())  # replaced object, version 0 again
    v2 = _weights_version(m)
    m.conv_in.bias.data = m.conv_in.bias.data.clone()  # .data re-assignment: new storage
    v3 = _weights_version(m)
    assert len({v0, v1, v2, v3}) == 4
    assert normalize_device("cpu") == torch.device("cpu")


def test_header_is_valid_c_and_links_from_a_c_program(tmp_path):
    """include/b2v.h compiles as strict C99 and a C program linked against libb2v.so can call the host-side entry
    points (the boundary is a C ABI, not a C++ one)"""
    import shutil
    import subprocess
    from v2v_b200 import _lib
    if shutil.which("gcc") is None:
        pytest.skip("no gcc")
    _lib.lib()
    exe = str(tmp_path / "host_check")
    libdir = os.path.dirname(_lib.LIB_PATH)
    subprocess.run(["gcc", "-std=c99", "-pedantic", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"),
                    os.path.join(ROOT, "tests", "c_abi", "host_check.c"), "-o", exe, "-L", libdir, "-l:libb2v.so",
                    "-Wl,-rpath," + libdir], check=True)
    r = subprocess.run([exe], capture_output=True, text=True)
    assert r.returncode == 0, (r.returncode, r.stdout, r.stderr)
    assert "ok abi=2" in r.stdout
