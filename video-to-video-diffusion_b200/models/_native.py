"""Shared plumbing for the nn.Module mirrors: keeps a libb2v object in sync with the module's parameters."""
import ctypes

import torch

from .. import _lib


def _weights_version(module):
    """identity + in-place version + storage address of every parameter / buffer: changes when a tensor is replaced
    (load_state_dict(assign=True), `p.data = ...`, .to()), updated in place (optimiser step, copy_) or re-allocated.
    In-place writes through `.data` / raw pointers bypass torch's version counter: call `invalidate_native()` then."""
    return tuple((id(t), t._version, t.data_ptr()) for t in list(module.parameters()) + list(module.buffers()))


def normalize_device(device):
    """torch.device with an explicit index ('cuda' -> the current device), so equality means 'same GPU'"""
    dev = torch.device(device)
    if dev.type == "cuda" and dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def check_sampler_args(model, shape, cond, device):
    """Shape / dtype / device contract of the native sampler entry points.  The C ABI copies B*latent_dim*T*h*w floats
    computed from `shape` and the model's latent_dim, so a conditioning tensor of another shape would be read out of
    bounds; the reference fails in torch.cat for the same inputs (models/unet3d.py:372) -- this raises ValueError."""
    shape = tuple(int(s) for s in shape)
    if len(shape) != 5:
        raise ValueError(f"sampler: shape must be (B, C, T, h, w), got {shape}")
    if shape[1] != model.latent_dim:
        raise ValueError(f"sampler: shape[1] = {shape[1]} does not match the U-Net's latent_dim = {model.latent_dim}")
    if tuple(cond.shape) != shape:
        raise ValueError(f"sampler: conditioning has shape {tuple(cond.shape)}, expected {shape} "
                         "(was the conditioning latent depth-upsampled to the target depth?)")
    dev = normalize_device(device)
    if dev.type != "cuda":
        raise RuntimeError(f"sampler: device {dev} -- this implementation runs on B200 only (no CPU fallback)")
    if not cond.is_floating_point():
        raise TypeError(f"sampler: conditioning must be a floating-point tensor, got {cond.dtype}")
    return shape, dev


class NativeHandle:
    """Owns one b2v_unet / b2v_vae.  (Re)built lazily from the module's state_dict whenever a parameter changed
    (load_state_dict, .to(), optimiser step), so reference checkpoints load through the usual torch path."""

    def __init__(self, kind):
        self.kind = kind  # "unet" | "vae"
        self.handle = None
        self.version = None
        self.device = None

    def get(self, module, desc, device, attention=None):
        """attention (U-Net only): the b2v_unet_set_attention mode, part of the cache key; None leaves the default"""
        device = normalize_device(device)
        ver = (_weights_version(module), attention)
        if self.handle is not None and self.version == ver and self.device == device:
            return self.handle
        self.close()
        L = _lib.lib()
        h = ctypes.c_void_p()
        with torch.cuda.device(device):
            _lib.check(getattr(L, f"b2v_{self.kind}_create")(ctypes.byref(h), ctypes.byref(desc)), f"{self.kind}_create")
            if attention is not None:
                _lib.check(L.b2v_unet_set_attention(h, int(attention)), "unet_set_attention")
            load = getattr(L, f"b2v_{self.kind}_load_weight")
            for key, val in module.state_dict().items():
                w = val.detach().to("cpu", torch.float32).contiguous()
                shape = (ctypes.c_int64 * max(1, w.dim()))(*w.shape)
                _lib.check(load(h, key.encode(), _lib.hptr(w), shape, w.dim()), f"load_weight({key})")
            _lib.check(getattr(L, f"b2v_{self.kind}_finalize")(h), f"{self.kind}_finalize")
        self.handle, self.version, self.device = h, ver, device
        return h

    def __deepcopy__(self, memo):  # copies of the module rebuild their own native object on first use
        return NativeHandle(self.kind)

    def __getstate__(self):
        return {"kind": self.kind, "handle": None, "version": None, "device": None}

    def invalidate(self):
        """force a rebuild on next use (after weight changes torch cannot see, e.g. writes through `.data`)"""
        self.version = None

    def close(self):
        if self.handle is not None:
            try:
                getattr(_lib.lib(), f"b2v_{self.kind}_destroy")(self.handle)
            except Exception:
                pass
            self.handle = None

    def __del__(self):
        self.close()


def require_cuda(t, what):
    if not t.is_cuda:
        raise RuntimeError(f"{what}: input is on {t.device}; this implementation runs on B200 only (no CPU fallback)")
    return t.detach().to(torch.float32).contiguous()


class ParamsOnly(torch.nn.Module):
    """Container that holds parameters under the reference's names; its math runs inside the parent's fused
    native call, so calling it directly is an error rather than a silent torch fallback."""

    def forward(self, *a, **k):
        raise RuntimeError(f"{type(self).__name__} is a parameter container; run the enclosing UNet3D / VAE module "
                           "(its forward executes on libb2v.so)")
