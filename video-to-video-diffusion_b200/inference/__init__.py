"""Drop-in names of the reference's `inference` package: the two samplers (CUDA-graph-replayed loops in libb2v.so),
plus `volume.generate_volume`, the thick->thin sliding-window stitcher.  `DPMSolverSampler` (DPM-Solver++(2M), ODE and
SDE) and `UniPCSampler` (UniPC, orders 1-3, bh1 / bh2) are additions of this package."""
from . import sampler as _sampler

DDIMSampler = _sampler.DDIMSampler
DDPMSampler = _sampler.DDPMSampler
DPMSolverSampler = _sampler.DPMSolverSampler
UniPCSampler = _sampler.UniPCSampler
EDMSampler = _sampler.EDMSampler

__all__ = ("DDIMSampler", "DDPMSampler", "DPMSolverSampler", "UniPCSampler", "EDMSampler")
