"""B200-native denoising hot path for dnnhhuy/stable-diffusion-pytorch.

Drop-in replacements for the reference's ``models/unet`` ``UNet.forward(x, timestep, cond)``
and ``models/scheduler`` samplers (plus a DPM-Solver++(2M) sampler), running on hand-written sm_100a CUDA kernels behind a C-ABI
library (include/sdb200.h).  See DESIGN.md / INTEGRATION.md.
"""
from .scheduler import DDIMSampler, DDPMSampler, DPMSolverSampler, x0_from_eps  # noqa: F401

__all__ = ["DDIMSampler", "DDPMSampler", "DPMSolverSampler", "x0_from_eps", "UNet", "VAE", "OpenCLIP", "CLIPTextModel", "CLIPTextConfig", "TextEncoder", "DenoiseLoop", "denoise", "one_step", "img2img", "inpaint"]


def __getattr__(name):
    # UNet / pipeline import torch.nn machinery lazily (keeps `import` cheap for host-only users)
    if name == "UNet":
        from .unet import UNet
        return UNet
    if name in ("OpenCLIP", "CLIPTextModel", "CLIPTextConfig", "TextEncoder"):
        from . import clip
        return getattr(clip, name)
    if name == "VAE":
        from .vae import VAE
        return VAE
    if name in ("DenoiseLoop", "denoise", "one_step", "img2img", "inpaint"):
        from . import pipeline
        return getattr(pipeline, name)
    raise AttributeError(name)
