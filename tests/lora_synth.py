"""Seeded synthetic LoRA adapters for the UNet, in kohya or PEFT form, and the float64 merge they stand for (test helper)."""
import torch

from stable_diffusion_pytorch_b200 import lora
from stable_diffusion_pytorch_b200.arch import param_spec


def make_adapter(arch, fmt="kohya", rank=4, alpha=None, seed=0, amp=1.0, select=None, linear_proj=False, dtype=torch.float32):
    """A LoRA on every target of the table (or those whose diffusers path contains one of ``select``).
    Returns (file state dict, {reference parameter name: (up [N][r] float64, down [r][...] float64, alpha / rank)}).
    Convs get LoCon factors; ``linear_proj``: proj_in / proj_out are Linears (SD2.1).  ΔW has about ``amp`` times the spread
    of the weight's default init."""
    g = torch.Generator().manual_seed(seed)
    shapes = dict(param_spec(arch))
    sd, truth = {}, {}
    for dpath, ref in sorted(lora.targets(arch).items()):
        if select is not None and not any(s in dpath for s in select):
            continue
        shape = shapes[ref]
        n, kshape = shape[0], tuple(shape[1:])
        if linear_proj and dpath.endswith(("proj_in", "proj_out")):
            kshape = kshape[:1]
        k = 1
        for d in kshape:
            k *= d
        down = torch.randn((rank,) + kshape, generator=g, dtype=torch.float64) / k ** 0.5
        up = torch.randn((n, rank), generator=g, dtype=torch.float64) * (amp / (3 * rank) ** 0.5)
        down, up = down.to(dtype).double(), up.to(dtype).double()      # the truth is what the file holds
        a = float(rank) if alpha is None else float(alpha)
        truth[ref] = (up, down, a / rank)
        up_file = up[:, :, None, None] if len(kshape) == 3 else up
        if fmt == "kohya":
            stem = "lora_unet_" + dpath.replace(".", "_")
            sd[f"{stem}.lora_down.weight"] = down.to(dtype)
            sd[f"{stem}.lora_up.weight"] = up_file.to(dtype)
            sd[f"{stem}.alpha"] = torch.tensor(a)
        else:
            sd[f"unet.{dpath}.lora_A.weight"] = down.to(dtype)
            sd[f"unet.{dpath}.lora_B.weight"] = up_file.to(dtype)
    if fmt == "kohya" and alpha is None:
        for key in sorted(k for k in sd if k.endswith(".alpha"))[::2]:
            del sd[key]                                           # alpha defaults to the rank
    return sd, truth


def merged(sd, truths_scales):
    """float64 state dict with every ``(truth, scale)`` delta applied."""
    out = {k: v.double().clone() for k, v in sd.items()}
    for truth, scale in truths_scales:
        for ref, (up, down, mult) in truth.items():
            w = out[ref]
            out[ref] = w + (scale * mult) * (up @ down.reshape(down.shape[0], -1)).reshape(w.shape)
    return out
