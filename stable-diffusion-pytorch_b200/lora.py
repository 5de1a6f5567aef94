"""LoRA / LoCon adapters for the UNet: file parsing and the map from a diffusers module to the packed tensors it feeds.

A LoRA replaces a weight W [N][K] by W + scale * alpha/rank * up @ down.  The packed layout (unet.PackedWeights) does not map a
diffusers module one-to-one onto a packed tensor -- q|k|v are one matrix, the cross-attention k|v of every layer are rows of
``kv2_all.w`` (bf16), GEGLU rows are interleaved, the 22 time projections are rows of ``tb.w``, conv taps are in NHWC order and the
upsample convs also exist as four parity convs -- so ``merge_ops`` turns one module into the ``sdk_lora_merge`` launches that
rebuild every packed tensor it feeds, from the fp32 master weight and the active adapters.

Supported files (a ``.safetensors`` path or a state dict):
  kohya   ``lora_unet_<diffusers module path, '.' -> '_'>.lora_down.weight / .lora_up.weight / .alpha``
  PEFT    ``unet.<diffusers module path>.lora_A.weight / .lora_B.weight``  (alpha = rank)
LoCon convs have down [r][Cin][kh][kw] and up [N][r][1][1].  Keys without a UNet prefix (text-encoder LoRA) are returned unapplied.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Tuple

import torch

from .arch import UNetArch, param_spec
from .program import _kmat, up2_parity_weights
from .weights import _module_pairs

KOHYA, PEFT = "lora_unet_", "unet."


@dataclass
class LoraModule:
    """One adapted module: up [N][r] and down [r][K] (linear) or [r][Cin][kh][kw] (conv), fp32; ``mult`` = alpha / rank."""
    up: torch.Tensor
    down: torch.Tensor
    mult: float


@dataclass
class Write:
    """One ``sdk_lora_merge`` destination of a module: rows [lo, hi) of the module's weight go to rows row_off + row_step * n of
    packed tensor ``key``; ``parity`` >= 0 selects one of the four parity blocks of an upsample conv's ``w_up2``."""
    key: str
    lo: int
    hi: int
    row_off: int = 0
    row_step: int = 1
    parity: int = -1


_LEAVES = ("conv_1", "conv_2", "proj_input", "t_embed", "conv_input", "conv_output")      # ResBlock / transformer convs and Linears


def targets(a: UNetArch) -> Dict[str, str]:
    """diffusers module path -> reference parameter name, for every module a LoRA may adapt."""
    resample = {st.resample.prefix for st in a.down + a.up if st.resample is not None}
    params = {n for n, _ in param_spec(a)}                  # ResBlocks without a channel change have no shortcut conv
    return {dif: ref + ".weight" for ref, dif in _module_pairs(a) if ref + ".weight" in params and (
            ref in resample or ref.rsplit(".", 1)[1] in _LEAVES or (".transformer_block." in ref and "layernorm" not in ref))}


def writes(a: UNetArch, pw, ref: str) -> List[Write]:
    """The packed destinations of reference parameter ``ref`` in pack ``pw`` (any precision)."""
    mod = ref[: -len(".weight")]
    for tr in a.transformers:
        p, b, c = tr.prefix, f"{tr.prefix}.transformer_block", tr.c
        if not mod.startswith(p + "."):
            continue
        leaf = mod[len(b) + 1:] if mod.startswith(b + ".") else mod[len(p) + 1:]
        if leaf in ("attn1.q_proj", "attn1.k_proj", "attn1.v_proj"):
            return [Write(f"{p}.qkv.w", 0, c, "qkv".index(leaf[6]) * c)]
        if leaf in ("attn2.k_proj", "attn2.v_proj"):
            off = (0 if leaf[6] == "k" else c)
            if "kv2_all.w" in pw.t:
                return [Write("kv2_all.w", 0, c, pw.kv_off[tr.index] + off)]
            return [Write(f"{p}.kv2.w", 0, c, off)]
        if leaf == "ffn.0.proj":                       # rows interleaved (value_j, gate_j)
            return [Write(f"{p}.ff0.w", 0, 4 * c, 0, 2), Write(f"{p}.ff0.w", 4 * c, 8 * c, 1, 2)]
        key = {"attn1.out_proj": "o1", "attn2.q_proj": "q2", "attn2.out_proj": "o2", "ffn.1": "ff1",
               "conv_input": "in", "conv_output": "out"}[leaf]
        return [Write(f"{p}.{key}.w", 0, c)]
    for r in a.res_blocks:
        if mod.startswith(r.prefix + "."):
            leaf = mod[len(r.prefix) + 1:]
            if leaf == "t_embed":
                return [Write("tb.w", 0, r.cout, r.tb_offset)]
            return [Write(f"{r.prefix}.{ {'conv_1': 'conv1', 'conv_2': 'conv2', 'proj_input': 'sc'}[leaf] }.w", 0, r.cout)]
    for st in a.down + a.up:
        if st.resample is not None and st.resample.prefix == mod:
            n = st.resample.cout
            out = [Write(f"{mod}.w", 0, n)]
            if f"{mod}.w_up2" in pw.t:
                out += [Write(f"{mod}.w_up2", 0, n, parity=q) for q in range(4)]
            return out
    raise KeyError(ref)


def _factors(w: torch.Tensor, four_d: bool, parity: int):
    """A weight-shaped tensor [N or r][...] -> [rows][K] fp32 in the packed k order of one destination."""
    if not four_d:
        return w
    if parity >= 0:
        w = up2_parity_weights(w)[parity // 2, parity % 2]
    return _kmat(w)


def merge_ops(a: UNetArch, pw, ref: str, weight: torch.Tensor, mods: List[Tuple[LoraModule, float]]):
    """The ``sdk_lora_merge`` launches that rebuild every packed tensor of reference parameter ``ref`` from its master ``weight``
    and the adapters ``mods`` [(module, user scale)] (concatenated along r in the given order).  Yields dicts of the kernel's
    arguments as device tensors on ``pw.device``: dst (the packed tensor), offset (elements), layout, dst_rows, row_off,
    row_step, base [n][K], up [n][R] or None, down [R][K] or None."""
    dev = pw.device
    w = weight.detach().to(device=dev, dtype=torch.float32)
    four_d = w.dim() == 4
    up = down = None
    if mods:
        up = torch.cat([m.up.to(dev) * (s * m.mult) for m, s in mods], 1)
        down = torch.cat([m.down.to(dev) for m, _ in mods], 0)
    for wr in writes(a, pw, ref):
        base = _factors(w, four_d, wr.parity)[wr.lo:wr.hi].contiguous()
        n, k = base.shape
        dst = pw.t[wr.key]
        if dst.dim() == 3:
            layout, rows, offset = 1, dst.shape[1], (wr.parity * (k // 64) * rows * 64 if wr.parity >= 0 else 0)
        else:
            if dst.shape[1] != k:
                raise RuntimeError(f"{wr.key}: row length {dst.shape[1]} != K {k}")
            layout, rows, offset = 0, dst.shape[0], 0
        yield dict(dst=dst, offset=offset, layout=layout, dst_rows=rows, row_off=wr.row_off, row_step=wr.row_step, base=base,
                   up=None if up is None else up[wr.lo:wr.hi].contiguous(),
                   down=None if down is None else _factors(down, four_d, wr.parity).contiguous())


def _load(src):
    if isinstance(src, (str, bytes)) or hasattr(src, "__fspath__"):
        path = str(src)
        if path.endswith(".safetensors"):
            from safetensors.torch import load_file
            return load_file(path)
        return torch.load(path, map_location="cpu")
    return dict(src)


def read_adapter(src, a: UNetArch) -> Tuple[Dict[str, LoraModule], List[str]]:
    """Parse a kohya or PEFT LoRA for the UNet of ``a`` -> ({reference parameter name: LoraModule}, [keys not applied]).
    Raises ValueError naming the key for a UNet key that does not resolve to a supported module, a factor missing its partner,
    ranks that disagree or a shape that does not fit the module's weight."""
    sd = _load(src)
    tgt = targets(a)
    kohya_names = {d.replace(".", "_"): d for d in tgt}
    shapes = dict(param_spec(a))
    groups: Dict[str, Dict[str, Tuple[str, torch.Tensor]]] = {}
    unapplied = []
    for key, val in sd.items():
        if key.startswith(KOHYA):
            stem, _, suffix = key[len(KOHYA):].partition(".")
            dpath = kohya_names.get(stem)
            role = {"lora_down.weight": "down", "lora_up.weight": "up", "alpha": "alpha"}.get(suffix)
        elif key.startswith(PEFT):
            stem, role = key[len(PEFT):], None
            for sfx, rl in ((".lora_A.weight", "down"), (".lora_B.weight", "up")):
                if stem.endswith(sfx):
                    stem, role = stem[: -len(sfx)], rl
            dpath = stem if stem in tgt else None
        else:
            unapplied.append(key)
            continue
        if dpath is None or role is None:
            raise ValueError(f"LoRA key {key!r} does not name a supported UNet module / factor (supported: attention and "
                             "feed-forward Linears, proj_in/proj_out, ResBlock convs and time_emb_proj, down/upsampler convs)")
        groups.setdefault(dpath, {})[role] = (key, val)
    mods = {}
    for dpath, g in groups.items():
        for role in ("up", "down"):
            if role not in g:
                other = next(iter(g.values()))[0]
                raise ValueError(f"LoRA key {other!r} has no matching {role} factor")
        (kd, down), (ku, up) = g["down"], g["up"]
        ref = tgt[dpath]
        shape = shapes[ref]
        down, up = down.detach().to("cpu", torch.float32), up.detach().to("cpu", torch.float32)
        if up.dim() == 4 and tuple(up.shape[2:]) == (1, 1):
            up = up[:, :, 0, 0]
        r = down.shape[0] if down.dim() >= 1 else -1
        if up.dim() != 2 or up.shape[1] != r:
            raise ValueError(f"LoRA key {ku!r}: up {tuple(up.shape)} and down {tuple(down.shape)} ranks disagree")
        if up.shape[0] != shape[0]:
            raise ValueError(f"LoRA key {ku!r}: up {tuple(up.shape)} does not fit {dpath} weight {tuple(shape)}")
        k_shape = tuple(shape[1:])
        ok = tuple(down.shape[1:]) == k_shape or (
            down.dim() in (2, 4) and tuple(down.shape[1:]) in ((k_shape[0],), (k_shape[0], 1, 1)) and all(s == 1 for s in k_shape[1:]))
        if not ok:
            raise ValueError(f"LoRA key {kd!r}: down {tuple(down.shape)} does not fit {dpath} weight {tuple(shape)}")
        alpha = float(g["alpha"][1]) if "alpha" in g else float(r)
        mods[ref] = LoraModule(up.contiguous(), down.reshape((r,) + k_shape).contiguous(), alpha / r)
    return mods, unapplied

