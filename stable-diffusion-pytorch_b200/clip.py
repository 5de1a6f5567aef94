"""B200-native TEXT ENCODERS — drop-ins for the reference's ``models/clip``: ``CLIPTextModel`` / ``OpenCLIP``
(models/clip/openclip.py:107-160, what models/diffusion.py:190-200 calls as ``clip.text_model(tokens)``) and ``TextEncoder``
(models/clip/clip.py:8-34).  SURVEY §8(f) rank 3: the stage right before the denoising loop.

Same construction as the UNet / VAE: parameters under the reference's names, ``forward(ids)`` runs a pre-planned launch list
on the shared C-ABI kernels -- token + position embedding gather, LayerNorm, fused q|k|v GEMM (tcgen05), CAUSAL tcgen05 flash
attention (head_dim 64), out-projection with the residual add in the epilogue, MLP (GEMM, GELU / QuickGELU, GEMM + residual).
77 tokens per prompt make every launch latency-bound; the point is that the stage runs on the same device-resident program
(CUDA-graph replay) instead of eager PyTorch.  No CPU fallback.  Precision modes: "bf16" (gate 1e-2) and "fp32" (gate 1e-4).
"""
from __future__ import annotations

import json
import os
from dataclasses import dataclass

import torch
from torch import nn

from ._lib import F32_T
from .program import GraphRunner, KernelWeights, LaunchProgram, ProgramModule


@dataclass
class CLIPTextConfig:
    """reference: models/clip/openclip.py:11-51 (same fields and defaults: OpenCLIP ViT-H text tower)."""
    attention_dropout: float = 0.0
    bos_token_id: int = 0
    dropout: float = 0.0
    eos_token_id: int = 2
    hidden_act: str = "gelu"
    hidden_size: int = 1024
    initializer_factor: float = 1.0
    initializer_range: float = 0.02
    intermediate_size: int = 4096
    layer_norm_eps: float = 1e-05
    max_position_embeddings: int = 77
    num_attention_heads: int = 16
    num_hidden_layers: int = 23
    pad_token_id: int = 1
    projection_dim: int = 512
    torch_dtype: str = "float32"
    vocab_size: int = 49408

    @classmethod
    def from_dict(cls, data):
        return cls(**{k: data[k] for k in cls.__dataclass_fields__ if k in data})


def text_param_spec(kind, vocab, hidden, heads, layers, inter, max_len):
    """(name, shape) in the reference's registration order (openclip.py:53-138 / clip.py:8-94)."""
    c = hidden
    attn = lambda p: [(f"{p}.{n}_proj.{l}", (c, c) if l == "weight" else (c,)) for n in ("q", "k", "v", "out") for l in ("weight", "bias")]
    ln = lambda p: [(f"{p}.weight", (c,)), (f"{p}.bias", (c,))]
    if kind == "openclip":
        s = [("embeddings.token_embedding.weight", (vocab, c)), ("embeddings.position_embedding.weight", (max_len, c))]
        for i in range(layers):
            p = f"encoder.layers.{i}"
            s += ln(f"{p}.layer_norm1") + ln(f"{p}.layer_norm2")
            s += [(f"{p}.mlp.fc1.weight", (inter, c)), (f"{p}.mlp.fc1.bias", (inter,)), (f"{p}.mlp.fc2.weight", (c, inter)), (f"{p}.mlp.fc2.bias", (c,))]
            s += attn(f"{p}.self_attn")
        return s + ln("final_layer_norm")
    s = [("text_embedding.embedding.weight", (vocab, c)), ("text_embedding.position_embedding.weight", (max_len, c))]
    for i in range(layers):
        p = f"encoder_layers.{i}"
        s += attn(f"{p}.self_attn") + ln(f"{p}.layernorm_1")
        s += [(f"{p}.ffn.0.weight", (inter, c)), (f"{p}.ffn.0.bias", (inter,)), (f"{p}.ffn.2.weight", (c, inter)), (f"{p}.ffn.2.bias", (c,))]
        s += ln(f"{p}.layernorm_2")
    return s + ln("final_layer_norm")


# key templates of one layer for the two reference classes
_KEYS = {
    "openclip": dict(tok="embeddings.token_embedding.weight", pos="embeddings.position_embedding.weight", layer="encoder.layers.{i}",
                     ln1="layer_norm1", ln2="layer_norm2", fc1="mlp.fc1", fc2="mlp.fc2", act=1),
    "clip": dict(tok="text_embedding.embedding.weight", pos="text_embedding.position_embedding.weight", layer="encoder_layers.{i}",
                 ln1="layernorm_1", ln2="layernorm_2", fc1="ffn.0", fc2="ffn.2", act=2),
}


class TextWeights(KernelWeights):
    """Kernel-layout copies of the parameters on one device for one precision (q|k|v fused, GEMM weights k-block-major bf16)."""

    def _pack(self, net):
        sd, t, dev, wdt = self.sd, self.t, self.dev, self.wdt
        K = _KEYS[net.kind]
        t["tok"], t["pos"] = dev(sd[K["tok"]]), dev(sd[K["pos"]])
        for i in range(net.layers):
            p = K["layer"].format(i=i)
            for j, nm in ((1, K["ln1"]), (2, K["ln2"])):
                t[f"{i}.ln{j}.g"], t[f"{i}.ln{j}.b"] = dev(sd[f"{p}.{nm}.weight"]), dev(sd[f"{p}.{nm}.bias"])
            t[f"{i}.qkv.w"] = dev(torch.cat([sd[f"{p}.self_attn.{n}_proj.weight"] for n in "qkv"], 0), wdt)
            t[f"{i}.qkv.b"] = dev(torch.cat([sd[f"{p}.self_attn.{n}_proj.bias"] for n in "qkv"], 0))
            t[f"{i}.o.w"], t[f"{i}.o.b"] = dev(sd[f"{p}.self_attn.out_proj.weight"], wdt), dev(sd[f"{p}.self_attn.out_proj.bias"])
            t[f"{i}.fc1.w"], t[f"{i}.fc1.b"] = dev(sd[f"{p}.{K['fc1']}.weight"], wdt), dev(sd[f"{p}.{K['fc1']}.bias"])
            t[f"{i}.fc2.w"], t[f"{i}.fc2.b"] = dev(sd[f"{p}.{K['fc2']}.weight"], wdt), dev(sd[f"{p}.{K['fc2']}.bias"])
        t["lnf.g"], t["lnf.b"] = dev(sd["final_layer_norm.weight"]), dev(sd["final_layer_norm.bias"])


class TextEncoderProgram(LaunchProgram):
    """One forward for fixed (B, S): openclip.py:133-137 / clip.py:28-34 as a flat launch list."""

    IO_REGIONS = (("out", "out"), ("ids", "ids_in"))

    def _build(self, S):
        net, B = self.net, self.B
        t, lib = self.pw.t, self.lib
        Cc, heads, inter = net.hidden, net.heads, net.inter
        D, M = Cc // heads, B * S
        es = 4 if self.act == F32_T else 2
        dev = self.device
        self.ids_in = torch.zeros((B, S), dtype=torch.int64, device=dev)
        x = self.pool.get(M, Cc, F32_T)
        self._emit(lib.sdk_embed_tokens, self.ids_in.data_ptr(), t["tok"].data_ptr(), t["pos"].data_ptr(), x.data_ptr(), M, S, Cc, net.vocab)
        for i in range(net.layers):
            n1 = self._ln(x, t[f"{i}.ln1.g"], t[f"{i}.ln1.b"], M, Cc, net.eps)
            qkv, _, _ = self._conv([(n1, Cc)], t[f"{i}.qkv.w"], t[f"{i}.qkv.b"], 1, 1, M, 3 * Cc, out_code=self.act)
            self.pool.put(n1)
            base = qkv.data_ptr()
            ao = self._attention(base, 3 * Cc, S * 3 * Cc, base + Cc * es, 3 * Cc, S * 3 * Cc, base + 2 * Cc * es, 3 * Cc, S * 3 * Cc,
                                 B, heads, S, S, D, Cc, causal=True)                       # lookahead_mask=True (openclip.py:97, clip.py:81)
            self.pool.put(qkv)
            x2, _, _ = self._conv([(ao, Cc)], t[f"{i}.o.w"], t[f"{i}.o.b"], 1, 1, M, Cc, residual=x)
            self.pool.put(ao)
            self.pool.put(x)
            n2 = self._ln(x2, t[f"{i}.ln2.g"], t[f"{i}.ln2.b"], M, Cc, net.eps)
            h, _, _ = self._conv([(n2, Cc)], t[f"{i}.fc1.w"], t[f"{i}.fc1.b"], 1, 1, M, inter)
            self.pool.put(n2)
            g = self.pool.get(M, inter, self.act)
            self._emit(lib.sdk_activation, h.data_ptr(), g.data_ptr(), self.act, M * inter, _KEYS[net.kind]["act"])
            self.pool.put(h)
            x, _, _ = self._conv([(g, inter)], t[f"{i}.fc2.w"], t[f"{i}.fc2.b"], 1, 1, M, Cc, residual=x2)
            self.pool.put(g)
            self.pool.put(x2)
        self.out = torch.empty((B, S, Cc), dtype=torch.float32, device=dev)
        self._emit(lib.sdk_layernorm, x.data_ptr(), t["lnf.g"].data_ptr(), t["lnf.b"].data_ptr(), float(net.eps), self.out.data_ptr(), F32_T, M, Cc)
        self.pool.put(x)


class _TextBase(ProgramModule):
    """Shared machinery of the two reference text-encoder classes."""

    def _setup(self, kind, vocab, hidden, heads, layers, inter, max_len, eps):
        if hidden % heads or hidden // heads not in (40, 64, 80, 160) or hidden % 64:
            raise ValueError(f"hidden_size {hidden} / heads {heads}: head_dim must be 40, 64, 80 or 160 and hidden_size a multiple of 64")
        self.kind, self.vocab, self.hidden, self.heads, self.layers, self.inter, self.max_len, self.eps = kind, vocab, hidden, heads, layers, inter, max_len, eps
        self._init_params(text_param_spec(kind, vocab, hidden, heads, layers, inter, max_len))

    def gradient_checkpointing_enabled(self, enabled=False):       # reference API no-ops (clip.py:19-27)
        return None

    def enable_flash_attn(self):
        return None

    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """token ids (B, S <= max_len) int -> (B, S, hidden) fp32 (openclip.py:133-137 / clip.py:28-34)."""
        if not isinstance(x, torch.Tensor) or not x.is_cuda:
            raise RuntimeError("text encoder: the B200 path only runs on CUDA tensors; there is no CPU fallback "
                               f"(got ids on {getattr(x, 'device', type(x))})")
        if x.dim() != 2 or x.shape[1] > self.max_len:
            raise RuntimeError(f"expected token ids of shape (B, S <= {self.max_len}), got {tuple(x.shape)}")
        B, S = x.shape
        dev = x.device
        key = (str(dev), self.precision)
        pw = self._packed.get(key)
        if pw is None:
            pw = self._packed[key] = TextWeights(self, dev, self.precision)
        pkey = key + (B, S)
        run = self._plans.get(pkey)
        if run is None:
            run = self._plans[pkey] = GraphRunner(TextEncoderProgram(self, pw, B, S), self.use_cuda_graph)
        run.prog.ids_in.copy_(x.to(torch.int64), non_blocking=True)
        run.run()
        return run.prog.out.clone()


class CLIPTextModel(_TextBase):
    """Drop-in for models/clip/openclip.py:107-138."""

    def __init__(self, cfg: CLIPTextConfig = None):
        super().__init__()
        self.cfg = cfg if cfg is not None else CLIPTextConfig()
        c = self.cfg
        self._setup("openclip", c.vocab_size, c.hidden_size, c.num_attention_heads, c.num_hidden_layers, c.intermediate_size,
                    c.max_position_embeddings, c.layer_norm_eps)


class TextEncoder(_TextBase):
    """Drop-in for models/clip/clip.py:8-34 (CLIP ViT-L text tower: 12 layers, 12 heads, QuickGELU)."""

    def __init__(self, n_vocab: int = 49408, embed_dim: int = 768, max_len: int = 77, num_layers: int = 12):
        super().__init__()
        self._setup("clip", n_vocab, embed_dim, 12, num_layers, embed_dim * 4, max_len, 1e-5)


class OpenCLIP(nn.Module):
    """Drop-in for models/clip/openclip.py:140-172: ``.text_model`` is what the pipeline calls."""

    def __init__(self):
        super().__init__()
        self.text_model = CLIPTextModel()

    @staticmethod
    def from_pretrained(text_encoder_pretrained_dir: str = "", image_encoder_pretrained_path: str = "", device: str = 'cpu'):
        from safetensors.torch import load_file
        with open(os.path.join(text_encoder_pretrained_dir, "config.json")) as f:
            cfg = CLIPTextConfig.from_dict(json.load(f))
        sd = load_file(os.path.join(text_encoder_pretrained_dir, "model.safetensors"), device=device)
        sd.pop("text_model.embeddings.position_ids", None)
        model = OpenCLIP.__new__(OpenCLIP)
        nn.Module.__init__(model)
        model.text_model = CLIPTextModel(cfg=cfg)
        model.load_state_dict(sd, strict=True)
        return model

    def encode_image(self):
        pass

    def encode_text(self, input_ids: torch.Tensor) -> torch.Tensor:
        return self.text_model(input_ids)

