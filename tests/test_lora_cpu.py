"""CPU suite: LoRA file parsing (kohya and PEFT) and the LoRA target table against the weight packer -- no device work."""
import re

import pytest
import torch

from oracle import unet_oracle as UO
from stable_diffusion_pytorch_b200 import UNet, lora
from stable_diffusion_pytorch_b200.arch import build_arch
from stable_diffusion_pytorch_b200.unet import PackedWeights

from lora_synth import make_adapter

ARCHS = {"sd15": (UO.SD15, False), "sd21": (UO.SD21, True)}
BLOCKS = [320, 640, 1280, 1280]
TYPES = ["CrossAttnDownBlock2D"] * 3 + ["DownBlock2D"]


def arch_of(name):
    cfg, _ = ARCHS[name]
    return build_arch(cfg["attention_head_dim"], cfg["cross_attention_dim"], 4, 4, BLOCKS, TYPES, 320, None, 1e-5)


@pytest.mark.parametrize("name", sorted(ARCHS))
@pytest.mark.parametrize("fmt,alpha", [("kohya", None), ("kohya", 3.0), ("peft", None)])
def test_parse_every_target(name, fmt, alpha):
    a = arch_of(name)
    sd, truth = make_adapter(a, fmt, rank=6, alpha=alpha, seed=1, linear_proj=ARCHS[name][1], dtype=torch.float16)
    te = {"lora_te_text_model_encoder_layers_0_mlp_fc1.lora_down.weight": torch.zeros(4, 768),
          "lora_te2_x.alpha": torch.tensor(1.0), "text_encoder.layer.lora_A.weight": torch.zeros(2, 3)}
    sd.update(te)
    mods, unapplied = lora.read_adapter(sd, a)
    assert sorted(unapplied) == sorted(te)
    assert set(mods) == set(truth) == set(lora.targets(a).values())
    kinds = set()
    for ref, m in mods.items():
        up, down, mult = truth[ref]
        assert m.up.dtype == m.down.dtype == torch.float32                       # fp16 factors are upcast
        assert torch.equal(m.up.double(), up)
        assert torch.equal(m.down.double().reshape(down.shape[0], -1), down.reshape(down.shape[0], -1))
        assert m.mult == (3.0 / 6 if alpha else 1.0) == mult
        kinds.add(ref)
    if fmt == "kohya" and alpha is None:
        assert any(k.endswith(".alpha") for k in sd)                               # both forms present: explicit and default alpha
    # every row of the table: attention q/k/v/out of both attentions, GEGLU and its output, proj_in/out, ResBlock convs, shortcut,
    # time projection, down- and upsampler convs
    for leaf in ("attn1.q_proj", "attn1.k_proj", "attn1.v_proj", "attn1.out_proj", "attn2.q_proj", "attn2.k_proj", "attn2.v_proj",
                 "attn2.out_proj", "ffn.0.proj", "ffn.1", "conv_input", "conv_output", "conv_1", "conv_2", "proj_input", "t_embed",
                 "downsample.conv", "upsample.conv"):
        assert any(f".{leaf}.weight" in k for k in kinds), leaf


def test_parse_scale_from_safetensors_file(tmp_path):
    from safetensors.torch import save_file
    a = arch_of("sd15")
    sd, truth = make_adapter(a, "kohya", rank=8, alpha=2.0, select=("attn2.to_k",), dtype=torch.bfloat16)
    path = str(tmp_path / "a.safetensors")
    save_file({k: v.contiguous() for k, v in sd.items()}, path)
    mods, unapplied = lora.read_adapter(path, a)
    assert not unapplied and set(mods) == set(truth) and len(mods) == 16
    assert all(m.mult == 0.25 for m in mods.values())


def _bad(a, key, val, extra=None):
    sd = {key: val}
    sd.update(extra or {})
    with pytest.raises(ValueError, match=re.escape(key)):
        lora.read_adapter(sd, a)


def test_parse_errors_name_the_key():
    a = arch_of("sd15")
    z = torch.zeros
    up_key = "lora_unet_down_blocks_0_attentions_0_transformer_blocks_0_attn1_to_q.lora_up.weight"
    down_key = up_key.replace("lora_up", "lora_down")
    for key in ("lora_unet_input_blocks_1_1_proj_in.lora_down.weight",             # LDM-style names
                "lora_unet_conv_in.lora_down.weight", "lora_unet_time_embedding_linear_1.lora_down.weight",
                "lora_unet_down_blocks_0_resnets_0_norm1.lora_down.weight", "unet.conv_out.lora_A.weight",
                "unet.mid_block.attentions.0.norm.lora_B.weight",
                down_key.replace("lora_down.weight", "dora_scale"),                  # DoRA: not supported
                "unet.down_blocks.0.attentions.0.transformer_blocks.0.attn1.to_q.lora_magnitude_vector"):
        _bad(a, key, z(4, 320))
    _bad(a, up_key, z(320, 4))                                                      # no down factor
    _bad(a, up_key, z(320, 3), {down_key: z(4, 320)})                               # ranks disagree
    _bad(a, up_key, z(321, 4), {down_key: z(4, 320)})                               # N does not fit
    _bad(a, down_key, z(4, 768), {up_key: z(320, 4)})                               # K does not fit
    conv = "lora_unet_down_blocks_0_resnets_0_conv1"
    _bad(a, f"{conv}.lora_down.weight", z(4, 320 * 9), {f"{conv}.lora_up.weight": z(320, 4, 1, 1)})     # LoCon down must be 4-D


def _emulate(dst, op):
    """sdk_lora_merge with r = 0, in torch: the base rows cast to the packed dtype, written through the layout and row map."""
    base = op["base"]
    n, k = base.shape
    rows = op["row_off"] + op["row_step"] * torch.arange(n)
    v = base.to(dst.dtype)
    if op["layout"] == 0:
        dst.view(-1, k)[rows] = v
    else:
        blk = dst.view(-1)[op["offset"]: op["offset"] + k * op["dst_rows"]].view(k // 64, op["dst_rows"], 64)
        blk[:, rows, :] = v.view(n, k // 64, 64).permute(1, 0, 2)


@pytest.mark.parametrize("name", sorted(ARCHS))
def test_target_table_rebuilds_the_packer_output(name):
    """Every packed tensor a LoRA can address, rebuilt from the raw parameters through the table's row maps, layouts and parity
    fold, equals the packer's output bit for bit (fp32 and bf16 packs)."""
    cfg, _ = ARCHS[name]
    torch.manual_seed(0)
    net = UNet(attention_head_dim=cfg["attention_head_dim"], cross_attention_dim=cfg["cross_attention_dim"])
    a, params = net.arch, dict(net.named_parameters())
    for precision in ("fp32", "bf16"):
        pw = PackedWeights(net, "cpu", precision)
        rebuilt, layouts = {}, set()
        for ref in lora.targets(a).values():
            for op in lora.merge_ops(a, pw, ref, params[ref], []):
                key = next(k for k, t in pw.t.items() if t is op["dst"])
                out = rebuilt.setdefault(key, torch.full_like(op["dst"], float("nan")))
                _emulate(out, op)
                layouts.add((op["dst"].dtype, op["layout"]))
        for key, t in rebuilt.items():
            bits = torch.int32 if t.dtype == torch.float32 else torch.int16
            assert torch.equal(t.view(bits), pw.t[key].view(bits)), (precision, key)
        assert "tb.w" in rebuilt and any(k.endswith(".qkv.w") for k in rebuilt)
        if precision == "bf16":
            assert "kv2_all.w" in rebuilt and sum(k.endswith(".w_up2") for k in rebuilt) == 3
            assert layouts == {(torch.bfloat16, 0), (torch.bfloat16, 1)}                 # tb.w row-major, the rest k-block-major
        else:
            assert sum(k.endswith(".kv2.w") for k in rebuilt) == 16 and layouts == {(torch.float32, 0)}
        del pw


def test_use_lora_still_raises():
    with pytest.raises(NotImplementedError, match="merge LoRA deltas"):
        UNet(use_lora=True)
