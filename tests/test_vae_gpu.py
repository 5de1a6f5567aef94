"""GPU parity of the VAE decoder (SURVEY 8(f) rank 1) against golden images produced by the UNMODIFIED reference
(tests/golden/make_golden_vae.py -> vae_golden.npz) and, at full size, against the CPU oracle.

Gates: fp32 mode rel-L2 <= 1e-4 (measured 4.6e-6).  bf16 mode: the decoder is a chain of ~38 tensor-core GEMM stages with NO long
skip connections, each adding ~1.7e-3 of independent bf16 operand rounding, so the image lands at sqrt(38) * 1.7e-3 ~ 1.0e-2 of
the fp32 result (measured 0.99e-2 ... 1.01e-2 at every size) -- exactly AT north_star's 1e-2 figure, which is stated for the final
LATENT of the denoising loop.  The bf16 image gate here is therefore 1.5e-2, with the measured value printed."""
import os

import numpy as np
import pytest
import torch

from oracle import vae_oracle as VO
from stable_diffusion_pytorch_b200 import VAE
from stable_diffusion_pytorch_b200.program import GraphRunner
from stable_diffusion_pytorch_b200.vae import VAEDecodeProgram, VAEWeights

pytestmark = pytest.mark.gpu
FP32_TOL, BF16_TOL = 1e-4, 1.5e-2
# the mid-block attention branch alone, with sharpened weights: bf16 measured 2.7e-3 ... 3.5e-3 on a B200 (1000 W); replacing the
# softmax by 1/S or dropping the value bias moves it by 0.078 ... 0.28
ATTN_BF16_TOL = 6e-3


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def vae(dev):
    net = VAE()
    sd = VO.make_state_dict(3)
    assert list(net.state_dict().keys()) == list(sd.keys())              # the reference's 248 names, in its order
    net.load_state_dict(sd, strict=True)
    return net.to(dev).eval(), sd


@pytest.mark.parametrize("precision,tol", [("fp32", FP32_TOL), ("bf16", BF16_TOL)])
def test_decode_matches_reference_golden(vae, golden_dir, dev, precision, tol):
    net, _ = vae
    net.set_precision(precision)
    g = np.load(os.path.join(golden_dir, "vae_golden.npz"))
    with torch.no_grad():
        for name in ("z8", "z8x16", "z24"):
            z = torch.from_numpy(g[name]).to(dev)
            y = net.decode(z)
            e = rel_l2(y.cpu().numpy(), g[f"img_{name}"])
            print(f"VAE.decode {precision} {name} -> {tuple(y.shape)}: rel-L2 {e:.3e}")
            assert y.shape == g[f"img_{name}"].shape and y.dtype == torch.float32 and e < tol
            y2 = net.decode(z)                                              # second call: CUDA-graph capture + replay
            y3 = net.decode(z)
            assert torch.equal(y2, y) and torch.equal(y3, y)
    net.set_precision("bf16")


def test_decode_full_size_bf16_vs_oracle(vae, dev):
    """512x512 image from a 64x64 latent (BASELINE configs 2/3/5): tcgen05 convs with the folded upsample, 4096-token attention."""
    net, sd = vae
    net.set_precision("bf16")
    g = torch.Generator().manual_seed(11)
    z = torch.randn((1, 4, 64, 64), generator=g) * 0.18215 * 4.0
    with torch.no_grad():
        y = net.decode(z.to(dev)).cpu()
        want = VO.decode(sd, z)
    e = rel_l2(y.numpy(), want.numpy())
    print(f"VAE.decode bf16 64x64 latent -> 512x512: rel-L2 {e:.3e}")
    assert y.shape == (1, 3, 512, 512) and e < BF16_TOL


def test_decode_rejects_cpu_and_bad_shapes(vae, dev):
    net, _ = vae
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        net.decode(torch.zeros((1, 4, 8, 8)))
    with pytest.raises(RuntimeError):
        net.decode(torch.zeros((1, 3, 8, 8), device=dev))
    with pytest.raises(RuntimeError, match="multiples of 8"):
        net.decode(torch.zeros((1, 4, 12, 8), device=dev))
    with pytest.raises(NotImplementedError):
        net.encode(torch.zeros((1, 3, 64, 64), device=dev))


class _MidAttentionProgram(VAEDecodeProgram):
    """The decoder's mid-block attention alone (VAEDecodeProgram._vattention) over an fp32 NHWC input [B*h*w][512], planned as the
    decoder plans it.  In bf16 the decoder's input to this block comes from a GEMM that reduced its per-channel statistics, so the
    input here carries such a table too and the GroupNorm takes the same statistics-from-sums route."""

    def _build(self, h, w):
        lib, B, dev = self.lib, self.B, self.device
        self.gn_ws = torch.zeros(int(lib.sdk_groupnorm_workspace_bytes(B, 64 * h * w)), dtype=torch.uint8, device=dev)
        self.gn_stats = torch.empty((B, 32, 2), dtype=torch.float32, device=dev)
        self.x_in = torch.empty((B * h * w, 512), dtype=torch.float32, device=dev)
        x = self.x_in
        if self.gn_from_sums:
            x._cstats = self._stat_table(B, 512)
            self._emit(lib.sdk_channel_stats, x.data_ptr(), B, h * w, 512, x._cstats.data_ptr())
        self.y = self._vattention(x, 512, B, h, w)


@pytest.fixture(scope="module")
def sharp_attention():
    """VO.make_state_dict(3) with the mid-block attention's query and key weights doubled: with the plain init the softmax is almost
    flat, and a kernel that returned 1/S would move the branch by little more than bf16 rounding."""
    sd = VO.make_state_dict(3)
    p = "decoder.mid_block.attentions.0"
    for n in ("query", "key"):
        sd[f"{p}.{n}.weight"] = sd[f"{p}.{n}.weight"] * 2
    net = VAE()
    net.load_state_dict(sd, strict=True)
    return net, sd, {}


@pytest.mark.parametrize("hw", [8, 24, 64])
@pytest.mark.parametrize("B", [1, 2])
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", ATTN_BF16_TOL)])
def test_mid_attention_block_sharpened(sharp_attention, dev, precision, tol, B, hw):
    """The planned attention block (GroupNorm, q / k / V^T GEMMs, scores, row softmax, P V + b_v, projection + residual) vs the
    oracle's AttentionBlock in float64.  Compared on the attention branch y - x, not the block output, which the residual x
    dominates.  B = 2 reuses the score buffers in stream order; a CUDA-graph replay must reproduce the eager launch bit for bit."""
    net, sd, packed = sharp_attention
    pw = packed.get(precision)
    if pw is None:
        pw = packed[precision] = VAEWeights(net, dev, precision)
    S = hw * hw
    prog = _MidAttentionProgram(net, pw, B, hw, hw)
    g = torch.Generator().manual_seed(171)
    x = torch.randn((B * S, 512), generator=g) * 1.5 + torch.randn((1, 512), generator=g)
    prog.x_in.copy_(x.to(dev))
    prog.launch(prog.ops)
    torch.cuda.synchronize()
    y = prog.y.clone()
    runner = GraphRunner(prog, True)
    for _ in range(3):                                             # eager, capture + replay, replay
        runner.run()
        torch.cuda.synchronize()
        assert torch.equal(prog.y.view(torch.int32), y.view(torch.int32))
    p = "decoder.mid_block.attentions.0"
    sd64 = {k: v.to(dev, torch.float64) for k, v in sd.items() if k.startswith(p)}
    xd = x.to(dev, torch.float64)
    with torch.no_grad():
        y_ref = VO.attention(sd64, p, xd.view(B, hw, hw, 512).permute(0, 3, 1, 2)).permute(0, 2, 3, 1).reshape(B * S, 512)
    e = rel_l2((y.double() - xd).cpu().numpy(), (y_ref - xd).cpu().numpy())
    print(f"VAE mid attention {precision} B={B} {hw}x{hw} (S={S}): branch rel-L2 {e:.3e}")
    assert not torch.isnan(y).any()
    assert e < tol
