"""B200-native VAE DECODER — drop-in for ``VAE.decode`` of the reference's ``models/vae/vae.py`` (SURVEY §8(f) rank 1: the stage
right after the denoising loop, models/diffusion.py:118,241).

Same construction as the UNet (unet.py): parameters under the reference's names (all 248 of them, encoder included, so that
``load_state_dict(strict=True)`` of a reference checkpoint works), and ``decode`` runs a pre-planned launch list over NHWC
activations on the SAME C-ABI kernels — tcgen05 implicit-GEMM 3x3 convs with the consumer GroupNorm's statistics reduced in the
epilogue, the 1x1 shortcut as a second K segment, nearest-2x upsample folded into the conv as four parity convs, GroupNorm(+SiLU)
apply.  The single-head head_dim = 512 attention of the mid block (vae.py:42-134) runs as three tensor-core GEMMs per sample
(Q K^T, V^T, P V) around a row-softmax kernel: its 4096 x 4096 score matrix is 64 MB, a rounding error beside the 512^2 convs.

There is no CPU / PyTorch fallback; the encoder (``VAE.encode``) is outside the hot-path scope and raises.
Precision modes as for the UNet: "bf16" (tensor cores, gate rel-L2 <= 1e-2) and "fp32" (FFMA, gate <= 1e-4).
"""
from __future__ import annotations

import ctypes as C
import json
import math
import os

import torch

from ._lib import F32_T, ConvParams
from .arch import vae_decoder_blocks, vae_param_spec
from .program import GraphRunner, KernelWeights, LaunchProgram, ProgramModule

SCALE = 0.18215                                            # models/vae/vae.py:271


class VAEWeights(KernelWeights):
    """Kernel-layout copies of the decoder's parameters on one device for one precision."""

    def _pack(self, net: "VAE"):
        sd, t, dev, wdt = self.sd, self.t, self.dev, self.wdt
        # post_quant_conv (1x1, 4 -> 4) and conv_in (3x3, 4 -> 512): fp32 FFMA kernels in both modes (K = 4 / 36)
        t["pq.w"] = dev(sd["post_quant_conv.weight"].reshape(sd["post_quant_conv.weight"].shape[0], -1))
        t["pq.b"] = dev(sd["post_quant_conv.bias"])
        self.conv_in("decoder.conv_in")

        def res(p):
            self.res_block(p, ("norm1", "norm2"), ("conv1", "conv2"), "conv_shortcut")

        res("decoder.mid_block.resnets.0")
        res("decoder.mid_block.resnets.1")
        a = "decoder.mid_block.attentions.0"
        t["attn.gn.g"], t["attn.gn.b"] = dev(sd[f"{a}.group_norm.weight"]), dev(sd[f"{a}.group_norm.bias"])
        for n in ("query", "key", "proj_attn"):
            t[f"attn.{n}.w"], t[f"attn.{n}.b"] = dev(sd[f"{a}.{n}.weight"], wdt), dev(sd[f"{a}.{n}.bias"])
        # V is produced TRANSPOSED ([C][S] = W_v x^T: W_v is the A operand, the normalised tokens the B operand); its bias moves to
        # the P V GEMM because the softmax rows sum to one:  P (V + 1 b^T) = P V + b^T
        t["attn.value.a"] = sd[f"{a}.value.weight"].to(device=self.device, dtype=wdt).contiguous()    # [C][C] row-major "activation"
        t["attn.value.b"] = dev(sd[f"{a}.value.bias"])
        for j, cin, cout, up in vae_decoder_blocks():
            for k in range(3):
                res(f"decoder.up_blocks.{j}.resnets.{k}")
            if up:
                self.upsample_conv(f"decoder.up_blocks.{j}.upsamplers.0.conv")
        t["out.gn.g"], t["out.gn.b"] = dev(sd["decoder.conv_norm_out.weight"]), dev(sd["decoder.conv_norm_out.bias"])
        t["out.w"], t["out.b"] = self.conv_w("decoder.conv_out.weight", wdt), dev(sd["decoder.conv_out.bias"])


class VAEDecodeProgram(LaunchProgram):
    """``VAE.decode`` for a fixed (B, h, w) latent shape as a flat launch list (models/vae/vae.py:229-241,270-274)."""

    IO_REGIONS = (("out", "out"), ("z", "z_in"))

    def __init__(self, net: "VAE", pw: VAEWeights, B, h, w):
        if h % 8 or w % 8:
            raise RuntimeError(f"latent {h}x{w}: height and width must be multiples of 8 (token count of the mid-block attention)")
        super().__init__(net, pw, B, h, w)

    def _vattention(self, x, Cc, B, H, W):
        """AttentionBlock (vae.py:121-134): GN -> q, k, v (with bias) -> softmax(q k^T / sqrt(C)) v -> proj -> + x, ONE head of
        dimension C.  Scores and P V are GEMMs whose B operand is an activation (row-major [N][K]); V is produced transposed."""
        t, S = self.pw.t, H * W
        M = B * S
        a, _ = self._gn([(x, Cc)], B, S, t["attn.gn.g"], t["attn.gn.b"], 1e-6, False)
        q, _, _ = self._conv([(a, Cc)], t["attn.query.w"], t["attn.query.b"], 1, 1, M, Cc, out_code=self.act)
        k, _, _ = self._conv([(a, Cc)], t["attn.key.w"], t["attn.key.b"], 1, 1, M, Cc, out_code=self.act)
        o = self.pool.get(M, Cc, self.act)
        vT = self.pool.get(Cc, S, self.act)
        sc = self.pool.get(S, S, F32_T)
        pr = self.pool.get(S, S, self.act)
        scale = 1.0 / math.sqrt(Cc)
        for b in range(B):                                     # per sample: the score matrix buffers are reused in stream order
            ab, qb, kb_, ob = a[b * S:(b + 1) * S], q[b * S:(b + 1) * S], k[b * S:(b + 1) * S], o[b * S:(b + 1) * S]
            # V^T [C][S] = W_v (A operand, C rows) x tokens^T (B operand = the normalised tokens, row-major [S][C]); bias deferred
            self._conv([(t["attn.value.a"], Cc)], ab, None, 1, 1, Cc, S, out_code=self.act, out=vT, w_rowmajor=True)
            self._conv([(qb, Cc)], kb_, None, 1, 1, S, S, out_code=F32_T, out=sc, w_rowmajor=True)                # q k^T
            self._emit(self.lib.sdk_softmax_rows, sc.data_ptr(), pr.data_ptr(), self.act, S, S, float(scale))
            self._conv([(pr, S)], vT, t["attn.value.b"], 1, 1, S, Cc, out_code=self.act, out=ob, w_rowmajor=True)    # P V + b_v
        for buf in (vT, sc, pr, q, k, a):
            self.pool.put(buf)
        out, _, _ = self._conv([(o, Cc)], t["attn.proj_attn.w"], t["attn.proj_attn.b"], B, H, W, Cc, residual=x, want_stats=True)
        self.pool.put(o)
        return out

    # ---- whole decoder --------------------------------------------------------------------
    def _build(self, h, w):
        t, lib = self.pw.t, self.lib
        B = self.B
        dev, f32 = self.device, torch.float32
        self.h, self.w = h, w
        # statistics kernels of the fp32 mode (bf16 takes them from the GEMM epilogues): sized for the final 8h x 8w image
        self.gn_ws = torch.zeros(int(lib.sdk_groupnorm_workspace_bytes(B, 64 * h * w)), dtype=torch.uint8, device=dev)
        self.gn_stats = torch.empty((B, 32, 2), dtype=f32, device=dev)
        zc = t["pq.w"].shape[0]
        top = t["conv_in.b"].shape[0]
        self.z_in = torch.empty((B, zc, h, w), dtype=f32, device=dev)
        zs = torch.empty_like(self.z_in)
        self.keep.append(zs)
        # z / 0.18215 (vae.py:271): the one-step kernel with sigma = 0 is exactly that division
        self._emit(lib.sdk_x0_from_eps, self.z_in.data_ptr(), self.z_in.data_ptr(), 0.0, float(SCALE), zs.data_ptr(), self.z_in.numel())
        zn = self.pool.get(B * h * w, zc, F32_T)
        self._emit(lib.sdk_nchw_to_nhwc, zs.data_ptr(), zn.data_ptr(), B, B, zc, h * w)
        # post_quant_conv 1x1 (vae.py:272): K = 4 -> FFMA kernel in both modes
        zq = self.pool.get(B * h * w, zc, F32_T)
        p = ConvParams()
        p.src0, p.C0, p.src1, p.C1 = zn.data_ptr(), zc, 0, 0
        p.weight, p.bias, p.tbias, p.tb_stride, p.residual, p.out = t["pq.w"].data_ptr(), t["pq.b"].data_ptr(), 0, 0, 0, zq.data_ptr()
        p.B, p.Hin, p.Win, p.Hout, p.Wout, p.ksize, p.stride, p.upsample, p.N = B, h, w, h, w, 1, 1, 0, zc
        p.in_dtype, p.out_dtype, p.out_nchw, p.geglu = F32_T, F32_T, 0, 0
        self.keep.append(p)
        self._emit(lib.sdk_conv_gemm_f32, C.byref(p))
        self.pool.put(zn)
        # conv_in 3x3, 4 -> 512 (vae.py:231): the K = 36 kernel, which also reduces the first GroupNorm's statistics
        x = self._conv_in(zq, zc, B, h, w, top)
        self.pool.put(zq)
        # mid block (vae.py:233-235)
        y = self._resblock("decoder.mid_block.resnets.0", [(x, top)], top, 1e-6, B, h, w)
        self.pool.put(x)
        x = self._vattention(y, top, B, h, w)
        self.pool.put(y)
        y = self._resblock("decoder.mid_block.resnets.1", [(x, top)], top, 1e-6, B, h, w)
        self.pool.put(x)
        x, xc = y, top
        # up blocks (vae.py:237-239)
        for j, cin, cout, up in vae_decoder_blocks():
            for k in range(3):
                y = self._resblock(f"decoder.up_blocks.{j}.resnets.{k}", [(x, cin if k == 0 else cout)], cout, 1e-6, B, h, w)
                self.pool.put(x)
                x, xc = y, cout
            if up:
                y, h, w = self._upsample_conv(f"decoder.up_blocks.{j}.upsamplers.0.conv", x, xc, B, h, w)
                self.pool.put(x)
                x = y
        # GN + SiLU + conv_out 128 -> 3, written straight to NCHW (vae.py:239-241)
        self.out = torch.empty((B, t["out.b"].shape[0], h, w), dtype=f32, device=dev)
        ao, _ = self._gn([(x, xc)], B, h * w, t["out.gn.g"], t["out.gn.b"], 1e-6, True)
        self.pool.put(x)
        self._conv([(ao, xc)], t["out.w"], t["out.b"], B, h, w, t["out.b"].shape[0], k=3, out=self.out, out_nchw=True)
        self.pool.put(ao)


class VAE(ProgramModule):
    """Drop-in for the reference ``VAE`` (models/vae/vae.py:244-288), decode path."""

    def __init__(self, in_channels: int = 3, z_channels: int = 4):
        super().__init__()
        self.in_channels, self.z_channels = in_channels, z_channels
        self._init_params(vae_param_spec(in_channels, z_channels))

    def encode(self, x, noise=None, generator=None):
        raise NotImplementedError("VAE.encode is outside the hot-path scope of this package (SURVEY 8(f)): run the reference encoder")

    def decode(self, z: torch.Tensor) -> torch.Tensor:
        """reference: vae.py:270-274.  z (B, z_channels, h, w) float on CUDA -> image (B, 3, 8h, 8w), same dtype."""
        if not isinstance(z, torch.Tensor) or not z.is_cuda:
            raise RuntimeError("VAE.decode: the B200 VAE only runs on CUDA tensors; there is no CPU fallback "
                               f"(got z on {getattr(z, 'device', type(z))})")
        if z.dim() != 4 or z.shape[1] != self.z_channels:
            raise RuntimeError(f"expected z of shape (B,{self.z_channels},h,w), got {tuple(z.shape)}")
        B, _, h, w = z.shape
        dev = z.device
        key = (str(dev), self.precision)
        pw = self._packed.get(key)
        if pw is None:
            pw = self._packed[key] = VAEWeights(self, dev, self.precision)
        pkey = key + (B, h, w)
        plan = self._plans.get(pkey)
        if plan is None:
            plan = self._plans[pkey] = GraphRunner(VAEDecodeProgram(self, pw, B, h, w), self.use_cuda_graph)
        plan.prog.z_in.copy_(z, non_blocking=True)
        plan.run()
        return plan.prog.out.clone().to(z.dtype)

    @staticmethod
    def from_pretrained(pretrained_path: str, device: str = 'cpu'):
        """reference: vae.py:276-288 (config.json + safetensors with the reference's parameter names)."""
        from safetensors.torch import load_file
        with open(os.path.join(pretrained_path, "config.json"), "r") as f:
            cfg = json.load(f)
        model = VAE(in_channels=cfg['in_channels'], z_channels=cfg['latent_channels'])
        sd = load_file(os.path.join(pretrained_path, 'diffusion_pytorch_model.safetensors'), device=device)
        model.load_state_dict(sd, strict=True)
        return model
