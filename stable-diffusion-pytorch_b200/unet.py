"""B200-native SD-1.5 / SD-2.1 conditional UNet — drop-in for the reference's
``models/unet/unet.py`` ``UNet`` (same constructor, same parameter names and shapes so
``load_state_dict(strict=True)`` of reference checkpoints works, same
``forward(x, timestep, cond)``).

Not a module tree of eager ops: ``forward`` runs a pre-planned STEP PROGRAM — a fixed list of
C-ABI kernel launches (include/sdb200.h) over NHWC activations with pre-packed weights and a
liveness-planned activation pool — optionally replayed as a CUDA graph.  There is no PyTorch/CPU
fallback: CPU tensors or a missing kernel library raise.

Precision modes (``net.precision``):
  "fp32"  exact path: FFMA implicit GEMM + fp32 attention          (parity gate rel-L2 <= 1e-4)
  "bf16"  tcgen05/TMEM tensor-core GEMMs, bf16 operands, fp32 accumulate, fp32 residual stream
          and norm statistics                                      (parity gate rel-L2 <= 1e-2)
"""
from __future__ import annotations

import json
import os
from typing import Dict, List, Optional, Union

import torch

from ._lib import BF16_T, F32_T
from . import _lib, lora
from .arch import BLOCK_OUT, Transformer, UNetArch, build_arch, param_spec
from .program import _DT, GraphRunner, KernelWeights, LaunchProgram, ProgramModule


def tensor_version(t: torch.Tensor):
    """``t._version`` or None for inference tensors (``torch.inference_mode()`` tensors do not track a version counter;
    the reference's inpaint path runs under it, models/diffusion.py:328).  None never compares equal to a cached version,
    so such a context is treated as changed on every call."""
    try:
        return t._version
    except RuntimeError:
        return None


def same_context(cond: torch.Tensor, ref, version) -> bool:
    """True when ``cond`` is the tensor object cached as ``ref`` and has not been written since (``version``)."""
    v = tensor_version(cond)
    return cond is ref and v is not None and v == version


# ======================================================================================
# weight packing
# ======================================================================================
class PackedWeights(KernelWeights):
    """Kernel-layout copies of the parameters on one device for one precision.

    conv  [N][Cin][kh][kw] -> [N][kh][kw][Cin]   (K-major rows, NHWC gather order)
    attn1 q|k|v            -> one [3C][C] matrix  (single QKV GEMM)
    attn2 k|v              -> one [2C][Dctx] matrix
    ffn.0.proj             -> rows interleaved (value_j, gate_j) so GEGLU fuses into the epilogue
    t_embed of all 22 ResBlocks -> one [sum Cout][1280] matrix (single batched mat-vec)

    ``version`` counts the in-place LoRA merges into these tensors (UNet.load_lora): results cached from the weights -- the
    cross-attention K/V of a context, the hoisted time projections of a sampling loop -- are recomputed when it changes.
    """

    version = 0

    def _pack(self, net: "UNet"):
        a, sd, t, wdt, dev, conv_w = net.arch, self.sd, self.t, self.wdt, self.dev, self.conv_w
        device, precision = self.device, self.precision
        for k in ("time_embedding.ffn.0.weight", "time_embedding.ffn.0.bias",
                  "time_embedding.ffn.2.weight", "time_embedding.ffn.2.bias"):
            t[k] = dev(sd[k])
        t["tb.w"] = torch.cat([sd[f"{r.prefix}.t_embed.weight"] for r in a.res_blocks], 0).to(device=device, dtype=wdt).contiguous()
        t["tb.b"] = dev(torch.cat([sd[f"{r.prefix}.t_embed.bias"] for r in a.res_blocks], 0))
        self.conv_in("encoder.conv_in")
        for r in a.res_blocks:
            self.res_block(r.prefix, ("groupnorm_1", "groupnorm_2"), ("conv_1", "conv_2"), "proj_input")
        kv_list = []
        for tr in a.transformers:
            p, b, c = tr.prefix, f"{tr.prefix}.transformer_block", tr.c
            t[f"{p}.gn.g"], t[f"{p}.gn.b"] = dev(sd[f"{p}.groupnorm.weight"]), dev(sd[f"{p}.groupnorm.bias"])
            t[f"{p}.in.w"], t[f"{p}.in.b"] = conv_w(f"{p}.conv_input.weight"), dev(sd[f"{p}.conv_input.bias"])
            t[f"{p}.out.w"], t[f"{p}.out.b"] = conv_w(f"{p}.conv_output.weight"), dev(sd[f"{p}.conv_output.bias"])
            for i in (1, 2, 3):
                t[f"{p}.ln{i}.g"], t[f"{p}.ln{i}.b"] = dev(sd[f"{b}.layernorm_{i}.weight"]), dev(sd[f"{b}.layernorm_{i}.bias"])
            t[f"{p}.qkv.w"] = dev(torch.cat([sd[f"{b}.attn1.{n}_proj.weight"] for n in "qkv"], 0), wdt)
            t[f"{p}.o1.w"], t[f"{p}.o1.b"] = dev(sd[f"{b}.attn1.out_proj.weight"], wdt), dev(sd[f"{b}.attn1.out_proj.bias"])
            t[f"{p}.q2.w"] = dev(sd[f"{b}.attn2.q_proj.weight"], wdt)
            if precision != "fp32" and getattr(net, "ln_fold", False):
                # (opt-in, SDB200_LN_FOLD=1) LayerNorm folded into the projection that consumes it (unet.py:137-149):
                #   LN(x) W^T + c = rstd * (x W'^T - mean * colsum) + (c + W beta),  W' = W * gamma (bf16), colsum[n] = sum_k W'[n][k]
                # colsum is taken from the ROUNDED W' so that the mean term cancels exactly against what the tensor core multiplies.
                def fold(key, w, bias, ln):
                    w = w.to(device=device, dtype=torch.float32)
                    gm, bt = sd[f"{b}.layernorm_{ln}.weight"].to(device, torch.float32), sd[f"{b}.layernorm_{ln}.bias"].to(device, torch.float32)
                    wg = (w * gm[None, :]).to(torch.bfloat16)
                    t[f"{p}.{key}.lnw"] = dev(wg, torch.bfloat16)
                    t[f"{p}.{key}.lncs"] = wg.float().sum(1).contiguous()
                    add = w.double() @ bt.double()
                    t[f"{p}.{key}.lnb"] = (add + (bias.to(device).double() if bias is not None else 0.0)).float().contiguous()
                fold("qkv", torch.cat([sd[f"{b}.attn1.{n}_proj.weight"] for n in "qkv"], 0), None, 1)
                fold("q2", sd[f"{b}.attn2.q_proj.weight"], None, 2)
            kv_w = torch.cat([sd[f"{b}.attn2.k_proj.weight"], sd[f"{b}.attn2.v_proj.weight"]], 0)
            if precision == "fp32":
                t[f"{p}.kv2.w"] = dev(kv_w, wdt)
            else:
                kv_list.append((tr.index, kv_w))           # bf16: all 16 context projections become ONE GEMM (see kv2_all.w)
            t[f"{p}.o2.w"], t[f"{p}.o2.b"] = dev(sd[f"{b}.attn2.out_proj.weight"], wdt), dev(sd[f"{b}.attn2.out_proj.bias"])
            w0, b0 = sd[f"{b}.ffn.0.proj.weight"], sd[f"{b}.ffn.0.proj.bias"]      # [8C, C]: rows [value(4C) ; gate(4C)]
            t[f"{p}.ff0.w"] = dev(torch.stack([w0[:4 * c], w0[4 * c:]], 1).reshape(8 * c, c), wdt)
            t[f"{p}.ff0.b"] = dev(torch.stack([b0[:4 * c], b0[4 * c:]], 1).reshape(8 * c))
            if precision != "fp32" and getattr(net, "ln_fold", False):
                fold("ff0", torch.stack([w0[:4 * c], w0[4 * c:]], 1).reshape(8 * c, c), torch.stack([b0[:4 * c], b0[4 * c:]], 1).reshape(8 * c), 3)
            t[f"{p}.ff1.w"], t[f"{p}.ff1.b"] = dev(sd[f"{b}.ffn.1.weight"], wdt), dev(sd[f"{b}.ffn.1.bias"])
        for st in a.down:
            if st.resample is not None:
                p = st.resample.prefix
                t[f"{p}.w"], t[f"{p}.b"] = conv_w(f"{p}.weight"), dev(sd[f"{p}.bias"])
        for st in a.up:
            if st.resample is not None:
                self.upsample_conv(st.resample.prefix)
        # cross-attention K/V projections of every transformer, rows concatenated: the context program is one [Bc*77, dctx] x
        # [sum 2C, dctx]^T GEMM (24960 output columns for SD1.5) instead of 16 launches; kv_off[index] = first column of a layer
        self.kv_off, self.kv_total = {}, 0
        if kv_list:
            for idx, w in kv_list:
                self.kv_off[idx] = self.kv_total
                self.kv_total += w.shape[0]
            t["kv2_all.w"] = dev(torch.cat([w for _, w in kv_list], 0), wdt)
        t["out.gn.g"], t["out.gn.b"] = dev(sd["output.0.weight"]), dev(sd["output.0.bias"])
        t["out.w"], t["out.b"] = conv_w("output.2.weight", wdt), dev(sd["output.2.bias"])


# ======================================================================================
# step program
# ======================================================================================
class StepProgram(LaunchProgram):
    """One UNet forward for fixed (B, H, W, n_timesteps, cond batch, Sk) as a flat launch list.  ``time_ops`` is its time-embedding
    chain (timestep -> self.tb) and ``body_ops`` the forward without it."""

    PROGRAM_IDS = {"ops": 0, "ctx_ops": 1, "time_ops": 2, "body_ops": 3}
    PROGRAM_LOOP_STEP = 4                   # one sampler step of DenoiseLoop.export_engine
    IO_REGIONS = (("x", "x_in"), ("timestep", "t_in"), ("context", "cond_in"), ("out", "out"))

    def __init__(self, net: "UNet", pw: PackedWeights, B, H, W, nt, Bc, Sk, b_src=None):
        if Bc not in (1, B):
            # anything else would silently broadcast the first context rows to every sample (the reference fails in SDPA)
            raise RuntimeError(f"context batch {Bc} neither matches nor broadcasts to the UNet batch {B}")
        if nt not in (1, B):
            raise RuntimeError(f"timestep count {nt} neither matches nor broadcasts to the UNet batch {B}")
        super().__init__(net, pw, B, H, W, nt, Bc, Sk, b_src)

    def _build(self, H, W, nt, Bc, Sk, b_src):
        self.b_src = self.B if b_src is None else b_src    # latent rows actually stored: B == 2*b_src folds latent.repeat(2,...)
        self.H, self.W, self.nt, self.Bc, self.Sk = H, W, nt, Bc, Sk
        a: UNetArch = self.net.arch
        self.arch = a
        t, lib = self.pw.t, self.lib
        B = self.B
        dev, f32 = self.device, torch.float32
        # static I/O staging (graph-stable addresses)
        self.x_in = torch.empty((self.b_src, a.in_channels, H, W), dtype=f32, device=dev)
        self.t_in = torch.zeros((nt,), dtype=torch.int64, device=dev)
        self.cond_in = torch.empty((Bc, Sk, a.dctx), dtype=f32, device=dev)
        self.out = torch.empty((B, a.out_channels, H, W), dtype=f32, device=dev)
        self.gn_ws = torch.zeros(int(lib.sdk_groupnorm_workspace_bytes(B, H * W)), dtype=torch.uint8, device=dev)
        self.gn_stats = torch.empty((B, 32, 2), dtype=f32, device=dev)
        self.kv: Dict[int, torch.Tensor] = {}
        # time embedding (unet.py:209-220) + all 22 ResBlock time projections (unet.py:182-183)
        te0 = torch.empty((self.nt, a.t_embed_dim), dtype=f32, device=dev)
        te1 = torch.empty((self.nt, a.temb), dtype=f32, device=dev)
        te2 = torch.empty((self.nt, a.temb), dtype=f32, device=dev)
        self.tb = torch.empty((self.nt, a.tb_total), dtype=f32, device=dev)
        self.keep += [te0, te1, te2]
        t_first = len(self.ops)
        self._emit(lib.sdk_time_sinusoid, self.t_in.data_ptr(), self.nt, a.t_embed_dim, te0.data_ptr())
        self._emit(lib.sdk_gemv, t["time_embedding.ffn.0.weight"].data_ptr(), F32_T, t["time_embedding.ffn.0.bias"].data_ptr(),
                   te0.data_ptr(), te1.data_ptr(), self.nt, a.temb, a.t_embed_dim, 0, 1)
        self._emit(lib.sdk_gemv, t["time_embedding.ffn.2.weight"].data_ptr(), F32_T, t["time_embedding.ffn.2.bias"].data_ptr(),
                   te1.data_ptr(), te2.data_ptr(), self.nt, a.temb, a.temb, 0, 0)
        self._emit(lib.sdk_gemv, t["tb.w"].data_ptr(), self.pw.wcode, t["tb.b"].data_ptr(),
                   te2.data_ptr(), self.tb.data_ptr(), self.nt, a.tb_total, a.temb, 1, 0)
        self.time_ops = self.ops[t_first:]       # timestep -> self.tb; a sampling loop precomputes them for its whole grid
        # context operand (context program)
        if self.act == F32_T:
            self.cond_act = self.cond_in.view(self.Bc * self.Sk, a.dctx)
        else:
            self.cond_act = torch.empty((self.Bc * self.Sk, a.dctx), dtype=_DT[self.act], device=dev)
            self._emit(lib.sdk_cast_upsample, self.cond_in.data_ptr(), self.cond_act.data_ptr(), self.act,
                       1, 1, self.Bc * self.Sk, a.dctx, 1, ctx=True)

        self.kv_all = None
        if self.pw.kv_total:
            self.kv_all = torch.empty((self.Bc * self.Sk, self.pw.kv_total), dtype=_DT[self.act], device=dev)
            self._conv([(self.cond_act, a.dctx)], t["kv2_all.w"], None, 1, 1, self.Bc * self.Sk, self.pw.kv_total,
                       out_code=self.act, out=self.kv_all, ctx=True)
        # conv_in (unet.py:256): NCHW latent -> NHWC, then 3x3 conv with Cin = 4 (FFMA kernel: K = 36)
        xin = self.pool.get(B * H * W, a.in_channels, F32_T)
        self._emit(lib.sdk_nchw_to_nhwc, self.x_in.data_ptr(), xin.data_ptr(), self.b_src, B, a.in_channels, H * W)
        x = self._conv_in(xin, a.in_channels, B, H, W, BLOCK_OUT[0])
        self.pool.put(xin)
        skips = [(x, BLOCK_OUT[0], H, W)]
        h, w = H, W
        xc = BLOCK_OUT[0]
        shared = {id(x)}                      # tensors referenced by the skip stack must not be recycled early
        tb_stride = a.tb_total if nt > 1 else 0

        def res(r, srcs, h, w):               # models/unet/unet.py:174-195
            return self._resblock(r.prefix, srcs, r.cout, r.eps, B, h, w, tbias=self.tb.data_ptr() + 4 * r.tb_offset,
                                  tb_stride=tb_stride)

        def release(tensor):
            if id(tensor) not in shared:
                self.pool.put(tensor)

        for st in a.down:
            for r, tr in st.blocks:
                y = res(r, [(x, xc)], h, w)
                release(x)
                x, xc = y, r.cout
                if tr is not None:
                    y = self._transformer(tr, x, B, h, w)
                    self.pool.put(x)
                    x = y
                skips.append((x, xc, h, w))
                shared.add(id(x))
            if st.resample is not None:
                wn, bn_ = t[f"{st.resample.prefix}.w"], t[f"{st.resample.prefix}.b"]
                if self.act == F32_T:
                    y, h, w = self._conv([(x, xc)], wn, bn_, B, h, w, xc, k=3, stride=2, want_stats=True)
                else:
                    # stride-2 3x3 (unet.py:236): the A boxes walk the bf16 input with element stride 2 (no im2col matrix) ...
                    ho, wo = (h - 1) // 2 + 1, (w - 1) // 2 + 1
                    y = None
                    if self.net.fold_gathers and B * ho * wo >= self.net.fold_min_rows_s2:
                        op, _ = self._operand(x, B, h, w, xc)
                        y, _, _ = self._conv([(op, xc)], wn, bn_, B, h, w, xc, k=3, stride=2, want_stats=True, fold_gather=True)
                        self.pool.put(op)
                    if y is None:
                        # ... or, for shapes the fold does not take: gather the 9 taps into bf16 rows, then a 1-tap tensor-core GEMM
                        col = self.pool.get(B * ho * wo, 9 * xc, BF16_T)
                        self._emit(lib.sdk_im2col_s2, x.data_ptr(), col.data_ptr(), B, h, w, xc)
                        y, _, _ = self._conv([(col, 9 * xc)], wn, bn_, B, ho, wo, xc, k=1, want_stats=True)
                        self.pool.put(col)
                    h, w = ho, wo
                x = y
                skips.append((x, xc, h, w))
                shared.add(id(x))
        # bottleneck (unet.py:383-391)
        y = res(a.mid[0], [(x, xc)], h, w)
        x = y                                   # previous x is still on the skip stack
        y = self._transformer(a.mid[1], x, B, h, w)
        self.pool.put(x)
        x = y
        y = res(a.mid[2], [(x, xc)], h, w)
        self.pool.put(x)
        x = y
        # decoder (unet.py:337-351)
        for st in a.up:
            prev_w = skips[-1][3]
            for r, tr in st.blocks:
                sk, skc, sh, sw = skips.pop()
                if (sh, sw) != (h, w):
                    raise RuntimeError(f"Sizes of tensors must match except in dimension 1 (skip {sh}x{sw} vs x {h}x{w}); "
                                       "latent H and W must be multiples of 8 (reference: unet.py:343)")
                y = res(r, [(x, xc), (sk, skc)], h, w)
                self.pool.put(x)
                shared.discard(id(sk))
                self.pool.put(sk)
                x, xc = y, r.cout
                if tr is not None:
                    y = self._transformer(tr, x, B, h, w)
                    self.pool.put(x)
                    x = y
            if st.resample is not None:
                up = not (skips and skips[-1][3] == prev_w)          # unet.py:346-349
                y, h, w = self._upsample_conv(st.resample.prefix, x, xc, B, h, w, up=up)
                self.pool.put(x)
                x = y
        # head (unet.py:398-401): GN + SiLU + conv 320 -> out_channels, written straight to NCHW
        ao, _ = self._gn([(x, xc)], B, h * w, t["out.gn.g"], t["out.gn.b"], a.eps, True)
        self.pool.put(x)
        self._conv([(ao, xc)], t["out.w"], t["out.b"], B, h, w, a.out_channels, k=3, out=self.out, out_nchw=True)
        self.pool.put(ao)

    def _finish(self):
        super()._finish()
        self.body_ops = [op for op in self.ops if all(op is not o for o in self.time_ops)]     # the step without the time embedding

    def _scratch(self):
        return super()._scratch() + [self.tb, self.cond_act, self.kv_all] + list(self.kv.values())

    def _transformer(self, tr: Transformer, x, B, H, W):
        """models/unet/unet.py:73-91 + 127-150 + attention.py:70-87, on [B*HW, C] tokens (NHWC == tokens)."""
        t, S, Cc = self.pw.t, H * W, tr.c
        M = B * S
        p = tr.prefix
        D = Cc // tr.heads
        es = 4 if self.act == F32_T else 2
        a, _ = self._gn([(x, Cc)], B, S, t[f"{p}.gn.g"], t[f"{p}.gn.b"], 1e-6, False)          # eps 1e-6: unet.py:66
        # bf16 program: the three LayerNorms (unet.py:137,141,147) are FOLDED into the projections that consume them -- the
        # producer's epilogue also writes a bf16 copy of the row and its (sum, sum of squares) partials, the consumer multiplies the
        # raw rows by gamma-scaled weights and normalises in ITS epilogue: no LayerNorm launch, no extra pass over the tensor.
        fold = self.act != F32_T and self.net.ln_fold and M >= self.net.ln_fold_min_rows

        def drop(tn):                                           # release a LayerNorm producer together with its side outputs
            for extra in ("_bf16", "_rowstats"):
                if getattr(tn, extra, None) is not None:
                    self.pool.put(getattr(tn, extra))
            self.pool.put(tn)

        fused = None if fold else self._linear_ln(a, t[f"{p}.in.w"], t[f"{p}.in.b"], None, t[f"{p}.ln1.g"], t[f"{p}.ln1.b"], M, Cc, Cc)
        if fused is not None:
            h, n1 = fused
        else:
            h, _, _ = self._conv([(a, Cc)], t[f"{p}.in.w"], t[f"{p}.in.b"], 1, 1, M, Cc, ln_out=fold)
        self.pool.put(a)
        # self-attention
        if fused is not None:
            qkv, _, _ = self._conv([(n1, Cc)], t[f"{p}.qkv.w"], None, 1, 1, M, 3 * Cc, out_code=self.act)
            self.pool.put(n1)
        elif fold:
            qkv, _, _ = self._conv([(h._bf16, Cc)], t[f"{p}.qkv.lnw"], t[f"{p}.qkv.lnb"], 1, 1, M, 3 * Cc, out_code=self.act,
                                   ln_in=(h._rowstats, t[f"{p}.qkv.lncs"]))
        else:
            n1 = self._ln(h, t[f"{p}.ln1.g"], t[f"{p}.ln1.b"], M, Cc)
            qkv, _, _ = self._conv([(n1, Cc)], t[f"{p}.qkv.w"], None, 1, 1, M, 3 * Cc, out_code=self.act)
            self.pool.put(n1)
        base = qkv.data_ptr()
        ao = self._attention(base, 3 * Cc, S * 3 * Cc, base + Cc * es, 3 * Cc, S * 3 * Cc, base + 2 * Cc * es, 3 * Cc, S * 3 * Cc,
                             B, tr.heads, S, S, D, Cc)
        self.pool.put(qkv)
        fused = None if fold else self._linear_ln(ao, t[f"{p}.o1.w"], t[f"{p}.o1.b"], h, t[f"{p}.ln2.g"], t[f"{p}.ln2.b"], M, Cc, Cc)
        if fused is not None:
            h2, n2 = fused
        else:
            h2, _, _ = self._conv([(ao, Cc)], t[f"{p}.o1.w"], t[f"{p}.o1.b"], 1, 1, M, Cc, residual=h, ln_out=fold)
        self.pool.put(ao)
        drop(h)
        # cross-attention: K/V of the context are loop-invariant -> context program
        if fused is not None:
            q2, _, _ = self._conv([(n2, Cc)], t[f"{p}.q2.w"], None, 1, 1, M, Cc, out_code=self.act)
            self.pool.put(n2)
        elif fold:
            q2, _, _ = self._conv([(h2._bf16, Cc)], t[f"{p}.q2.lnw"], t[f"{p}.q2.lnb"], 1, 1, M, Cc, out_code=self.act,
                                  ln_in=(h2._rowstats, t[f"{p}.q2.lncs"]))
        else:
            n2 = self._ln(h2, t[f"{p}.ln2.g"], t[f"{p}.ln2.b"], M, Cc)
            q2, _, _ = self._conv([(n2, Cc)], t[f"{p}.q2.w"], None, 1, 1, M, Cc, out_code=self.act)
            self.pool.put(n2)
        if self.kv_all is not None:                               # one GEMM for all layers (context program, emitted in _build)
            kv_row = self.pw.kv_total
            kvb = self.kv_all.data_ptr() + self.pw.kv_off[tr.index] * es
        else:
            kv_row = 2 * Cc
            kv = torch.empty((self.Bc * self.Sk, 2 * Cc), dtype=_DT[self.act], device=self.device)
            self.kv[tr.index] = kv
            self._conv([(self.cond_act, tr.dctx)], t[f"{p}.kv2.w"], None, 1, 1, self.Bc * self.Sk, 2 * Cc,
                       out_code=self.act, out=kv, ctx=True)
            kvb = kv.data_ptr()
        kv_batch = self.Sk * kv_row if self.Bc == B else 0
        ao2 = self._attention(q2.data_ptr(), Cc, S * Cc, kvb, kv_row, kv_batch, kvb + Cc * es, kv_row, kv_batch,
                              B, tr.heads, S, self.Sk, D, Cc)
        self.pool.put(q2)
        fused = None if fold else self._linear_ln(ao2, t[f"{p}.o2.w"], t[f"{p}.o2.b"], h2, t[f"{p}.ln3.g"], t[f"{p}.ln3.b"], M, Cc, Cc)
        if fused is not None:
            h3, n3 = fused
        else:
            h3, _, _ = self._conv([(ao2, Cc)], t[f"{p}.o2.w"], t[f"{p}.o2.b"], 1, 1, M, Cc, residual=h2, ln_out=fold)
        self.pool.put(ao2)
        drop(h2)
        # GEGLU feed-forward (activation_fn.py:17-20), GEGLU fused into the first GEMM's epilogue
        if fused is not None:
            g, _, _ = self._conv([(n3, Cc)], t[f"{p}.ff0.w"], t[f"{p}.ff0.b"], 1, 1, M, 8 * Cc, geglu=True, out_code=self.act)
            self.pool.put(n3)
        elif fold:
            g, _, _ = self._conv([(h3._bf16, Cc)], t[f"{p}.ff0.lnw"], t[f"{p}.ff0.lnb"], 1, 1, M, 8 * Cc, geglu=True, out_code=self.act,
                                 ln_in=(h3._rowstats, t[f"{p}.ff0.lncs"]))
        else:
            n3 = self._ln(h3, t[f"{p}.ln3.g"], t[f"{p}.ln3.b"], M, Cc)
            g, _, _ = self._conv([(n3, Cc)], t[f"{p}.ff0.w"], t[f"{p}.ff0.b"], 1, 1, M, 8 * Cc, geglu=True, out_code=self.act)
            self.pool.put(n3)
        h4, _, _ = self._conv([(g, 4 * Cc)], t[f"{p}.ff1.w"], t[f"{p}.ff1.b"], 1, 1, M, Cc, residual=h3, out_code=self.act)
        self.pool.put(g)
        drop(h3)
        # conv_output + long residual feeds the next GroupNorm: (B, H, W) form so that tiles can be attributed to samples
        out, _, _ = self._conv([(h4, Cc)], t[f"{p}.out.w"], t[f"{p}.out.b"], B, H, W, Cc, residual=x, want_stats=True)
        self.pool.put(h4)
        return out


# ======================================================================================
# module
# ======================================================================================
class UNet(ProgramModule):
    """Drop-in for the reference ``UNet`` (models/unet/unet.py:353-461)."""

    NORM_PARAMS = ("output.0",)             # the head's GroupNorm (unet.py:398) is the first module of a Sequential

    def __init__(self,
                 attention_head_dim: Union[int, List[int]] = 8,
                 cross_attention_dim: Union[int, List[int]] = 768,
                 in_channels: int = 4,
                 out_channels: int = 4,
                 block_out_channels: List[int] = [320, 640, 1280, 1280],
                 down_block_types: List[str] = ["CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "CrossAttnDownBlock2D", "DownBlock2D"],
                 t_embed_dim: int = 320,
                 use_lora=False,
                 num_attention_heads: Optional[Union[int, List[int]]] = None,
                 eps: float = 1e-05):
        super().__init__()
        if use_lora:
            # the reference raises AttributeError('proj_q') for use_lora=True (unet.py:114-123); at inference a
            # LoRA is a merged weight — merge it into the state dict before loading.
            raise NotImplementedError("use_lora=True is not supported (merge LoRA deltas into the weights instead)")
        if in_channels > 8:
            raise ValueError("in_channels > 8 is not supported by the conv_in kernel")
        self.arch = build_arch(attention_head_dim, cross_attention_dim, in_channels, out_channels, block_out_channels,
                               down_block_types, t_embed_dim, num_attention_heads, eps)
        self._init_params(param_spec(self.arch))
        self._lora: Dict[str, list] = {}       # adapter name -> [scale, {reference parameter name: lora.LoraModule}]

    # reference API no-ops (unet.py:404-428): inference path has no checkpointing; attention is always fused
    def gradient_checkpointing_enabled(self, enabled=False):
        return None

    def enable_flash_attn(self):
        return None

    # ---- forward ----------------------------------------------------------------------
    def _weights(self, device) -> PackedWeights:
        key = (str(device), self.precision, bool(getattr(self, "ln_fold", False)))      # the opt-in LayerNorm fold packs extra weights
        pw = self._packed.get(key)
        if pw is None:
            pw = PackedWeights(self, device, self.precision)
            self._merge(pw, {ref for _, mods in self._lora.values() for ref in mods})
            self._packed[key] = pw
        return pw

    # ---- LoRA adapters, merged into the packed weights in place ----------------------------------
    @property
    def lora_adapters(self) -> Dict[str, float]:
        """{adapter name: scale} of the loaded adapters."""
        return {n: s for n, (s, _) in self._lora.items()}

    def load_lora(self, src, scale: float = 1.0, name: str = "default") -> List[str]:
        """Merge a kohya or PEFT LoRA (``.safetensors`` path or state dict; LoCon convs included) into the packed weights as
        ``scale * alpha / rank * up @ down``, replacing an adapter of the same name.  The parameters keep the base weights
        (``state_dict()`` is unchanged); plans and captured graphs stay valid because the packed tensors are rewritten in place.
        Returns the keys that are not for the UNet (text-encoder LoRA), which are not applied.  Raises ValueError naming the key
        for a UNet key that does not fit, before anything changes."""
        if self.ln_fold:
            raise NotImplementedError("load_lora: the opt-in LayerNorm fold (SDB200_LN_FOLD=1) packs weights derived from the "
                                      "LayerNorm parameters, which a merge does not rebuild")
        mods, unapplied = lora.read_adapter(src, self.arch)
        old = self._lora.get(name, [0.0, {}])[1]
        self._lora[name] = [float(scale), mods]
        self._remerge(set(old) | set(mods))
        return unapplied

    def set_lora_scale(self, name: str, scale: float):
        """Change the scale of a loaded adapter and re-merge the targets it touches."""
        if name not in self._lora:
            raise KeyError(f"no LoRA adapter named {name!r} (loaded: {sorted(self._lora)})")
        self._lora[name][0] = float(scale)
        self._remerge(set(self._lora[name][1]))

    def unload_lora(self, name: Optional[str] = None):
        """Remove one adapter (or all, ``name=None``): the targets are rebuilt from the base weights, bit for bit."""
        names = list(self._lora) if name is None else [name]
        refs = set()
        for n in names:
            if n not in self._lora:
                raise KeyError(f"no LoRA adapter named {n!r} (loaded: {sorted(self._lora)})")
            refs |= set(self._lora.pop(n)[1])
        self._remerge(refs)

    def _remerge(self, refs):
        for pw in self._packed.values():
            self._merge(pw, refs)

    def _merge(self, pw: PackedWeights, refs):
        """Rebuild every packed tensor of the parameters ``refs`` from the fp32 master and the adapters with a non-zero scale, in
        adapter-name order (so the result does not depend on the order of the calls)."""
        if not refs:
            return
        lib = _lib.lib()
        params = dict(self.named_parameters())
        with torch.inference_mode(False), torch.no_grad(), torch.cuda.device(pw.device):
            # an fp32 pack on the parameters' device shares the storage of the weights it did not have to transform: give such a
            # parameter its own copy, so that merges into the pack never change the master weights
            shared = {p.untyped_storage().data_ptr(): p for p in params.values()}
            for t in pw.t.values():
                p = shared.pop(t.untyped_storage().data_ptr(), None)
                if p is not None:
                    p.data = p.data.clone()
            stream = torch.cuda.current_stream(pw.device).cuda_stream
            for ref in sorted(refs):
                mods = [(m[ref], s) for _, (s, m) in sorted(self._lora.items()) if ref in m and s != 0.0]
                for op in lora.merge_ops(self.arch, pw, ref, params[ref], mods):
                    dst, up, down = op["dst"], op["up"], op["down"]
                    r = 0 if up is None else up.shape[1]
                    n, k = op["base"].shape
                    # not a PDL launch (lora_merge.cu): kernels of this stream read packed weights before their own grid-dependency
                    # wait, so the next launch must start after the merge has completed
                    code = BF16_T if dst.dtype == torch.bfloat16 else F32_T
                    _lib.check(lib.sdk_lora_merge(op["base"].data_ptr(), k, 0 if up is None else up.data_ptr(),
                                                  0 if down is None else down.data_ptr(), r, dst.data_ptr() + op["offset"] * dst.element_size(),
                                                  code, op["layout"], op["dst_rows"], op["row_off"], op["row_step"], n, k, stream))
        pw.version += 1

    def forward(self, x: torch.Tensor, timestep: torch.LongTensor, cond: torch.Tensor) -> torch.Tensor:
        """reference: unet.py:431-443.  x (B,C,h,w) NCHW float; timestep int64 (1,) or (B,); cond (B|1,Sk,Dctx)."""
        if not isinstance(x, torch.Tensor) or not x.is_cuda:
            raise RuntimeError("UNet.forward: the B200 UNet only runs on CUDA tensors; there is no CPU fallback "
                               f"(got x on {getattr(x, 'device', type(x))})")
        a = self.arch
        if x.dim() != 4 or x.shape[1] != a.in_channels:
            raise RuntimeError(f"expected x of shape (B,{a.in_channels},h,w), got {tuple(x.shape)}")
        if cond.dim() == 2:
            cond = cond.unsqueeze(1)                                   # attention.py:76-77
        if cond.dim() != 3 or cond.shape[2] != a.dctx:
            raise RuntimeError(f"expected cond of shape (B,S,{a.dctx}), got {tuple(cond.shape)}")
        B, _, H, W = x.shape
        if not isinstance(timestep, torch.Tensor):
            timestep = torch.tensor([int(timestep)], dtype=torch.int64)
        timestep = timestep.reshape(-1)
        nt, Bc, Sk = timestep.numel(), cond.shape[0], cond.shape[1]
        if nt not in (1, B):
            raise RuntimeError(f"The size of tensor a ({B}) must match the size of tensor b ({nt}) at non-singleton dimension 0")
        if Bc not in (1, B):
            raise RuntimeError(f"cond batch {Bc} does not match / broadcast to latent batch {B}")
        dev = x.device
        pw = self._weights(dev)
        key = (str(dev), self.precision, B, H, W, nt, Bc, Sk)
        plan = self._plans.get(key)
        if plan is None:
            plan = _Runner(StepProgram(self, pw, B, H, W, nt, Bc, Sk), self.use_cuda_graph)
            self._plans[key] = plan
        return plan(x, timestep, cond).to(x.dtype)

    def export_engine(self, path: str, batch: int, height: int, width: int, *, context_len: int = 77,
                      context_batch: Optional[int] = None, per_sample_timesteps: bool = False, device=None):
        """Plan ``forward`` for a (batch, 4, height, width) latent and write its engine file (sdk_plan_save): a host without Python
        loads it with sdk_plan_load, fills the regions "x", "timestep", "context" and runs program 1 (context) then 0 (forward);
        the result is region "out".  See INTEGRATION.md 2b; the whole sampling loop exports through DenoiseLoop.export_engine."""
        dev = torch.device(device) if device is not None else next(self.parameters()).device
        if dev.type != "cuda":
            raise RuntimeError("export_engine needs the UNet on a CUDA device (the plan is built for that device's kernels)")
        bc = batch if context_batch is None else context_batch
        nt = batch if per_sample_timesteps else 1
        key = (str(dev), self.precision, batch, height, width, nt, bc, context_len)
        plan = self._plans.get(key)
        if plan is None:
            plan = _Runner(StepProgram(self, self._weights(dev), batch, height, width, nt, bc, context_len), self.use_cuda_graph)
            self._plans[key] = plan
        plan.prog.export_engine(path)

    @staticmethod
    def from_pretrained(pretrained_dir: str, device: str = 'cpu', sd_version: str = "1.5"):
        """reference: unet.py:445-461 — diffusers-layout directory (config.json + safetensors)."""
        from .weights import load_unet_state_dict
        with open(os.path.join(pretrained_dir, "config.json"), "r") as f:
            cfg = json.load(f)
        model = UNet(attention_head_dim=cfg["attention_head_dim"], cross_attention_dim=cfg["cross_attention_dim"],
                     in_channels=cfg["in_channels"], out_channels=cfg["out_channels"],
                     block_out_channels=cfg["block_out_channels"], down_block_types=cfg["down_block_types"],
                     eps=cfg["norm_eps"])
        sd = load_unet_state_dict(os.path.join(pretrained_dir, "diffusion_pytorch_model.safetensors"), model.arch, device)
        model.load_state_dict(sd, strict=True)
        return model


class _Runner(GraphRunner):
    """Runs a StepProgram; the context program runs only when ``cond`` is a new tensor or was written since the last call."""

    def __init__(self, prog: StepProgram, use_graph: bool):
        super().__init__(prog, use_graph)
        self._cond_ref = None
        self._cond_version = -1
        self._weights_version = prog.pw.version

    def __call__(self, x, timestep, cond):
        p = self.prog
        p.x_in.copy_(x, non_blocking=True)
        p.t_in.copy_(timestep.to(torch.int64), non_blocking=True)
        if not same_context(cond, self._cond_ref, self._cond_version) or p.pw.version != self._weights_version:
            p.cond_in.copy_(cond, non_blocking=True)
            p.launch(p.ctx_ops)                       # cross-attention K/V: once per context and weights, not per step
            self._cond_ref, self._cond_version = cond, tensor_version(cond)
            self._weights_version = p.pw.version
        self.run()
        return p.out.clone()
