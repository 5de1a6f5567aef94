"""GPU kernel-level parity: every C-ABI kernel against a plain PyTorch fp32 reference of the same op
(TF32 disabled) on seeded inputs.  Tolerances: fp32 kernels 2e-5 rel-L2; bf16-operand kernels are
compared on bf16-ROUNDED inputs with fp32 reference math, so only accumulation order and the final
output rounding differ (<= 4e-3 for bf16 outputs, <= 2e-5 for fp32 outputs).  The causal attention, row softmax, token embedding,
activation and VAE-attention GEMM tests compare with float64 references, element- or row-wise where a global norm could hide one bad
row."""
import ctypes as C
import math

import numpy as np
import pytest
import torch
import torch.nn.functional as Fn

from stable_diffusion_pytorch_b200 import _lib
from stable_diffusion_pytorch_b200._lib import BF16_T, F32_T, ConvParams, TcGemmDesc

pytestmark = pytest.mark.gpu
torch.backends.cuda.matmul.allow_tf32 = False
torch.backends.cudnn.allow_tf32 = False


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def rel_l2(a, b):
    a, b = a.double(), b.double()
    return float((a - b).norm() / b.norm().clamp_min(1e-30))


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def gen(shape, seed, dev, scale=1.0):
    g = torch.Generator().manual_seed(seed)
    return (torch.randn(shape, generator=g) * scale).to(dev)


# ------------------------------------------------------------------------------------------------
# reference for the implicit GEMM: NHWC in, torch conv2d in fp32
# ------------------------------------------------------------------------------------------------
def ref_conv(srcs, w_nkkc, bias, k, stride, up, tbias, residual, geglu):
    x = torch.cat([s.float() for s in srcs], dim=-1)                   # [B,H,W,C]
    x = x.permute(0, 3, 1, 2)
    if up:
        x = Fn.interpolate(x, scale_factor=2, mode="nearest")
    N = w_nkkc.shape[0]
    w = w_nkkc.float().view(N, k, k, -1).permute(0, 3, 1, 2)
    y = Fn.conv2d(x, w, bias, stride=stride, padding=k // 2)           # [B,N,Ho,Wo]
    if tbias is not None:
        y = y + tbias[:, :, None, None]
    y = y.permute(0, 2, 3, 1)
    if geglu:
        y = y[..., 0::2] * Fn.gelu(y[..., 1::2])
    if residual is not None:
        y = y + residual
    return y


CONV_CASES = [
    # B, H, W, (C0, C1), N, k, stride, up, tbias, residual, geglu
    (2, 16, 16, (320, 0), 320, 3, 1, False, "per", True, False),
    (2, 8, 8, (1280, 1280), 1280, 3, 1, False, "one", False, False),
    (1, 16, 16, (640, 320), 640, 1, 1, False, None, False, False),
    (2, 16, 16, (320, 0), 320, 3, 2, False, None, False, False),
    (2, 8, 8, (640, 0), 640, 3, 1, True, None, False, False),
    (1, 1, 300, (320, 0), 2560, 1, 1, False, None, False, True),
    (1, 8, 16, (4, 0), 320, 3, 1, False, None, False, False),
    (3, 5, 7, (32, 0), 20, 3, 1, False, None, True, False),
]


@pytest.mark.parametrize("case", CONV_CASES)
def test_conv_gemm_f32(dev, case):
    B, H, W, (C0, C1), N, k, stride, up, tbm, res, geglu = case
    lib = _lib.lib()
    s0 = gen((B, H, W, C0), 1, dev)
    s1 = gen((B, H, W, C1), 2, dev) if C1 else None
    Cin = C0 + C1
    w = gen((N, k * k * Cin), 3, dev, 1.0 / math.sqrt(k * k * Cin))
    bias = gen((N,), 4, dev, 0.1)
    upf = 2 if up else 1
    Ho = (H * upf + 2 * (k // 2) - k) // stride + 1
    Wo = (W * upf + 2 * (k // 2) - k) // stride + 1
    tb = None if tbm is None else gen((B if tbm == "per" else 1, N), 5, dev)
    Nout = N // 2 if geglu else N
    resid = gen((B, Ho, Wo, Nout), 6, dev) if res else None
    out = torch.empty((B, Ho, Wo, Nout), device=dev)
    p = ConvParams()
    p.src0, p.src1, p.C0, p.C1 = s0.data_ptr(), (s1.data_ptr() if C1 else 0), C0, C1
    p.weight, p.bias = w.data_ptr(), bias.data_ptr()
    p.tbias, p.tb_stride = (tb.data_ptr() if tb is not None else 0), (N if tbm == "per" else 0)
    p.residual, p.out = (resid.data_ptr() if res else 0), out.data_ptr()
    p.B, p.Hin, p.Win, p.Hout, p.Wout = B, H, W, Ho, Wo
    p.ksize, p.stride, p.upsample, p.N = k, stride, int(up), N
    p.in_dtype, p.out_dtype, p.out_nchw, p.geglu = F32_T, F32_T, 0, int(geglu)
    _lib.check(lib.sdk_conv_gemm_f32(C.byref(p), stream()))
    tbe = None if tb is None else tb.expand(B, N)
    want = ref_conv([s0] + ([s1] if C1 else []), w, bias, k, stride, up, tbe, resid, geglu)
    assert rel_l2(out, want) < 2e-5


TC_CASES = [
    # name, B, H, W, C, N, k, tbias, residual, geglu, out_dtype, out_nchw, block_n, splits
    ("lin_L0", 1, 1, 8192, 320, 320, 1, None, True, False, F32_T, 0, 0, 0),
    ("lin_ragged_kv", 1, 1, 154, 768, 640, 1, None, False, False, BF16_T, 0, 0, 0),
    ("conv_L0", 2, 64, 64, 320, 320, 3, "one", False, False, F32_T, 0, 0, 0),
    ("conv_L1", 2, 32, 32, 640, 640, 3, "per", True, False, F32_T, 0, 0, 0),
    ("conv_L3_splitk", 2, 8, 8, 1280, 1280, 3, None, True, False, F32_T, 0, 0, 0),
    ("conv_L2_bn256", 2, 16, 16, 1280, 1280, 3, None, False, False, F32_T, 0, 256, 1),
    ("conv_bn128", 2, 16, 16, 640, 1280, 3, None, False, False, BF16_T, 0, 128, 3),
    ("conv_bn64", 1, 16, 16, 320, 320, 3, None, False, False, F32_T, 0, 64, 2),
    ("geglu", 1, 1, 2048, 640, 5120, 1, None, False, True, BF16_T, 0, 0, 0),
    ("geglu_small", 1, 1, 128, 1280, 10240, 1, None, False, True, BF16_T, 0, 0, 0),
    ("head_nchw", 2, 32, 32, 320, 4, 3, None, False, False, F32_T, 1, 0, 0),
    ("odd_hw", 3, 24, 24, 320, 640, 3, None, True, False, F32_T, 0, 0, 0),
    ("tiny_hw", 2, 4, 4, 1280, 1280, 3, None, False, False, F32_T, 0, 0, 0),
    ("conv1x1_sp", 2, 16, 16, 2560, 1280, 1, None, False, False, F32_T, 0, 0, 0),
    ("lin_bf16_res", 1, 1, 4096, 640, 640, 1, "one", True, False, BF16_T, 0, 0, 0),
    ("conv_res_bn256", 2, 32, 32, 640, 1280, 3, "per", True, False, F32_T, 0, 256, 1),
    ("conv_res_bn32", 4, 8, 8, 320, 320, 3, "per", True, False, F32_T, 0, 32, 1),
    ("splitk_geglu", 1, 1, 256, 1280, 10240, 1, None, False, True, BF16_T, 0, 256, 4),
    # weight-stationary persistent walk (short K, several waves of tiles): GEGLU-in and q|k|v at level 0, a 1x1 conv at UNet batch 16
    ("ws_geglu_L0", 1, 1, 8192, 320, 2560, 1, None, False, True, BF16_T, 0, 160, 1),
    ("ws_qkv_L0", 1, 1, 8192, 320, 960, 1, None, False, False, BF16_T, 0, 160, 1),
    ("ws_lin_L1_bn64", 1, 1, 16384, 640, 1920, 1, None, False, False, BF16_T, 0, 64, 1),
    # text encoders (OpenCLIP-H, batch 2 x 77 tokens): q|k|v projection and fc2 + residual
    ("clip_qkv", 1, 1, 154, 1024, 3072, 1, None, False, False, BF16_T, 0, 0, 0),
    ("clip_fc2_res", 1, 1, 154, 4096, 1024, 1, None, True, False, F32_T, 0, 0, 0),
]


def kmajor(w):
    n, k = w.shape
    return w.view(n, k // 64, 64).permute(1, 0, 2).contiguous()


@pytest.mark.parametrize("wk", [1, 0], ids=["kmajor", "rowmajor"])
@pytest.mark.parametrize("case", TC_CASES, ids=[c[0] for c in TC_CASES])
def test_tc_gemm(dev, case, wk):
    name, B, H, W, Cc, N, k, tbm, res, geglu, odt, nchw, bn, splits = case
    lib = _lib.lib()
    a = gen((B, H, W, Cc), 11, dev).bfloat16()
    w = gen((N, k * k * Cc), 12, dev, 1.0 / math.sqrt(k * k * Cc)).bfloat16()
    bias = gen((N,), 13, dev, 0.1)
    tb = None if tbm is None else gen((B if tbm == "per" else 1, N), 14, dev)
    Nout = N // 2 if geglu else N
    resid = gen((B, H, W, Nout), 15, dev) if res else None
    odtype = torch.float32 if odt == F32_T else torch.bfloat16
    out = torch.full((B, Nout, H, W) if nchw else (B, H, W, Nout), float("nan"), device=dev, dtype=odtype)
    d = TcGemmDesc()
    wp = kmajor(w) if wk else w
    d.w_kmajor = wk
    d.a[0], d.w[0], d.C[0], d.ksize[0], d.nseg = a.data_ptr(), wp.data_ptr(), Cc, k, 1
    d.B, d.H, d.W, d.N = B, H, W, N
    d.bias = bias.data_ptr()
    d.tbias, d.tb_stride = (tb.data_ptr() if tb is not None else 0), (N if tbm == "per" else 0)
    d.residual, d.out = (resid.data_ptr() if res else 0), out.data_ptr()
    d.out_dtype, d.geglu, d.out_nchw, d.block_n, d.splits = odt, int(geglu), nchw, bn, splits
    d.weight_stationary = 2 if name.startswith("ws_") else 0
    h = C.c_void_p()
    _lib.check(lib.sdk_tc_gemm_create(C.byref(d), C.byref(h)))
    info = (C.c_int * 11)()
    _lib.check(lib.sdk_tc_gemm_info(h, info, 11))
    ws = torch.zeros(max(int(lib.sdk_tc_gemm_workspace_bytes(h)), 256), dtype=torch.uint8, device=dev)
    _lib.check(lib.sdk_tc_gemm_set_workspace(h, ws.data_ptr()))
    for _ in range(2):                                    # twice: split-K tickets must self-reset
        _lib.check(lib.sdk_tc_gemm_launch(h, stream()))
    torch.cuda.synchronize()
    lib.sdk_tc_gemm_destroy(h)
    tbe = None if tb is None else tb.expand(B, N)
    want = ref_conv([a], w, bias, k, 1, False, tbe, resid, geglu)
    if nchw:
        want = want.permute(0, 3, 1, 2)
    e = rel_l2(out.float(), want)
    print(f"{name}: block_n={info[0]} splits={info[1]} grid=({info[2]},{info[3]}) tile=({info[4]},{info[5]},{info[6]}) kb={info[7]} "
          f"kernel={('plain', 'persistent', 'persistent weight-stationary')[info[10]]} rel-L2={e:.2e}")
    assert not torch.isnan(out.float()).any()
    assert e < (4e-3 if odt == BF16_T else 2e-5)
    if name.startswith("ws_"):
        assert info[10] == 2, "expected the weight-stationary persistent form"


TWO_CTA_CASES = [
    # name, B, H, W, C, N, k, block_n, splits, tbias, residual, geglu, out_dtype
    ("conv_L0_cg2", 2, 64, 64, 320, 320, 3, 160, 1, "one", True, False, F32_T),
    ("conv_L1_cg2_splitk", 2, 32, 32, 640, 640, 3, 128, 2, None, False, False, F32_T),
    ("lin_geglu_cg2", 1, 1, 2048, 640, 5120, 1, 256, 1, None, False, True, BF16_T),
    ("lin_ragged_cg2", 1, 1, 200, 1280, 256, 1, 256, 1, None, True, False, F32_T),
]


@pytest.mark.parametrize("case", TWO_CTA_CASES, ids=[c[0] for c in TWO_CTA_CASES])
def test_tc_gemm_cta_pair(dev, case):
    """tcgen05 cta_group::2: CTA pairs run one 256-row MMA; same results as the 1-CTA path."""
    name, B, H, W, Cc, N, k, bn, splits, tbm, res, geglu, odt = case
    lib = _lib.lib()
    a = gen((B, H, W, Cc), 81, dev).bfloat16()
    w = gen((N, k * k * Cc), 82, dev, 1.0 / math.sqrt(k * k * Cc)).bfloat16()
    bias = gen((N,), 83, dev, 0.1)
    tb = None if tbm is None else gen((1, N), 84, dev)
    Nout = N // 2 if geglu else N
    resid = gen((B, H, W, Nout), 85, dev) if res else None
    outs = []
    for two in (2, 1):
        out = torch.full((B, H, W, Nout), float("nan"), device=dev, dtype=torch.float32 if odt == F32_T else torch.bfloat16)
        d = TcGemmDesc()
        wp = kmajor(w)
        d.w_kmajor, d.two_cta = 1, two
        d.a[0], d.w[0], d.C[0], d.ksize[0], d.nseg = a.data_ptr(), wp.data_ptr(), Cc, k, 1
        d.B, d.H, d.W, d.N = B, H, W, N
        d.bias = bias.data_ptr()
        d.tbias, d.tb_stride = (tb.data_ptr() if tb is not None else 0), 0
        d.residual, d.out = (resid.data_ptr() if res else 0), out.data_ptr()
        d.out_dtype, d.geglu, d.block_n, d.splits = odt, int(geglu), bn, splits
        h = C.c_void_p()
        _lib.check(lib.sdk_tc_gemm_create(C.byref(d), C.byref(h)))
        info = (C.c_int * 9)()
        _lib.check(lib.sdk_tc_gemm_info(h, info, 9))
        assert info[8] == two
        ws = torch.zeros(max(int(lib.sdk_tc_gemm_workspace_bytes(h)), 256), dtype=torch.uint8, device=dev)
        _lib.check(lib.sdk_tc_gemm_set_workspace(h, ws.data_ptr()))
        _lib.check(lib.sdk_tc_gemm_launch(h, stream()))
        torch.cuda.synchronize()
        lib.sdk_tc_gemm_destroy(h)
        outs.append(out)
    tbe = None if tb is None else tb.expand(B, N)
    want = ref_conv([a], w, bias, k, 1, False, tbe, resid, geglu)
    e = rel_l2(outs[0].float(), want)
    print(f"{name}: cta_group::2 rel-L2 {e:.2e}")
    assert not torch.isnan(outs[0].float()).any()
    assert e < (4e-3 if odt == BF16_T else 2e-5)
    assert torch.equal(outs[0], outs[1]), "2-CTA and 1-CTA paths accumulate in the same order"


def test_tc_gemm_two_segments(dev):
    """conv_2 (3x3 over a2) + fused 1x1 shortcut over the raw concat input (unet.py:188-193)."""
    lib = _lib.lib()
    B, H, W, C2, Cs, N = 2, 16, 16, 640, 1920, 640
    a2 = gen((B, H, W, C2), 21, dev).bfloat16()
    raw = gen((B, H, W, Cs), 22, dev).bfloat16()
    w2 = gen((N, 9 * C2), 23, dev, 1 / math.sqrt(9 * C2)).bfloat16()
    ws_ = gen((N, Cs), 24, dev, 1 / math.sqrt(Cs)).bfloat16()
    bias = gen((N,), 25, dev, 0.1)
    out = torch.empty((B, H, W, N), device=dev)
    d = TcGemmDesc()
    w2k, wsk = kmajor(w2), kmajor(ws_)
    d.w_kmajor = 1
    d.a[0], d.w[0], d.C[0], d.ksize[0] = a2.data_ptr(), w2k.data_ptr(), C2, 3
    d.a[1], d.w[1], d.C[1], d.ksize[1] = raw.data_ptr(), wsk.data_ptr(), Cs, 1
    d.nseg, d.B, d.H, d.W, d.N = 2, B, H, W, N
    d.bias, d.out, d.out_dtype = bias.data_ptr(), out.data_ptr(), F32_T
    h = C.c_void_p()
    _lib.check(lib.sdk_tc_gemm_create(C.byref(d), C.byref(h)))
    ws = torch.zeros(max(int(lib.sdk_tc_gemm_workspace_bytes(h)), 256), dtype=torch.uint8, device=dev)
    _lib.check(lib.sdk_tc_gemm_set_workspace(h, ws.data_ptr()))
    _lib.check(lib.sdk_tc_gemm_launch(h, stream()))
    torch.cuda.synchronize()
    lib.sdk_tc_gemm_destroy(h)
    want = ref_conv([a2], w2, bias, 3, 1, False, None, None, False) + ref_conv([raw], ws_, None, 1, 1, False, None, None, False)
    assert rel_l2(out, want) < 2e-5


def bits(t):
    """The raw bits of a bf16 / fp32 tensor: equality that tells -0 from 0."""
    return t.view(torch.int16 if t.element_size() == 2 else torch.int32)


# causal self-attention of the text encoders (clip.py:120-121): (B, heads, S, S, D, "causal").  S crosses the fp32 kernel's 32-key
# tiles and 64-row blocks and the tcgen05 kernel's 32-key streams, 64-key tiles and 128-row query tiles; every D at S = 77 and 129
CAUSAL_CASES = [(1, 4, 1, 1, 64), (2, 4, 20, 20, 40), (1, 16, 33, 33, 80), (2, 4, 64, 64, 160), (1, 16, 65, 65, 64),
                (2, 16, 77, 77, 40), (2, 16, 77, 77, 64), (1, 16, 77, 77, 80), (2, 16, 77, 77, 160), (1, 4, 128, 128, 80),
                (2, 4, 129, 129, 40), (2, 4, 129, 129, 64), (1, 4, 129, 129, 80), (2, 16, 129, 129, 160), (2, 16, 300, 300, 64)]
CAUSAL_PARAMS = [pytest.param(c + ("causal",), id=f"causal-B{c[0]}-h{c[1]}-S{c[2]}-D{c[4]}") for c in CAUSAL_CASES]
# prefix split points: the 32-key streams / tiles, the 64-key tiles and 64-row blocks, the 128-row query tiles
CAUSAL_SPLITS = (1, 31, 32, 33, 63, 64, 65, 127, 128, 129)


def causal_reference(qkv, B, Hh, S, D):
    """softmax(Q K^T / sqrt(D) + mask) V in float64, mask = -inf where key > query; qkv [B][S][q|k|v] -> [B][S][heads * D]."""
    t = qkv.double().view(B, S, 3, Hh, D).permute(2, 0, 3, 1, 4)
    s = (t[0] @ t[1].transpose(-1, -2)) * D ** -0.5
    s = s.masked_fill(torch.ones((S, S), dtype=torch.bool, device=qkv.device).triu(1), float("-inf"))
    return (torch.softmax(s, -1) @ t[2]).permute(0, 2, 1, 3).reshape(B, S, Hh * D)


def check_causal_attention(dev, B, Hh, S, D, kernel):
    """Causal self-attention of the fp32 kernel (sdk_attention_f32_ex, causal = 1) or the tcgen05 kernel (sdk_attention_tc_set_causal)
    on a q|k|v buffer with per-batch K / V: against float64 globally and row by row, and prefix-invariant bit for bit (rows < p do
    not see keys >= p).  The tcgen05 handle must give the non-causal result again once the mask is switched off."""
    lib = _lib.lib()
    Cc = Hh * D
    dt = torch.float32 if kernel == "f32" else torch.bfloat16
    qkv = gen((B, S, 3 * Cc), 131, dev).to(dt)
    buf = torch.empty_like(qkv)
    out = torch.full((B, S, Cc), float("nan"), device=dev, dtype=dt)
    st = (3 * Cc, S * 3 * Cc)
    args = (buf.data_ptr(), *st, buf.data_ptr() + Cc * qkv.element_size(), *st, buf.data_ptr() + 2 * Cc * qkv.element_size(), *st,
            out.data_ptr(), Cc, S * Cc, B, Hh, S, S, D, float(D ** -0.5))
    h = C.c_void_p()
    if kernel == "tc":
        _lib.check(lib.sdk_attention_tc_create(*args, C.byref(h)))
        _lib.check(lib.sdk_attention_tc_set_causal(h, 1))

    def run(x):
        buf.copy_(x)
        out.fill_(float("nan"))
        for _ in range(2):
            if kernel == "tc":
                _lib.check(lib.sdk_attention_tc_launch(h, stream()))
            else:
                _lib.check(lib.sdk_attention_f32_ex(*args, 1, stream()))
        torch.cuda.synchronize()
        return out.clone()

    try:
        y = run(qkv)
        assert not torch.isnan(y.float()).any()
        want = causal_reference(qkv, B, Hh, S, D)
        e = rel_l2(y, want)
        dy, w4 = (y.double() - want).view(B, S, Hh, D), want.view(B, S, Hh, D)
        rows = dy.norm(dim=-1) / w4.norm(dim=-1)                       # [B][S][heads]
        worst, at = float(rows.max()), int(rows.argmax())
        print(f"causal attention {kernel} B{B} heads{Hh} S{S} D{D}: rel-L2 {e:.2e}, worst (b, row, head) {worst:.2e} "
              f"at {(at // (S * Hh), at // Hh % S, at % Hh)}")
        assert e < (2e-5 if kernel == "f32" else 8e-3)
        assert worst < (1e-4 if kernel == "f32" else 2e-2)
        fresh = gen((B, S, 3 * Cc), 132, dev).to(dt)
        for p in CAUSAL_SPLITS:
            if p >= S:
                break
            alt = qkv.clone()
            alt[:, p:, Cc:] = fresh[:, p:, Cc:]                    # new keys and values from position p on
            y2 = run(alt)
            assert torch.equal(bits(y2[:, :p]), bits(y[:, :p])), f"rows < {p} read keys >= {p}"
            changed = (bits(y2[:, p]) != bits(y[:, p])).view(B, Hh, D).any(-1)
            assert bool(changed.all()), f"row {p} does not read key {p}"
        if kernel == "tc":
            _lib.check(lib.sdk_attention_tc_set_causal(h, 0))
            y0 = run(qkv)
            t = qkv.double().view(B, S, 3, Hh, D).permute(2, 0, 3, 1, 4)
            full = (torch.softmax((t[0] @ t[1].transpose(-1, -2)) * D ** -0.5, -1) @ t[2]).permute(0, 2, 1, 3).reshape(B, S, Cc)
            e0 = rel_l2(y0, full)
            print(f"  same handle, causal off: rel-L2 {e0:.2e} vs non-causal")
            assert e0 < 8e-3
    finally:
        if kernel == "tc":
            lib.sdk_attention_tc_destroy(h)


ATT_CASES = [(2, 8, 1024, 1024, 40), (2, 8, 256, 256, 160), (1, 8, 1024, 77, 80), (2, 5, 576, 576, 64),
             (2, 8, 64, 77, 160), (1, 8, 100, 77, 40), (2, 20, 144, 144, 64)]


@pytest.mark.parametrize("case", ATT_CASES + CAUSAL_PARAMS)
@pytest.mark.parametrize("mode", ["f32", "bf16"])
def test_attention(dev, case, mode):
    B, Hh, Sq, Sk, D = case[:5]
    if len(case) > 5:
        if mode == "bf16":
            pytest.skip("sdk_attention_bf16 has no causal path: bf16 causal attention runs on the tcgen05 kernel")
        check_causal_attention(dev, B, Hh, Sq, D, "f32")
        return
    lib = _lib.lib()
    Cc = Hh * D
    dt = torch.float32 if mode == "f32" else torch.bfloat16
    self_attn = Sq == Sk
    if self_attn:
        qkv = gen((B, Sq, 3 * Cc), 31, dev).to(dt)
        q, k, v = qkv[..., :Cc], qkv[..., Cc:2 * Cc], qkv[..., 2 * Cc:]
        strides = (3 * Cc, Sq * 3 * Cc, 3 * Cc, Sk * 3 * Cc, 3 * Cc, Sk * 3 * Cc)
    else:
        q = gen((B, Sq, Cc), 32, dev).to(dt)
        kv = gen((1, Sk, 2 * Cc), 33, dev).to(dt)                       # batch-broadcast context
        k, v = kv[..., :Cc], kv[..., Cc:]
        strides = (Cc, Sq * Cc, 2 * Cc, 0, 2 * Cc, 0)
    out = torch.empty((B, Sq, Cc), device=dev, dtype=dt)
    fn = lib.sdk_attention_f32 if mode == "f32" else lib.sdk_attention_bf16
    _lib.check(fn(q.data_ptr(), strides[0], strides[1], k.data_ptr(), strides[2], strides[3], v.data_ptr(), strides[4], strides[5],
                  out.data_ptr(), Cc, Sq * Cc, B, Hh, Sq, Sk, D, float(D ** -0.5), stream()))

    def heads(t):
        return t.float().expand(B, -1, -1).reshape(B, t.shape[1], Hh, D).permute(0, 2, 1, 3)

    qh, kh, vh = heads(q), heads(k), heads(v)
    w = torch.softmax((qh @ kh.transpose(-1, -2)) * D ** -0.5, dim=-1)
    want = (w @ vh).permute(0, 2, 1, 3).reshape(B, Sq, Cc)
    e = rel_l2(out.float(), want)
    print(f"attention {mode} {case}: rel-L2 {e:.2e}")
    assert e < (2e-5 if mode == "f32" else 6e-3)


ATT_TC_CASES = [(2, 8, 4096, 4096, 40), (1, 8, 1024, 77, 40), (2, 5, 2304, 2304, 64), (2, 8, 200, 333, 40), (1, 10, 576, 77, 64),
                (3, 8, 128, 128, 40), (2, 8, 256, 40, 40), (1, 5, 300, 9216, 64),
                # head dims spanning several swizzle atoms (SD-1.5 levels 1 / 2 / mid), self- and 77-key cross-attention
                (2, 8, 1024, 1024, 80), (2, 8, 1024, 77, 80), (2, 8, 256, 256, 160), (2, 8, 256, 77, 160), (2, 8, 64, 64, 160),
                (2, 8, 64, 77, 160), (16, 8, 1024, 1024, 80), (3, 8, 200, 333, 80), (1, 8, 100, 130, 160)]


@pytest.mark.parametrize("case", ATT_TC_CASES + CAUSAL_PARAMS)
def test_attention_tc(dev, case):
    """tcgen05 flash attention (head_dim 40 / 64 / 80 / 160) vs fp32 softmax(QK^T/sqrt(D))V on the bf16-rounded inputs."""
    B, Hh, Sq, Sk, D = case[:5]
    if len(case) > 5:
        check_causal_attention(dev, B, Hh, Sq, D, "tc")
        return
    lib = _lib.lib()
    Cc = Hh * D
    dt = torch.bfloat16
    if Sq == Sk:
        qkv = gen((B, Sq, 3 * Cc), 91, dev).to(dt)
        q, k, v = qkv[..., :Cc], qkv[..., Cc:2 * Cc], qkv[..., 2 * Cc:]
        strides = (3 * Cc, Sq * 3 * Cc, 3 * Cc, Sk * 3 * Cc, 3 * Cc, Sk * 3 * Cc)
    else:
        q = gen((B, Sq, Cc), 92, dev).to(dt)
        kv = gen((1, Sk, 2 * Cc), 93, dev).to(dt)                       # batch-broadcast context
        k, v = kv[..., :Cc], kv[..., Cc:]
        strides = (Cc, Sq * Cc, 2 * Cc, 0, 2 * Cc, 0)
    out = torch.full((B, Sq, Cc), float("nan"), device=dev, dtype=dt)
    h = C.c_void_p()
    _lib.check(lib.sdk_attention_tc_create(q.data_ptr(), strides[0], strides[1], k.data_ptr(), strides[2], strides[3],
                                           v.data_ptr(), strides[4], strides[5], out.data_ptr(), Cc, Sq * Cc, B, Hh, Sq, Sk, D,
                                           float(D ** -0.5), C.byref(h)))
    for _ in range(2):
        _lib.check(lib.sdk_attention_tc_launch(h, stream()))
    torch.cuda.synchronize()
    lib.sdk_attention_tc_destroy(h)

    def heads(t):
        return t.float().expand(B, -1, -1).reshape(B, t.shape[1], Hh, D).permute(0, 2, 1, 3)

    w = torch.softmax((heads(q) @ heads(k).transpose(-1, -2)) * D ** -0.5, dim=-1)
    want = (w @ heads(v)).permute(0, 2, 1, 3).reshape(B, Sq, Cc)
    e = rel_l2(out.float(), want)
    print(f"attention tcgen05 {case}: rel-L2 {e:.2e}")
    assert not torch.isnan(out.float()).any()
    assert e < 8e-3                                        # two different bf16 roundings (before / after the normalisation)


@pytest.mark.parametrize("shape", [(2, 256, 320, 0), (2, 64, 1280, 640), (1, 4096, 640, 320), (3, 16, 2560, 0), (2, 1024, 960, 0)])
@pytest.mark.parametrize("odt", [F32_T, BF16_T])
def test_groupnorm(dev, shape, odt):
    B, HW, C0, C1 = shape
    lib = _lib.lib()
    s0 = gen((B, HW, C0), 41, dev) * 2 + 0.5
    s1 = gen((B, HW, C1), 42, dev) if C1 else None
    Ct = C0 + C1
    gamma, beta = gen((Ct,), 43, dev) * 0.1 + 1, gen((Ct,), 44, dev) * 0.1
    stats = torch.empty((B, 32, 2), device=dev)
    ws = torch.zeros(int(lib.sdk_groupnorm_workspace_bytes(B, HW)), dtype=torch.uint8, device=dev)
    odtype = torch.float32 if odt == F32_T else torch.bfloat16
    out = torch.empty((B, HW, Ct), device=dev, dtype=odtype)
    raw = torch.empty((B, HW, Ct), device=dev, dtype=odtype)
    for _ in range(2):
        _lib.check(lib.sdk_groupnorm_stats(s0.data_ptr(), C0, s1.data_ptr() if C1 else 0, C1, B, HW, 1e-5, stats.data_ptr(), ws.data_ptr(), stream()))
        _lib.check(lib.sdk_groupnorm_apply(s0.data_ptr(), C0, s1.data_ptr() if C1 else 0, C1, B, HW, stats.data_ptr(), gamma.data_ptr(),
                                           beta.data_ptr(), 1, out.data_ptr(), raw.data_ptr(), odt, stream()))
    x = torch.cat([s0] + ([s1] if C1 else []), -1)
    want = Fn.silu(Fn.group_norm(x.permute(0, 2, 1), 32, gamma, beta, 1e-5)).permute(0, 2, 1)
    assert rel_l2(out.float(), want) < (2e-5 if odt == F32_T else 4e-3)
    assert rel_l2(raw.float(), x) < (1e-7 if odt == F32_T else 4e-3)
    # fused (single cooperative launch) variant used by the step program: same answer, run-to-run identical
    out2, raw2 = torch.empty_like(out), torch.empty_like(raw)
    for dst in (out2, out):
        _lib.check(lib.sdk_groupnorm_fused(s0.data_ptr(), C0, s1.data_ptr() if C1 else 0, C1, B, HW, 1e-5, gamma.data_ptr(), beta.data_ptr(), 1,
                                           dst.data_ptr(), raw2.data_ptr(), odt, ws.data_ptr(), stream()))
    assert rel_l2(out2.float(), want) < (2e-5 if odt == F32_T else 4e-3)
    assert torch.equal(out2, out) and torch.equal(raw2, raw)
    # cluster / DSMEM variant (the step program's default)
    out3, raw3 = torch.full_like(out, float("nan")), torch.full_like(raw, float("nan"))
    for dst in (out3, out2):
        _lib.check(lib.sdk_groupnorm_cluster(s0.data_ptr(), C0, s1.data_ptr() if C1 else 0, C1, B, HW, 1e-5, gamma.data_ptr(), beta.data_ptr(), 1,
                                             dst.data_ptr(), raw3.data_ptr(), odt, stream()))
    assert rel_l2(out3.float(), want) < (2e-5 if odt == F32_T else 4e-3)
    assert torch.equal(out3, out2) and rel_l2(raw3.float(), x) < (1e-7 if odt == F32_T else 4e-3)


@pytest.mark.parametrize("shape", [(2, 256, 320, 0), (2, 64, 1280, 640), (1, 4096, 640, 320), (3, 16, 2560, 0), (2, 1024, 960, 0)])
def test_groupnorm_from_channel_sums(dev, shape):
    """sdk_channel_stats + sdk_groupnorm_apply_cs (statistics from per-channel sums, the bf16 step program's route) vs nn.GroupNorm."""
    B, HW, C0, C1 = shape
    lib = _lib.lib()
    s0 = gen((B, HW, C0), 41, dev) * 2 + 0.5
    s1 = gen((B, HW, C1), 42, dev) if C1 else None
    Ct = C0 + C1
    gamma, beta = gen((Ct,), 43, dev) * 0.1 + 1, gen((Ct,), 44, dev) * 0.1
    cs0 = torch.zeros((B, C0, 2), device=dev, dtype=torch.float64)             # the kernel accumulates into a zeroed table
    cs1 = torch.zeros((B, max(C1, 1), 2), device=dev, dtype=torch.float64)
    _lib.check(lib.sdk_channel_stats(s0.data_ptr(), B, HW, C0, cs0.data_ptr(), stream()))
    if C1:
        _lib.check(lib.sdk_channel_stats(s1.data_ptr(), B, HW, C1, cs1.data_ptr(), stream()))
    assert rel_l2(cs0[..., 0], s0.double().sum(1)) < 1e-6 and rel_l2(cs0[..., 1], (s0.double() ** 2).sum(1)) < 1e-6
    x = torch.cat([s0] + ([s1] if C1 else []), -1)
    want = Fn.silu(Fn.group_norm(x.permute(0, 2, 1), 32, gamma, beta, 1e-5)).permute(0, 2, 1)
    for odt, dt, tol in ((F32_T, torch.float32, 2e-5), (BF16_T, torch.bfloat16, 4e-3)):
        out = torch.full((B, HW, Ct), float("nan"), device=dev, dtype=dt)
        raw = torch.full((B, HW, Ct), float("nan"), device=dev, dtype=dt)
        _lib.check(lib.sdk_groupnorm_apply_cs(s0.data_ptr(), C0, cs0.data_ptr(), s1.data_ptr() if C1 else 0, C1, cs1.data_ptr() if C1 else 0,
                                              B, HW, 1e-5, gamma.data_ptr(), beta.data_ptr(), 1, out.data_ptr(), raw.data_ptr(), odt, stream()))
        assert rel_l2(out.float(), want) < tol
        assert rel_l2(raw.float(), x) < (1e-7 if odt == F32_T else 4e-3)


@pytest.mark.parametrize("shape", [(2, 64, 64, 320), (3, 24, 40, 320), (1, 8, 8, 64), (2, 96, 96, 320), (1, 6, 10, 64), (2, 5, 7, 320)])
def test_conv_in(dev, shape):
    """conv_in kernels (3x3, Cin=4, fp32: four-pixel register-blocked for W % 4 == 0, per-pixel otherwise) and their statistics
    table vs F.conv2d."""
    B, H, W, N = shape
    lib = _lib.lib()
    x = gen((B, H, W, 4), 71, dev)
    w = gen((N, 3, 3, 4), 72, dev, 1.0 / 6.0)
    bias = gen((N,), 73, dev, 0.1)
    out = torch.full((B, H, W, N), float("nan"), device=dev)
    cs = torch.zeros((B, N, 2), device=dev, dtype=torch.float64)
    w_t = w.reshape(N, 36).t().contiguous()                      # [kh][kw][cin][N]
    _lib.check(lib.sdk_conv_in(x.data_ptr(), w_t.data_ptr(), bias.data_ptr(), out.data_ptr(), cs.data_ptr(), B, H, W, N, stream()))
    want = Fn.conv2d(x.permute(0, 3, 1, 2), w.permute(0, 3, 1, 2), bias, padding=1).permute(0, 2, 3, 1)
    assert rel_l2(out, want) < 2e-6
    flat = out.view(B, H * W, N).double()
    assert rel_l2(cs[..., 0], flat.sum(1)) < 1e-6 and rel_l2(cs[..., 1], (flat * flat).sum(1)) < 1e-6


TC_STATS_CASES = [
    # name, B, H, W, C, N, k, tbias, residual, block_n, splits
    ("L0_conv", 2, 64, 64, 320, 320, 3, "per", False, 0, 0),
    ("L1_conv_res", 2, 32, 32, 640, 640, 3, None, True, 0, 1),
    ("L1_1x1_res", 3, 32, 32, 640, 640, 1, None, True, 0, 1),
    ("L2_conv_bn256", 2, 16, 16, 1280, 1280, 3, "one", False, 256, 1),
    ("L3_two_samples_per_tile", 3, 8, 8, 1280, 1280, 3, "per", True, 0, 1),
    ("L3_splitk", 2, 8, 8, 1280, 1280, 3, "per", True, 0, 0),
    ("odd_hw", 3, 24, 24, 320, 640, 3, None, True, 0, 1),
    ("sd21_96", 1, 96, 96, 320, 320, 1, None, False, 0, 1),
]


@pytest.mark.parametrize("case", TC_STATS_CASES, ids=[c[0] for c in TC_STATS_CASES])
def test_tc_gemm_channel_stats(dev, case):
    """The GEMM epilogue's per-channel (sum, sum of squares) table == sums of the tensor it wrote."""
    name, B, H, W, Cc, N, k, tbm, res, bn, splits = case
    lib = _lib.lib()
    a = gen((B, H, W, Cc), 11, dev).bfloat16()
    w = gen((N, k * k * Cc), 12, dev, 1.0 / math.sqrt(k * k * Cc)).bfloat16()
    bias = gen((N,), 13, dev, 0.1) + 0.3
    tb = None if tbm is None else gen((B if tbm == "per" else 1, N), 14, dev)
    resid = gen((B, H, W, N), 15, dev) if res else None
    out = torch.full((B, H, W, N), float("nan"), device=dev)
    d = TcGemmDesc()
    wp = kmajor(w)
    d.w_kmajor = 1
    d.a[0], d.w[0], d.C[0], d.ksize[0], d.nseg = a.data_ptr(), wp.data_ptr(), Cc, k, 1
    d.B, d.H, d.W, d.N = B, H, W, N
    d.bias = bias.data_ptr()
    d.tbias, d.tb_stride = (tb.data_ptr() if tb is not None else 0), (N if tbm == "per" else 0)
    d.residual, d.out = (resid.data_ptr() if res else 0), out.data_ptr()
    d.out_dtype, d.geglu, d.out_nchw, d.block_n, d.splits = F32_T, 0, 0, bn, splits
    h = C.c_void_p()
    _lib.check(lib.sdk_tc_gemm_create(C.byref(d), C.byref(h)))
    info = (C.c_int * 8)()
    _lib.check(lib.sdk_tc_gemm_info(h, info, 8))
    ws = torch.zeros(max(int(lib.sdk_tc_gemm_workspace_bytes(h)), 256), dtype=torch.uint8, device=dev)
    _lib.check(lib.sdk_tc_gemm_set_workspace(h, ws.data_ptr()))
    cs = torch.full((2, B, N, 2), float("nan"), device=dev, dtype=torch.float64)
    for i in range(2):                                     # the launch accumulates into a table the caller zeroed
        _lib.check(lib.sdk_zero(cs[i].data_ptr(), cs[i].numel() * 8, stream()))
        _lib.check(lib.sdk_tc_gemm_set_stats(h, cs[i].data_ptr()))
        _lib.check(lib.sdk_tc_gemm_launch(h, stream()))
    torch.cuda.synchronize()
    lib.sdk_tc_gemm_destroy(h)
    tbe = None if tb is None else tb.expand(B, N)
    want = ref_conv([a], w, bias, k, 1, False, tbe, resid, False)
    e = rel_l2(out, want)
    flat = out.view(B, H * W, N).double()
    e_sum, e_sq = rel_l2(cs[0, ..., 0].double(), flat.sum(1)), rel_l2(cs[0, ..., 1].double(), (flat * flat).sum(1))
    print(f"{name}: block_n={info[0]} splits={info[1]} grid=({info[2]},{info[3]}) tile=({info[4]},{info[5]},{info[6]}) out {e:.2e} sum {e_sum:.2e} sumsq {e_sq:.2e}")
    assert e < 2e-5
    assert e_sum < 2e-6 and e_sq < 2e-6
    assert rel_l2(cs[0], cs[1]) < 1e-13                    # atomics in double: order-independent to the last bits


def upsample_parity_weights(w):
    """[N][3][3][C] conv weights -> [2][2][N][2][2][C]: the 3x3 taps of a conv over a nearest-2x upsampled image that read the same
    low-res pixel, pre-summed per output parity (what PackedWeights does for sdk_tc_gemm up2)."""
    rows = {0: ([0], [1, 2]), 1: ([0, 1], [2])}                 # parity -> 3x3 taps folded onto input offsets (p-1, p)
    n, _, _, c = w.shape
    out = torch.zeros((2, 2, n, 2, 2, c), dtype=torch.float32, device=w.device)
    for py in (0, 1):
        for px in (0, 1):
            for a in (0, 1):
                for b in (0, 1):
                    for kh in rows[py][a]:
                        for kw in rows[px][b]:
                            out[py, px, :, a, b] += w[:, kh, kw].float()
    return out


GATHER_CASES = [
    # name, B, H_in, W_in, C, N, mode, block_n
    ("up_L2", 2, 8, 8, 1280, 1280, "up2", 0),
    ("up_L1", 2, 16, 16, 1280, 1280, "up2", 0),
    ("up_L0", 2, 32, 32, 640, 640, "up2", 0),
    ("up_batch3_bn64", 3, 16, 16, 320, 320, "up2", 64),
    ("down_L0", 2, 64, 64, 320, 320, "s2", 0),
    ("down_L1", 2, 32, 32, 640, 640, "s2", 0),
    ("down_L2", 2, 16, 16, 1280, 1280, "s2", 0),
    ("down_odd", 1, 24, 40, 320, 320, "s2", 0),
]


@pytest.mark.parametrize("case", GATHER_CASES, ids=[c[0] for c in GATHER_CASES])
def test_tc_gemm_gather_folds(dev, case):
    """Upsample (unet.py:248-251) and stride-2 conv (unet.py:236-240) with the gather folded into the TMA coordinates: no upsampled
    tensor, no im2col matrix.  Reference: F.interpolate(nearest, 2x) + conv2d / conv2d(stride 2) in fp32 on the bf16-rounded input."""
    name, B, H, W, Cc, N, mode, bn = case
    lib = _lib.lib()
    a = gen((B, H, W, Cc), 61, dev).bfloat16()
    w = gen((N, 3, 3, Cc), 62, dev, 1.0 / math.sqrt(9 * Cc))
    bias = gen((N,), 63, dev, 0.1)
    d = TcGemmDesc()
    d.w_kmajor = 1
    if mode == "up2":
        wp = upsample_parity_weights(w).bfloat16()                           # [2][2][N][2][2][C]
        wk = torch.cat([kmajor(wp[py, px].reshape(N, 4 * Cc)) for py in (0, 1) for px in (0, 1)], 0).contiguous()
        Ho, Wo = 2 * H, 2 * W
        d.B, d.H, d.W, d.up2 = B, H, W, 1
        # reference on what the kernel multiplies: the pre-summed bf16 weights act on the low-res pixels
        x = a.float().permute(0, 3, 1, 2)
        want = torch.zeros((B, N, Ho, Wo), device=dev)
        xp = Fn.pad(x, (1, 1, 1, 1))
        for py in (0, 1):
            for px in (0, 1):
                k2 = wp[py, px].float().permute(0, 3, 1, 2)                    # [N][C][2][2]
                y = Fn.conv2d(xp[:, :, py:py + H + 1, px:px + W + 1], k2)
                want[:, :, py::2, px::2] = y
        want = (want + bias[None, :, None, None]).permute(0, 2, 3, 1)
        # and the un-folded definition (fp32 weights): differs only by the bf16 rounding of the summed weights
        ref = Fn.conv2d(Fn.interpolate(x, scale_factor=2, mode="nearest"), w.permute(0, 3, 1, 2), bias, padding=1).permute(0, 2, 3, 1)
    else:
        wk = kmajor(w.reshape(N, 9 * Cc).bfloat16())
        Ho, Wo = (H - 1) // 2 + 1, (W - 1) // 2 + 1
        d.B, d.H, d.W, d.a_stride, d.a_h, d.a_w = B, Ho, Wo, 2, H, W
        x = a.float().permute(0, 3, 1, 2)
        want = Fn.conv2d(x, w.bfloat16().float().permute(0, 3, 1, 2), bias, stride=2, padding=1).permute(0, 2, 3, 1)
        ref = want
    out = torch.full((B, Ho, Wo, N), float("nan"), device=dev)
    cs = torch.zeros((B, N, 2), device=dev, dtype=torch.float64)
    d.a[0], d.w[0], d.C[0], d.ksize[0], d.nseg = a.data_ptr(), wk.data_ptr(), Cc, 3, 1
    d.N, d.bias, d.out, d.out_dtype, d.block_n = N, bias.data_ptr(), out.data_ptr(), F32_T, bn
    h = C.c_void_p()
    _lib.check(lib.sdk_tc_gemm_create(C.byref(d), C.byref(h)))
    info = (C.c_int * 11)()
    _lib.check(lib.sdk_tc_gemm_info(h, info, 11))
    ws = torch.zeros(max(int(lib.sdk_tc_gemm_workspace_bytes(h)), 256), dtype=torch.uint8, device=dev)
    _lib.check(lib.sdk_tc_gemm_set_workspace(h, ws.data_ptr()))
    rc = lib.sdk_tc_gemm_set_stats(h, cs.data_ptr())
    _lib.check(lib.sdk_tc_gemm_launch(h, stream()))
    torch.cuda.synchronize()
    lib.sdk_tc_gemm_destroy(h)
    e, e_ref = rel_l2(out, want), rel_l2(out, ref)
    print(f"{name}: block_n={info[0]} splits={info[1]} grid=({info[2]},{info[3]}) tile=({info[4]},{info[5]},{info[6]}) persistent={info[10]} "
          f"rel-L2 {e:.2e} (vs un-folded fp32-weight definition {e_ref:.2e})")
    assert not torch.isnan(out).any()
    assert e < 2e-5 and e_ref < 4e-3
    if rc == 0:
        flat = out.view(B, Ho * Wo, N).double()
        assert rel_l2(cs[..., 0], flat.sum(1)) < 2e-6 and rel_l2(cs[..., 1], (flat * flat).sum(1)) < 2e-6


LN_FOLD_CASES = [
    # name, M, C, N_consumer, geglu, producer (block_n, splits), consumer (block_n, splits)
    ("L0_qkv", 8192, 320, 960, False, (0, 0), (0, 0)),
    ("L1_geglu", 2048, 640, 5120, True, (0, 0), (0, 0)),
    ("L2_q2_splitk_both", 512, 1280, 1280, False, (128, 4), (160, 4)),
    ("mid_ragged_rows", 200, 1280, 3840, False, (256, 5), (0, 0)),
    ("L1_splitk_many", 2048, 640, 640, False, (128, 2), (128, 2)),
]


@pytest.mark.parametrize("case", LN_FOLD_CASES, ids=[c[0] for c in LN_FOLD_CASES])
def test_tc_gemm_layernorm_fold(dev, case):
    """LayerNorm folded across two GEMMs (unet.py:137-149): the PRODUCER (out_proj + residual) also writes a bf16 copy of its fp32
    rows and their per-chunk (sum, sum of squares); the CONSUMER multiplies the raw bf16 rows by gamma-scaled weights and applies
    mean / rstd in its epilogue.  Reference: fp32 LayerNorm of the producer's fp32 output, rounded to bf16, times the bf16 weights."""
    name, M, Cc, N2, geglu, (bn1, sp1), (bn2, sp2) = case
    lib = _lib.lib()
    a = gen((1, 1, M, Cc), 31, dev).bfloat16()
    w1 = gen((Cc, Cc), 32, dev, 1.0 / math.sqrt(Cc)).bfloat16()
    b1 = gen((Cc,), 33, dev, 0.1)
    resid = gen((1, 1, M, Cc), 34, dev) * 2 + 0.5                      # non-zero row means
    gamma, beta = 1 + 0.2 * gen((Cc,), 35, dev), 0.1 * gen((Cc,), 36, dev)
    w2 = gen((N2, Cc), 37, dev, 1.0 / math.sqrt(Cc))
    b2 = gen((N2,), 38, dev, 0.1)
    out1 = torch.full((1, 1, M, Cc), float("nan"), device=dev)
    out1_bf = torch.full((1, 1, M, Cc), float("nan"), device=dev, dtype=torch.bfloat16)
    rowst = torch.full((M, Cc // 32, 2), float("nan"), device=dev)
    Nout = N2 // 2 if geglu else N2
    out2 = torch.full((1, 1, M, Nout), float("nan"), device=dev, dtype=torch.bfloat16)
    # host-side folding (what PackedWeights does)
    wg = (w2 * gamma[None, :]).bfloat16()
    colsum = wg.float().sum(1).contiguous()
    bias2 = (w2.double() @ beta.double() + b2.double()).float().contiguous()
    handles, infos = [], []
    for which in (0, 1):
        d = TcGemmDesc()
        d.w_kmajor = 1
        if which == 0:
            wp = kmajor(w1)
            d.a[0], d.w[0], d.C[0], d.ksize[0], d.nseg = a.data_ptr(), wp.data_ptr(), Cc, 1, 1
            d.B, d.H, d.W, d.N = 1, 1, M, Cc
            d.bias, d.residual, d.out, d.out_dtype = b1.data_ptr(), resid.data_ptr(), out1.data_ptr(), F32_T
            d.out2, d.row_stats = out1_bf.data_ptr(), rowst.data_ptr()
            d.block_n, d.splits = bn1, sp1
        else:
            wp2 = kmajor(wg)
            d.a[0], d.w[0], d.C[0], d.ksize[0], d.nseg = out1_bf.data_ptr(), wp2.data_ptr(), Cc, 1, 1
            d.B, d.H, d.W, d.N = 1, 1, M, N2
            d.bias, d.out, d.out_dtype, d.geglu = bias2.data_ptr(), out2.data_ptr(), BF16_T, int(geglu)
            d.ln_stats, d.ln_colsum, d.ln_parts, d.ln_eps = rowst.data_ptr(), colsum.data_ptr(), Cc // 32, 1e-5
            d.block_n, d.splits = bn2, sp2
        h = C.c_void_p()
        _lib.check(lib.sdk_tc_gemm_create(C.byref(d), C.byref(h)))
        info = (C.c_int * 11)()
        _lib.check(lib.sdk_tc_gemm_info(h, info, 11))
        handles.append((h, d, wp if which == 0 else wp2))
        infos.append(tuple(info))
    ws = torch.zeros(max(max(int(lib.sdk_tc_gemm_workspace_bytes(h)) for h, _, _ in handles), 256), dtype=torch.uint8, device=dev)
    for h, _, _ in handles:
        _lib.check(lib.sdk_tc_gemm_set_workspace(h, ws.data_ptr()))
    for _ in range(3):                                     # repeated: the split-K tile counters must re-arm themselves
        for h, _, _ in handles:
            _lib.check(lib.sdk_tc_gemm_launch(h, stream()))
    torch.cuda.synchronize()
    for h, _, _ in handles:
        lib.sdk_tc_gemm_destroy(h)
    for nm, info, sp in (("producer", infos[0], sp1), ("consumer", infos[1], sp2)):
        print(f"{name} {nm}: block_n={info[0]} splits={info[1]} grid=({info[2]},{info[3]}) fixup={info[9]} persistent={info[10]}")
        assert info[1] == 1 or info[9] == 1, "split-K with fused LayerNorm work must be reduced inside the kernel (or not split)"
    x = ref_conv([a], w1, b1, 1, 1, False, None, resid, False)            # [1,1,M,C] fp32
    assert rel_l2(out1, x) < 2e-5
    assert rel_l2(out1_bf.float(), out1.bfloat16().float()) == 0.0           # the copy is the rounded fp32 output
    xs = out1.view(M, Cc // 32, 32).double()
    assert rel_l2(rowst[..., 0].double(), xs.sum(-1)) < 1e-6 and rel_l2(rowst[..., 1].double(), (xs * xs).sum(-1)) < 1e-6
    ln = Fn.layer_norm(out1.view(M, Cc), (Cc,), gamma, beta, 1e-5)
    want = ln.bfloat16().float() @ w2.bfloat16().float().t() + b2
    if geglu:
        want = want[:, 0::2] * Fn.gelu(want[:, 1::2])
    e = rel_l2(out2.view(M, Nout).float(), want)
    print(f"{name}: folded LayerNorm -> GEMM rel-L2 {e:.2e} vs LN-then-bf16-GEMM")
    assert not torch.isnan(out2.float()).any()
    assert e < 8e-3                                        # two different bf16 roundings (before / after the normalisation)


# (name, M, K, N, residual, bias): the three projection -> LayerNorm pairs of a transformer block (unet.py:86,137-149) at the token
# counts of UNet batch 2 (64x64 ... 8x8), a ragged row count, and the 128-wide tile (OpenCLIP width 1024)
LINEAR_LN_CASES = [
    ("L0_o1", 8192, 320, 320, True, True),
    ("L0_in", 8192, 320, 320, False, True),
    ("L1_o2", 2048, 640, 640, True, True),
    ("L2_o1", 512, 1280, 1280, True, True),
    ("mid", 128, 1280, 1280, True, False),
    ("ragged", 200, 640, 640, True, True),
    ("bn128", 308, 1024, 1024, True, True),
]


@pytest.mark.parametrize("case", LINEAR_LN_CASES, ids=[c[0] for c in LINEAR_LN_CASES])
def test_linear_layernorm_fused(dev, case):
    """sdk_linear_ln (projection + bias + residual + LayerNorm in one cluster launch) against fp32 torch on the same bf16 operands:
    the fp32 output to accumulation-order accuracy, the normalised bf16 output to bf16 rounding."""
    name, M, K, N, has_res, has_bias = case
    lib = _lib.lib()
    a = gen((M, K), 71, dev).to(torch.bfloat16)
    w = (gen((N, K), 72, dev) / math.sqrt(K)).to(torch.bfloat16)
    bias = gen((N,), 73, dev) * 0.1 if has_bias else None
    res = (gen((M, N), 74, dev) * 2 + 0.5) if has_res else None
    gamma, beta = gen((N,), 75, dev) * 0.1 + 1, gen((N,), 76, dev) * 0.1
    out = torch.full((M, N), float("nan"), device=dev)
    ln = torch.full((M, N), float("nan"), device=dev, dtype=torch.bfloat16)
    wk = kmajor(w)
    d = _lib.LinearLnDesc()
    d.a, d.w, d.bias, d.residual = a.data_ptr(), wk.data_ptr(), (bias.data_ptr() if has_bias else 0), (res.data_ptr() if has_res else 0)
    d.out, d.ln_out, d.gamma, d.beta, d.eps, d.M, d.K, d.N = out.data_ptr(), ln.data_ptr(), gamma.data_ptr(), beta.data_ptr(), 1e-5, M, K, N
    h = C.c_void_p()
    _lib.check(lib.sdk_linear_ln_create(C.byref(d), C.byref(h)))
    info = (C.c_int * 4)()
    _lib.check(lib.sdk_linear_ln_info(h, info, 4))
    assert info[0] * info[1] == N and info[2] == (M + 127) // 128 * info[1]
    for _ in range(2):                                            # relaunchable: no state is left behind
        _lib.check(lib.sdk_linear_ln_launch(h, stream()))
    torch.cuda.synchronize()
    _lib.check(lib.sdk_linear_ln_destroy(h))
    ref = a.float() @ w.float().t()
    if has_bias:
        ref = ref + bias
    if has_res:
        ref = ref + res
    e_out = rel_l2(out, ref)
    ref_ln = Fn.layer_norm(out, (N,), gamma, beta, 1e-5)          # statistics of the kernel's OWN fp32 rows
    e_ln = rel_l2(ln.float(), ref_ln)
    print(f"{name}: out rel-L2 {e_out:.2e}, LayerNorm rel-L2 {e_ln:.2e} (cluster of {info[1]}, {info[2]} CTAs)")
    assert not torch.isnan(out).any() and not torch.isnan(ln.float()).any()
    assert e_out < 2e-6
    assert e_ln < 3e-3                                            # bf16 rounding of the normalised row
    # the bf16 result must equal the stand-alone LayerNorm kernel's on the same rows up to rare rounding flips
    ln2 = torch.empty_like(ln)
    _lib.check(lib.sdk_layernorm(out.data_ptr(), gamma.data_ptr(), beta.data_ptr(), 1e-5, ln2.data_ptr(), BF16_T, M, N, stream()))
    torch.cuda.synchronize()
    flips = (ln.float() != ln2.float()).float().mean().item()
    assert flips < 2e-3, flips


def test_linear_layernorm_unsupported_width(dev):
    """Row widths that do not split into <= 8 tiles of 160 / 128 columns are refused (the caller keeps GEMM + LayerNorm)."""
    lib = _lib.lib()
    x = torch.zeros((128, 768), device=dev, dtype=torch.bfloat16)
    o = torch.zeros((128, 768), device=dev)
    d = _lib.LinearLnDesc()
    d.a, d.w, d.out, d.ln_out, d.gamma, d.beta, d.eps, d.M, d.K, d.N = x.data_ptr(), x.data_ptr(), o.data_ptr(), x.data_ptr(), o.data_ptr(), o.data_ptr(), 1e-5, 128, 768, 1600
    h = C.c_void_p()
    assert lib.sdk_linear_ln_create(C.byref(d), C.byref(h)) == -3


@pytest.mark.parametrize("C_", [320, 640, 1280, 768, 256, 1024])
def test_layernorm(dev, C_):
    lib = _lib.lib()
    x = gen((1000, C_), 51, dev) * 3 + 1
    g, b = gen((C_,), 52, dev) * 0.1 + 1, gen((C_,), 53, dev) * 0.1
    for odt, dt, tol in ((F32_T, torch.float32, 2e-6), (BF16_T, torch.bfloat16, 4e-3)):
        out = torch.empty((1000, C_), device=dev, dtype=dt)
        _lib.check(lib.sdk_layernorm(x.data_ptr(), g.data_ptr(), b.data_ptr(), 1e-5, out.data_ptr(), odt, 1000, C_, stream()))
        assert rel_l2(out.float(), Fn.layer_norm(x, (C_,), g, b, 1e-5)) < tol


def test_time_embedding_and_gemv(dev):
    lib = _lib.lib()
    t = torch.tensor([981, 1, 500], device=dev)
    out = torch.empty((3, 320), device=dev)
    _lib.check(lib.sdk_time_sinusoid(t.data_ptr(), 3, 320, out.data_ptr(), stream()))
    freqs = torch.exp(-math.log(10000) * torch.arange(0, 160, dtype=torch.float32, device=dev) / 160)
    xx = t[:, None].float() * freqs[None]
    want = torch.cat([torch.cos(xx), torch.sin(xx)], -1)
    assert (out - want).abs().max() < 2e-4            # |arg| up to ~1e3: a few ulp of the argument
    W = gen((2000, 1280), 61, dev, 0.03)
    bias = gen((2000,), 62, dev)
    x = gen((3, 1280), 63, dev)
    for wdt, code, tol in ((torch.float32, F32_T, 2e-6), (torch.bfloat16, BF16_T, 2e-6)):
        Wd = W.to(wdt)
        y = torch.empty((3, 2000), device=dev)
        _lib.check(lib.sdk_gemv(Wd.data_ptr(), code, bias.data_ptr(), x.data_ptr(), y.data_ptr(), 3, 2000, 1280, 1, 1, stream()))
        want = Fn.silu(Fn.linear(Fn.silu(x), Wd.float(), bias))
        assert rel_l2(y, want) < 1e-5


def test_cast_upsample_im2col_nchw(dev):
    lib = _lib.lib()
    x = gen((2, 6, 10, 64), 71, dev)
    up = torch.empty((2, 12, 20, 64), device=dev, dtype=torch.bfloat16)
    _lib.check(lib.sdk_cast_upsample(x.data_ptr(), up.data_ptr(), BF16_T, 2, 6, 10, 64, 2, stream()))
    want = Fn.interpolate(x.permute(0, 3, 1, 2), scale_factor=2, mode="nearest").permute(0, 2, 3, 1).bfloat16()
    assert torch.equal(up, want)
    col = torch.empty((2 * 3 * 5, 9 * 64), device=dev, dtype=torch.bfloat16)
    _lib.check(lib.sdk_im2col_s2(x.data_ptr(), col.data_ptr(), 2, 6, 10, 64, stream()))
    unf = Fn.unfold(x.permute(0, 3, 1, 2), 3, padding=1, stride=2)           # [B, C*9, L], index c*9 + tap
    want = unf.view(2, 64, 9, 15).permute(0, 3, 2, 1).reshape(30, 576).bfloat16()
    assert torch.equal(col, want)
    lat = gen((1, 4, 8, 8), 72, dev)
    nhwc = torch.empty((2, 64, 4), device=dev)
    _lib.check(lib.sdk_nchw_to_nhwc(lat.data_ptr(), nhwc.data_ptr(), 1, 2, 4, 64, stream()))
    assert torch.equal(nhwc, lat.repeat(2, 1, 1, 1).permute(0, 2, 3, 1).reshape(2, 64, 4))


# ------------------------------------------------------------------------------------------------
# row softmax of the VAE attention (vae.py:90), the text encoders' token embedding and activations (clip.py:114,130)
# ------------------------------------------------------------------------------------------------
FLT_MIN = 2.0 ** -126                                   # smallest normal fp32: below it the kernel's exp2 / product are subnormal


@pytest.mark.parametrize("rows,cols", [(300, 4), (300, 64), (300, 1020), (300, 1024), (200, 4096), (64, 9216), (24, 16384)])
def test_softmax_rows(dev, rows, cols):
    """sdk_softmax_rows vs float64 softmax of the same fp32 scores: logits spanning +-80 in the exp2 domain, a row with one dominant
    entry, a row of equal values.  Every element within 1e-5 relative (absolute FLT_MIN where fp32 underflows), every row sums to 1;
    the bf16 output is the fp32 output rounded."""
    lib = _lib.lib()
    scale = 512 ** -0.5
    sl2 = float(np.float32(np.float32(scale) * np.float32(1.4426950408889634)))      # the kernel's fp32 scale * log2(e)
    g = torch.Generator().manual_seed(141)
    x = (torch.rand((rows, cols), generator=g, dtype=torch.float64) * 160 - 80) / sl2
    x[1] = torch.randn(cols, generator=g, dtype=torch.float64) / sl2
    x[1, cols // 3] += 80 / sl2                                                     # one entry 2^80 above the rest
    x[2] = 3.0                                                                      # all equal: 1 / cols
    x = x.float().to(dev)
    want = torch.softmax(x.double() * (sl2 * math.log(2.0)), dim=-1)
    y = torch.full((rows, cols), float("nan"), device=dev)
    yb = torch.full((rows, cols), float("nan"), device=dev, dtype=torch.bfloat16)
    for out, odt in ((y, F32_T), (yb, BF16_T)):
        _lib.check(lib.sdk_softmax_rows(x.data_ptr(), out.data_ptr(), odt, rows, cols, scale, stream()))
    torch.cuda.synchronize()
    err = (y.double() - want).abs()
    worst = float(((err - FLT_MIN).clamp_min(0) / want).max())
    row_sum = float((y.double().sum(-1) - 1).abs().max())
    print(f"softmax rows={rows} cols={cols}: worst element rel err {worst:.2e}, worst |row sum - 1| {row_sum:.2e}")
    assert not torch.isnan(y).any()
    assert bool((err <= 1e-5 * want + FLT_MIN).all())
    assert row_sum <= 1e-5
    assert float((y[2].double() - 1.0 / cols).abs().max()) <= 1e-5 / cols
    assert torch.equal(bits(yb), bits(y.bfloat16()))


def test_softmax_rows_contract(dev):
    lib = _lib.lib()
    buf = torch.zeros(64, device=dev)
    p = buf.data_ptr()
    assert lib.sdk_softmax_rows(p, p, F32_T, 1, 6, 1.0, stream()) == -1               # cols % 4 != 0
    assert lib.sdk_softmax_rows(p, p, F32_T, 1, 16388, 1.0, stream()) == -1           # wider than 16384
    assert lib.sdk_softmax_rows(p, p, 2, 1, 16, 1.0, stream()) == -1                  # no such output type
    assert lib.sdk_softmax_rows(p, p, F32_T, 0, 16, 1.0, stream()) == 0               # no rows: nothing to do


EMBED_CASES = [(77, 1, 256), (77, 2, 768), (77, 2, 1024), (20, 1, 1024), (20, 2, 256), (20, 2, 768),
               (77, 32, 1024)]                                  # 2464 rows x 256 float4: more than one pass of the capped grid


@pytest.mark.parametrize("S,B,C_", EMBED_CASES)
def test_embed_tokens(dev, S, B, C_):
    """sdk_embed_tokens == tok[ids] + pos[r % S] exactly; ids outside [0, vocab) are clamped to the table."""
    lib = _lib.lib()
    vocab, rows = 1000, B * S
    tok = gen((vocab, C_), 151, dev)
    pos = gen((77, C_), 152, dev)                               # the encoders' max_len positions; S of them are read
    g = torch.Generator().manual_seed(153)
    ids = torch.randint(0, vocab, (B, S), generator=g, dtype=torch.int64)
    ids.view(-1)[:5] = torch.tensor([0, vocab - 1, -1, vocab, 2 ** 40])
    ids.view(-1)[-3:] = torch.tensor([-(2 ** 40), vocab - 1, 0])
    ids = ids.to(dev)
    out = torch.full((B, S, C_), float("nan"), device=dev)
    _lib.check(lib.sdk_embed_tokens(ids.data_ptr(), tok.data_ptr(), pos.data_ptr(), out.data_ptr(), rows, S, C_, vocab, stream()))
    torch.cuda.synchronize()
    want = tok[ids.clamp(0, vocab - 1)] + pos[:S][None]
    assert torch.equal(bits(out), bits(want))
    if B == 32:
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        assert rows * C_ // 4 > sms * 8 * 256, "the grid-stride loop must run more than once"


@pytest.mark.parametrize("n", [4, 1020, 1 << 21])              # 2^21 / 4 float4 > 8 CTAs x 256 threads per SM: grid-stride
@pytest.mark.parametrize("kind", [1, 2], ids=["gelu", "quickgelu"])
def test_activation(dev, kind, n):
    """sdk_activation (1: exact-erf GELU, 2: QuickGELU x * sigmoid(1.702 x)) vs float64 on a dense grid over [-30, 30] plus 0, -0,
    +-1e4: absolute error <= 1e-6 * max(1, |x|), never NaN; the bf16 output is the fp32 output rounded."""
    lib = _lib.lib()
    x = torch.cat([torch.tensor([0.0, -0.0, 1e4, -1e4], dtype=torch.float64), torch.linspace(-30, 30, n - 4, dtype=torch.float64)])
    x = x.float().to(dev)
    xd = x.double()
    want = 0.5 * xd * torch.special.erfc(-xd / math.sqrt(2.0)) if kind == 1 else xd * torch.sigmoid(1.702 * xd)
    y = torch.full((n,), float("nan"), device=dev)
    yb = torch.full((n,), float("nan"), device=dev, dtype=torch.bfloat16)
    for out, odt in ((y, F32_T), (yb, BF16_T)):
        _lib.check(lib.sdk_activation(x.data_ptr(), out.data_ptr(), odt, n, kind, stream()))
    torch.cuda.synchronize()
    err = (y.double() - want).abs() / xd.abs().clamp_min(1.0)
    print(f"activation kind {kind} n={n}: worst abs err / max(1, |x|) {float(err.max()):.2e}")
    assert not torch.isnan(y).any()
    assert float(err.max()) <= 1e-6
    assert float(y[3]) == 0.0                                   # x = -1e4: -0 or 0 (QuickGELU's exp overflows to inf)
    assert torch.equal(bits(yb), bits(y.bfloat16()))


# ------------------------------------------------------------------------------------------------
# the VAE mid-block attention's three GEMMs (vae.py:85-91), each on its own bf16-rounded operands
# ------------------------------------------------------------------------------------------------
def vae_attention_operands(dev, S, Cc=512):
    """Operands of one sample's attention GEMMs.  The token, q and k buffers hold two samples, and sample 1 is read through its
    slice pointer as in the per-sample loop.  P is a row softmax, so the bias of P V is a visible part of the output."""
    g = torch.Generator().manual_seed(161)

    def r(*shape, s=1.0):
        return (torch.randn(shape, generator=g) * s).to(dev)

    ops = dict(tokens=r(2 * S, Cc), wv=r(Cc, Cc, s=Cc ** -0.5), q=r(2 * S, Cc), k=r(2 * S, Cc),
               p=torch.softmax(r(S, S, s=2.0), -1), vT=r(Cc, S), bv=r(Cc, s=0.1))
    return ops


def vae_attention_stage(ops, stage, S, Cc=512):
    """(A [M][K], B operand [N][K] row-major, bias, M, N, K, output rows offset) of one stage: V^T = W_v tokens^T (N = S),
    scores = q k^T (fp32 [S][S]), out = P V + b_v (K = S, written to rows S..2S of the batch's output)."""
    if stage == "vT":
        return ops["wv"], ops["tokens"][S:], None, Cc, S, Cc, 0
    if stage == "scores":
        return ops["q"][S:], ops["k"][S:], None, S, S, Cc, 0
    return ops["p"], ops["vT"], ops["bv"], S, Cc, S, S


VAE_ATT_STAGES = ([pytest.param("vT", (0, 0), id="vT-auto"), pytest.param("scores", (0, 0), id="scores-auto")] +
                  [pytest.param("pv", t, id=f"pv-bn{t[0]}-sp{t[1]}") for t in ((0, 0), (64, 1), (128, 2), (256, 4))])


@pytest.mark.parametrize("S", [64, 128, 576, 4096, 9216])
@pytest.mark.parametrize("stage,tiling", VAE_ATT_STAGES)
def test_tc_gemm_vae_attention(dev, stage, tiling, S):
    """The tensor-core GEMMs of the VAE attention with an ACTIVATION as the row-major B operand (w_kmajor = 0, w_const = 0, as
    _emit_tc_conv sets them for w_rowmajor) vs float64 on the bf16 operands; P V also with forced (block_n, split-K) tilings."""
    lib = _lib.lib()
    ops = {k: v.bfloat16() if k != "bv" else v for k, v in vae_attention_operands(dev, S).items()}
    a, w, bias, M, N, K, row0 = vae_attention_stage(ops, stage, S)
    odt = F32_T if stage == "scores" else BF16_T
    out_all = torch.full((row0 + M, N), float("nan"), device=dev, dtype=torch.float32 if odt == F32_T else torch.bfloat16)
    out = out_all[row0:]
    d = TcGemmDesc()
    d.w_kmajor, d.w_const = 0, 0
    d.a[0], d.w[0], d.C[0], d.ksize[0], d.nseg = a.data_ptr(), w.data_ptr(), K, 1, 1
    d.B, d.H, d.W, d.N = 1, 1, M, N
    d.bias = bias.data_ptr() if bias is not None else 0
    d.out, d.out_dtype = out.data_ptr(), odt
    d.block_n, d.splits = tiling
    h = C.c_void_p()
    _lib.check(lib.sdk_tc_gemm_create(C.byref(d), C.byref(h)))
    info = (C.c_int * 11)()
    _lib.check(lib.sdk_tc_gemm_info(h, info, 11))
    ws = torch.zeros(max(int(lib.sdk_tc_gemm_workspace_bytes(h)), 256), dtype=torch.uint8, device=dev)
    _lib.check(lib.sdk_tc_gemm_set_workspace(h, ws.data_ptr()))
    for _ in range(2):                                    # twice: split-K tickets must re-arm
        _lib.check(lib.sdk_tc_gemm_launch(h, stream()))
    torch.cuda.synchronize()
    lib.sdk_tc_gemm_destroy(h)
    want = a.double() @ w.double().t()
    if bias is not None:
        want = want + bias.double()
    e = rel_l2(out, want)
    print(f"VAE attention {stage} S={S} M={M} N={N} K={K}: block_n={info[0]} splits={info[1]} grid=({info[2]},{info[3]}) "
          f"kernel={('plain', 'persistent', 'persistent weight-stationary')[info[10]]} rel-L2 {e:.2e}")
    assert not torch.isnan(out.float()).any()
    assert e < (2e-5 if odt == F32_T else 4e-3)
    if row0:
        assert torch.isnan(out_all[:row0].float()).all(), "wrote outside the sample's rows"
    if tiling != (0, 0):                                  # the forced split count, as the library rounds it to whole k-blocks
        kb = K // 64
        per = -(-kb // min(tiling[1], kb))
        assert info[0] == tiling[0] and info[1] == -(-kb // per)


@pytest.mark.parametrize("S", [64, 576, 4096])
@pytest.mark.parametrize("stage", ["vT", "scores", "pv"])
def test_conv_gemm_f32_vae_attention(dev, stage, S):
    """The same three products in the fp32 mode (sdk_conv_gemm_f32, the B operand a plain [N][K] matrix) vs float64."""
    lib = _lib.lib()
    ops = vae_attention_operands(dev, S)
    a, w, bias, M, N, K, row0 = vae_attention_stage(ops, stage, S)
    out_all = torch.full((row0 + M, N), float("nan"), device=dev)
    out = out_all[row0:]
    p = ConvParams()
    p.src0, p.src1, p.C0, p.C1 = a.data_ptr(), 0, K, 0
    p.weight, p.bias = w.data_ptr(), (bias.data_ptr() if bias is not None else 0)
    p.tbias, p.tb_stride, p.residual, p.out = 0, 0, 0, out.data_ptr()
    p.B, p.Hin, p.Win, p.Hout, p.Wout = 1, 1, M, 1, M
    p.ksize, p.stride, p.upsample, p.N = 1, 1, 0, N
    p.in_dtype, p.out_dtype, p.out_nchw, p.geglu = F32_T, F32_T, 0, 0
    _lib.check(lib.sdk_conv_gemm_f32(C.byref(p), stream()))
    torch.cuda.synchronize()
    want = a.double() @ w.double().t()
    if bias is not None:
        want = want + bias.double()
    e = rel_l2(out, want)
    print(f"VAE attention fp32 {stage} S={S}: rel-L2 {e:.2e}")
    assert e < 2e-5
    if row0:
        assert torch.isnan(out_all[:row0]).all(), "wrote outside the sample's rows"
