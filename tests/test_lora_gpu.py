"""GPU suite: LoRA adapters merged into the packed UNet weights (sdk_lora_merge, UNet.load_lora / set_lora_scale / unload_lora)."""
import ctypes as C
import os

import pytest
import torch

import dpmpp_oracle as DO
from lora_synth import make_adapter, merged
from oracle import sampler_oracle as SO
from oracle import unet_oracle as UO
from stable_diffusion_pytorch_b200 import DDIMSampler, DenoiseLoop, DPMSolverSampler, UNet, _lib, lora

pytestmark = pytest.mark.gpu
GATE = {"fp32": 1e-4, "bf16": 1e-2}


def rel_l2(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return float((a - b).norm() / b.norm())


def bits(t):
    return t.view(torch.int32 if t.element_size() == 4 else torch.int16)


def packed_bits(net):
    return {(pk, k): bits(t).clone() for pk, pw in net._packed.items() for k, t in pw.t.items()}


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


def make_net(cfg, seed, dev):
    sd = UO.make_state_dict(seed, **cfg)
    net = UNet(attention_head_dim=cfg["attention_head_dim"], cross_attention_dim=cfg["cross_attention_dim"])
    net.load_state_dict(sd, strict=True)
    return net.to(dev).eval(), sd


@pytest.fixture(scope="module")
def net15(dev):
    return make_net(UO.SD15, 0, dev)


@pytest.fixture(scope="module")
def inputs(dev):
    lat, ctx = UO.synthetic_inputs(1, 16, 16)
    return lat.repeat(2, 1, 1, 1).to(dev), torch.tensor([481], device=dev), ctx.to(dev)


def oracle(sd64, x, t, ctx, cfg):
    """The oracle forward on the device with the float64-merged weights rounded once to fp32, without TF32."""
    flags = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = False
    try:
        sd = {k: v.to(x.device, torch.float32) for k, v in sd64.items()}
        with torch.no_grad():
            return UO.unet_forward(sd, x.float(), t, ctx.float(), **cfg)
    finally:
        torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = flags


def merge(lib, base, up, down, r, dst, dtype, layout, rows, off, step, n, k):
    return lib.sdk_lora_merge(base.data_ptr(), base.shape[1], up.data_ptr() if up is not None else 0,
                              down.data_ptr() if down is not None else 0, r, dst.data_ptr(), dtype, layout, rows, off, step, n, k,
                              C.c_void_p(torch.cuda.current_stream().cuda_stream))


# ---------------------------------------------------------------------------------------------------------------- kernel
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_kernel_r0_reproduces_every_packed_tensor(net15, dev, precision):
    net, _ = net15
    net.unload_lora()
    net.set_precision(precision)
    pw = net._weights(dev)
    lib, params, rebuilt = _lib.lib(), dict(net.named_parameters()), {}
    for ref in lora.targets(net.arch).values():
        for op in lora.merge_ops(net.arch, pw, ref, params[ref], []):
            key = next(k for k, t in pw.t.items() if t is op["dst"])
            out = rebuilt.setdefault(key, torch.full_like(op["dst"], float("nan")))
            n, k = op["base"].shape
            code = _lib.BF16_T if out.dtype == torch.bfloat16 else _lib.F32_T
            view = out.view(-1)[op["offset"]:]
            assert merge(lib, op["base"], None, None, 0, view, code, op["layout"], op["dst_rows"], op["row_off"], op["row_step"], n, k) == 0
    torch.cuda.synchronize()
    assert len(rebuilt) > 100
    for key, t in rebuilt.items():
        assert torch.equal(bits(t), bits(pw.t[key])), key


@pytest.mark.parametrize("dtype", ["fp32", "bf16"])
@pytest.mark.parametrize("layout", [0, 1])
@pytest.mark.parametrize("r", [0, 1, 4, 64, 192])
@pytest.mark.parametrize("n,k,step", [(1, 64, 1), (100, 320, 2), (320, 1280, 1), (63, 576, 2)])
def test_kernel_against_float64(dev, dtype, layout, r, n, k, step):
    g = torch.Generator().manual_seed(n * 7 + k + r)
    base = torch.randn((n, k + 3), generator=g)[:, :k]                 # ld_base > K
    base_c = base.contiguous()
    up = torch.randn((n, r), generator=g) / max(r, 1) ** 0.5
    down = torch.randn((r, k), generator=g)
    rows, off = step * n + 5, 3
    tdt = torch.float32 if dtype == "fp32" else torch.bfloat16
    dst = torch.full(((k // 64, rows, 64) if layout else (rows, k)), float("nan"), dtype=tdt, device=dev)
    b = torch.randn((n, k + 3), generator=g).to(dev)
    b[:, :k] = base_c.to(dev)
    lib = _lib.lib()
    up_d, down_d = up.to(dev), down.to(dev)
    rc = lib.sdk_lora_merge(b.data_ptr(), k + 3, up_d.data_ptr() if r else 0, down_d.data_ptr() if r else 0, r,
                            dst.data_ptr(), 0 if dtype == "fp32" else 1, layout, rows, off, step, n, k,
                            C.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, lib.sdk_last_error()
    got = dst.float().cpu()
    got = got.permute(1, 0, 2).reshape(rows, k) if layout else got
    idx = off + step * torch.arange(n)
    untouched = torch.ones(rows, dtype=torch.bool)
    untouched[idx] = False
    assert torch.isnan(got[untouched]).all()
    ref = base_c.double() + up.double() @ down.double()
    out = got[idx]
    if r == 0:
        assert torch.equal(out, base_c.to(tdt).float())
    elif dtype == "fp32":
        err = (out.double() - ref).abs().amax(1) / ref.abs().amax(1)
        assert float(err.max()) <= 1e-6
    else:
        want = ref.to(torch.bfloat16)
        mism = bits(out.to(torch.bfloat16)) != bits(want)
        ulp = (bits(out.to(torch.bfloat16)).int() - bits(want).int()).abs()
        # within 1 bf16 ulp, except where base + up @ down cancels below the fp32 rounding of its terms: there the bf16 ulp of
        # the result is smaller than what any fp32 accumulation can resolve
        terms = base_c.double().abs() + up.double().abs() @ down.double().abs()
        fp32_noise = (out.double() - ref).abs() <= 2.0 ** -8 * ref.abs() + 2.0 ** -22 * terms
        assert bool((ulp <= 1).logical_or(fp32_noise).all()) and float(mism.float().mean()) < 1e-3
        print(f"bf16 n{n} k{k} r{r}: {int(mism.sum())} mismatches of {mism.numel()}, {int((ulp > 1).sum())} beyond 1 ulp (cancellation)")


def test_kernel_bad_arguments(dev):
    lib = _lib.lib()
    t = torch.zeros((128, 128), device=dev)
    s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    p = t.data_ptr()
    ok = (p, 128, p, p, 4, p, 0, 0, 128, 0, 1, 64, 128, s)
    assert lib.sdk_lora_merge(*ok) == 0
    bad = {0: 0, 5: 0, 1: 64, 4: -1, 6: 2, 7: 2, 11: 0, 12: 0, 10: 0, 9: -1, 8: 63}
    for i, v in bad.items():
        a = list(ok)
        a[i] = v
        if i == 1:
            a[12] = 100                                              # ld_base < K
        assert lib.sdk_lora_merge(*a) == -1, i
    assert lib.sdk_lora_merge(p, 128, 0, p, 4, p, 0, 0, 128, 0, 1, 64, 128, s) == -1            # r > 0 without up
    assert lib.sdk_lora_merge(p, 128, p, p, 4, p, 0, 1, 128, 0, 1, 64, 100, s) == -1            # k-block layout, K % 64 != 0
    assert lib.sdk_lora_merge(p, 128, p, p, 4, p, 0, 0, 128, 2, 2, 64, 128, s) == -1            # last row 2 + 2*63 >= dst_rows
    torch.cuda.synchronize()


# ----------------------------------------------------------------------------------------------------------------- model
@pytest.mark.parametrize("arch", ["sd15", "sd21"])
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_model_matches_oracle_with_merged_weights(net15, dev, arch, precision):
    if arch == "sd15":
        net, sd = net15
        cfg = UO.SD15
    else:
        net, sd = make_net(UO.SD21, 2, dev)
        cfg = UO.SD21
    net.unload_lora()
    net.set_precision(precision)
    lat, ctx = UO.synthetic_inputs(1, 16, 16, dctx=cfg["cross_attention_dim"])
    x, t, ctx = lat.repeat(2, 1, 1, 1).to(dev), torch.tensor([481], device=dev), ctx.to(dev)
    # bf16: a milder adapter -- a merged weight three times the spread of the base one widens the bf16 rounding error of the
    # whole forward past the 1e-2 gate (1.02e-2 / 1.04e-2 on SD1.5 / SD2.1, against 7.3e-3 / 7.6e-3 without an adapter)
    amp = 3.0 if precision == "fp32" else 1.0
    adapter, truth = make_adapter(net.arch, "kohya", rank=4, alpha=2.0, seed=11, amp=amp, linear_proj=arch == "sd21")
    with torch.no_grad():
        y0 = net(x, t, ctx)
        assert net.load_lora(adapter, scale=0.8) == []
        y = net(x, t, ctx)
    ref = oracle(merged(sd, [(truth, 0.8)]), x, t, ctx, cfg)
    e, moved = rel_l2(y, ref), rel_l2(y0, ref)
    print(f"{arch} {precision}: rel-L2 {e:.3e}, adapter moves the output by {moved:.3e}; "
          f"without the adapter {rel_l2(y0, oracle(sd, x, t, ctx, cfg)):.3e}")
    assert e <= GATE[precision] and moved > (100 if precision == "fp32" else 10) * GATE[precision]
    net.unload_lora()


def test_in_place_exact_undo_and_order(net15, dev, inputs):
    net, sd = net15
    net.unload_lora()
    net.set_precision("bf16")
    x, t, ctx = inputs
    a1, tr1 = make_adapter(net.arch, "kohya", rank=4, alpha=3.0, seed=21)
    a2, tr2 = make_adapter(net.arch, "peft", rank=8, seed=22, select=("attn", "resnets.1", "upsamplers"))
    with torch.no_grad():
        for _ in range(3):                                                  # eager, capture, replay
            y0 = net(x, t, ctx)
        fresh = packed_bits(net)
        plans = {k: (p, p.graph, p.prog.ops, list(p.prog.tc_handles)) for k, p in net._plans.items()}
        ptrs = {(pk, k): v.data_ptr() for pk, pw in net._packed.items() for k, v in pw.t.items()}

        def same_objects():
            for k, (p, g, ops, hs) in plans.items():
                assert net._plans[k] is p and p.graph is g and g is not None and p.prog.ops is ops and p.prog.tc_handles == hs
            assert {(pk, k): v.data_ptr() for pk, pw in net._packed.items() for k, v in pw.t.items()} == ptrs

        net.load_lora(a1, scale=0.5, name="a")
        y_half = net(x, t, ctx)                                             # replayed from the graph captured before the load
        same_objects()
        assert not torch.equal(y_half, y0)
        half = packed_bits(net)
        net.set_lora_scale("a", 1.0)
        net.set_lora_scale("a", 0.5)
        assert all(torch.equal(half[k], v) for k, v in packed_bits(net).items())
        net.unload_lora("a")
        net.load_lora(a1, scale=1.0, name="a")
        net.set_lora_scale("a", 0.5)                                        # load(1) + set(0.5) == load(0.5)
        assert all(torch.equal(half[k], v) for k, v in packed_bits(net).items())
        net.set_lora_scale("a", 0.0)                                        # scale 0 == unloaded
        assert all(torch.equal(fresh[k], v) for k, v in packed_bits(net).items())
        # two adapters, both orders
        net.set_lora_scale("a", 0.7)
        net.load_lora(a2, scale=0.6, name="b")
        both = packed_bits(net)
        y_both = net(x, t, ctx)
        net.unload_lora()
        net.load_lora(a2, scale=0.6, name="b")
        net.load_lora(a1, scale=0.7, name="a")
        assert net.lora_adapters == {"a": 0.7, "b": 0.6}
        assert all(torch.equal(both[k], v) for k, v in packed_bits(net).items())
        assert torch.equal(net(x, t, ctx), y_both)
        same_objects()
        net.unload_lora()
        assert all(torch.equal(fresh[k], v) for k, v in packed_bits(net).items())
        assert torch.equal(net(x, t, ctx), y0)
        same_objects()
    ref = oracle(merged(sd, [(tr1, 0.7), (tr2, 0.6)]), x, t, ctx, UO.SD15)
    assert rel_l2(y_both, ref) <= GATE["bf16"]
    assert list(net.state_dict().keys()) == list(sd.keys())
    assert all(torch.equal(v.cpu(), sd[k]) for k, v in net.state_dict().items())          # the master weights never change


def test_scale_change_seen_without_host_sync(net15, dev, inputs):
    """A forward enqueued right after set_lora_scale reads the merged weights (the merge is not a PDL launch)."""
    net, _ = net15
    net.unload_lora()
    net.set_precision("bf16")
    x, t, ctx = inputs
    a, _ = make_adapter(net.arch, "kohya", rank=16, seed=31, select=("attn", "ff."))
    with torch.no_grad():
        net.load_lora(a, scale=0.3)
        want = [net(x, t, ctx) for _ in range(3)][-1]
        net.set_lora_scale("default", 1.0)
        net(x, t, ctx)
        for _ in range(3):
            net.set_lora_scale("default", 0.3)
            y = net(x, t, ctx)                                               # no synchronise between the merge and the forward
            net.set_lora_scale("default", 1.0)
        net.set_lora_scale("default", 0.3)
        y2 = net(x, t, ctx)
    assert torch.equal(y, want) and torch.equal(y2, want)
    net.unload_lora()


# ---------------------------------------------------------------------------------------------------------------- caches
def test_same_cond_object_follows_new_weights(net15, dev, inputs):
    net, sd = net15
    net.unload_lora()
    net.set_precision("fp32")
    x, t, ctx = inputs
    a, tr = make_adapter(net.arch, "peft", rank=8, seed=41, select=("attn2.to_k", "attn2.to_v"), amp=3.0)
    with torch.no_grad():
        y0 = net(x, t, ctx)
        net.load_lora(a)
        y = net(x, t, ctx)                                                   # the same cond tensor object
    ref = oracle(merged(sd, [(tr, 1.0)]), x, t, ctx, UO.SD15)
    assert rel_l2(y, ref) <= GATE["fp32"] and rel_l2(y0, ref) > 100 * GATE["fp32"]
    net.unload_lora()


@pytest.mark.parametrize("kind", ["ddim", "dpmpp"])
def test_denoise_loop_follows_new_weights(net15, dev, kind):
    net, sd = net15
    net.unload_lora()
    net.set_precision("fp32")
    lat, ctx = UO.synthetic_inputs(1, 16, 16, seed=5)
    smp = DDIMSampler() if kind == "ddim" else DPMSolverSampler()
    smp._set_inference_steps(5)
    a, tr = make_adapter(net.arch, "kohya", rank=8, alpha=4.0, seed=51, select=("time_emb_proj", "attn2.to_k", "attn2.to_v"), amp=2.0)
    ctx_d, lat_d = ctx.to(dev), lat.to(dev)
    with torch.no_grad():
        loop = DenoiseLoop(net, smp, 1, 16, 16, do_cfg=True, cfg_scale=7.5)
        before = loop.run(lat_d, ctx_d).cpu()
        loop.run(lat_d, ctx_d)                                              # graph captured, tables and K/V cached
        table = loop.tb_table.data_ptr()
        net.load_lora(a)
        got = loop.run(lat_d, ctx_d).cpu()
    assert loop.tb_table.data_ptr() == table
    sd64 = merged(sd, [(tr, 1.0)])
    x, hist = lat.numpy(), None
    a_hat = smp.alphas_hat.numpy() if hasattr(smp, "alphas_hat") else None
    tab = smp.coefficient_table().numpy() if kind == "dpmpp" else None
    for i, tv in enumerate(smp.timesteps.tolist()):
        pred = oracle(sd64, torch.from_numpy(x).to(dev).repeat(2, 1, 1, 1), torch.tensor([tv], device=dev), ctx_d, UO.SD15).cpu().numpy()
        eps = SO.cfg_combine(*SO.cfg_blend(pred), 7.5)
        if kind == "ddim":
            x = SO.ddim_reverse(x, tv, eps, smp.alphas.numpy(), a_hat, 1000, 5)
        else:
            x, hist = DO.dpmpp_reverse(x, tv, eps, hist, tab, hist_valid=i > 0)
    e = rel_l2(got, x)
    print(f"loop {kind}: rel-L2 {e:.3e} vs oracle, {rel_l2(before, x):.3e} before the load")
    assert e <= GATE["fp32"] and rel_l2(before, x) > 10 * GATE["fp32"]
    net.unload_lora()


# ----------------------------------------------------------------------------------------------------------- repack paths
def test_repacks_include_active_adapter(dev, inputs):
    net, sd = make_net(UO.SD15, 3, dev)
    net.set_precision("fp32")
    x, t, ctx = inputs
    a, tr = make_adapter(net.arch, "kohya", rank=4, seed=61, amp=1.5)
    ref = oracle(merged(sd, [(tr, 1.0)]), x, t, ctx, UO.SD15)
    with torch.no_grad():
        net(x, t, ctx)
        before = packed_bits(net)
        with pytest.raises(ValueError, match="lora_unet_conv_in"):
            net.load_lora(dict(a, **{"lora_unet_conv_in.lora_down.weight": torch.zeros(4, 4, 3, 3)}))
        assert net.lora_adapters == {}
        assert all(torch.equal(before[k], v) for k, v in packed_bits(net).items())        # a failed load changes nothing
        net.load_lora(a)
        y32 = net(x, t, ctx)
        assert rel_l2(y32, ref) <= GATE["fp32"]
        net.set_precision("bf16")                                           # a new pack, built with the adapter ...
        y16 = net(x, t, ctx)
        b16 = packed_bits(net)
        net.unload_lora()
        assert not torch.equal(net(x, t, ctx), y16)
        net.load_lora(a)                                                    # ... equals the adapter merged into an existing pack
        assert all(torch.equal(b16[k], v) for k, v in packed_bits(net).items()) and torch.equal(net(x, t, ctx), y16)
        net.set_precision("fp32")
        assert torch.equal(net(x, t, ctx), y32)
        net.load_state_dict(sd, strict=True)                               # invalidate() + repack of the same base weights
        assert not net._packed
        assert torch.equal(net(x, t, ctx), y32)
        net.to("cpu")                                                       # parameters on the host, pack on the device
        assert not net._packed
        y_host = net(x, t, ctx)
        assert torch.equal(y_host, y32)
        if torch.cuda.device_count() > 1:
            d1 = torch.device("cuda:1")
            net.to(d1)
            assert torch.equal(net(x.to(d1), t.to(d1), ctx.to(d1)).cpu(), y32.cpu())
    del net


# ---------------------------------------------------------------------------------------------------------------- engine
def test_engine_after_load_lora(net15, dev, tmp_path):
    import shutil
    if shutil.disk_usage(str(tmp_path)).free < 4 << 30:
        pytest.skip("needs 4 GiB of scratch space for the engine file")
    net, _ = net15
    net.unload_lora()
    net.set_precision("bf16")
    lib = _lib.lib()
    a, _ = make_adapter(net.arch, "kohya", rank=8, seed=71)
    lat, ctx = UO.synthetic_inputs(1, 16, 16, seed=7)
    smp = DDIMSampler()
    smp._set_inference_steps(10)
    steps = 4
    with torch.no_grad():
        loop = DenoiseLoop(net, smp, 1, 16, 16, do_cfg=True, cfg_scale=7.5)
        loop.run(lat.to(dev), ctx.to(dev), steps=steps)
        net.load_lora(a)
        ref = loop.run(lat.to(dev), ctx.to(dev), steps=steps).cpu()
        loop.reset(lat.to(dev), ctx.to(dev))
        path = str(tmp_path / "loop.engine")
        loop.export_engine(path)
    h = C.c_void_p()
    _lib.check(lib.sdk_plan_load(path.encode(), C.byref(h)))
    os.remove(path)
    try:
        s = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        xs, cs, zero = lat.contiguous(), ctx.contiguous(), torch.zeros(1, dtype=torch.int32)
        _lib.check(lib.sdk_plan_upload(h, b"x", xs.data_ptr(), xs.numel() * 4, s))
        _lib.check(lib.sdk_plan_upload(h, b"context", cs.data_ptr(), cs.numel() * 4, s))
        _lib.check(lib.sdk_plan_upload(h, b"counter", zero.data_ptr(), 4, s))
        _lib.check(lib.sdk_plan_launch(h, 1, s))
        for _ in range(steps):
            _lib.check(lib.sdk_plan_launch(h, 4, s))
        out = torch.empty_like(xs)
        _lib.check(lib.sdk_plan_download(h, b"x", out.data_ptr(), out.numel() * 4, s))
        torch.cuda.synchronize()
        assert torch.equal(out, ref)
    finally:
        _lib.check(lib.sdk_plan_destroy(h))
    net.unload_lora()
