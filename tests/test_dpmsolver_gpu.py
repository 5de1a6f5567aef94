"""GPU parity of the DPM-Solver++(2M) sampler: the fused CFG + multistep update kernels (sdk_dpmpp_step,
sdk_dpmpp_inpaint_step) bit for bit against the numpy oracle, the graph-replayed loop against the step-by-step API and an
oracle loop, and the exported engine run by the plain-C host."""
import ctypes as C
import os
import shutil
import subprocess

import numpy as np
import pytest
import torch

import dpmpp_oracle as DO
from oracle import sampler_oracle as SO
from oracle import unet_oracle as UO
from stable_diffusion_pytorch_b200 import DPMSolverSampler, UNet, _lib
from stable_diffusion_pytorch_b200.pipeline import DenoiseLoop, denoise, img2img, inpaint

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def rel_l2(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b) / np.linalg.norm(b))


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available()
    return torch.device("cuda:0")


@pytest.fixture(scope="module")
def net15(dev):
    net = UNet()
    net.load_state_dict(UO.make_state_dict(0, **UO.SD15), strict=True)
    return net.to(dev).eval()


def sampler(n=20, ptype="epsilon", strength=None):
    s = DPMSolverSampler(prediction_type=ptype)
    s._set_inference_steps(n)
    if strength is not None:
        s.set_strength(strength)
    return s


@pytest.mark.parametrize("ptype", ["epsilon", "v_prediction"])
@pytest.mark.parametrize("cfg", [True, False])
@pytest.mark.parametrize("t_on_device", [True, False])
def test_step_bit_exact(dev, ptype, cfg, t_on_device):
    """A first-order step, then second-order steps reading the history it left, against the oracle."""
    s = sampler(20, ptype)
    tab = s.coefficient_table().numpy()
    g = torch.Generator().manual_seed(11)
    x = torch.randn((2, 4, 24, 40), generator=g)
    hist = None
    for i in (0, 1, 2, 10, 18, 19):
        t = int(s.timesteps[i])
        mo = torch.randn((4 if cfg else 2, 4, 24, 40), generator=g)
        tt = torch.tensor([t], device=dev) if t_on_device else t
        got = s.reverse_process(x.to(dev), tt, mo.to(dev), cfg_scale=7.5 if cfg else None)
        e = SO.cfg_combine(*SO.cfg_blend(mo.numpy()), 7.5) if cfg else mo.numpy()
        want, hist = DO.dpmpp_reverse(x.numpy(), t, e, hist, tab, ptype, hist_valid=i > 0)
        assert np.array_equal(got.cpu().numpy(), want), (i, t)
        assert np.array_equal(s._hist.cpu().numpy(), hist)
        x = got.cpu()


def test_step_scalar_tail_and_misaligned(dev):
    s = sampler(20)
    tab = s.coefficient_table().numpy()
    g = torch.Generator().manual_seed(12)
    for n, off in ((7, 0), (1027, 0), (1024, 1), (4099, 3)):
        buf = torch.randn(n + off, generator=g)
        x = buf.to(dev)[off:]                                 # off != 0: 4-byte aligned only, the scalar path
        s.reset()
        hist = None
        for i in (0, 1, 2):
            t = int(s.timesteps[i])
            mo = torch.randn(2 * n + off, generator=g).to(dev)[off:].view(2, n)
            got = s.reverse_process(x.view(1, n), torch.tensor([t], device=dev), mo, cfg_scale=3.0)
            e = SO.cfg_combine(mo[0:1].cpu().numpy(), mo[1:2].cpu().numpy(), 3.0)
            want, hist = DO.dpmpp_reverse(x.view(1, n).cpu().numpy(), t, e, hist, tab, hist_valid=i > 0)
            assert np.array_equal(got.cpu().numpy(), want), (n, off, i)
            x = got.view(n)


def test_nan_history_unread_when_invalid(dev):
    """hist_valid = 0 on an order-2 row: the history (NaN here) is not read, the step is the first-order one."""
    s = sampler(20)
    tab = s.coefficient_table().numpy()
    t = int(s.timesteps[5])
    assert tab[t, 7] == 1
    g = torch.Generator().manual_seed(13)
    x, e = torch.randn((1, 4, 16, 16), generator=g), torch.randn((1, 4, 16, 16), generator=g)
    s.reset()
    s._hist = torch.full((1, 4, 16, 16), float("nan"), device=dev)
    got = s.reverse_process(x.to(dev), t, e.to(dev)).cpu().numpy()
    want, _ = DO.dpmpp_reverse(x.numpy(), t, e.numpy(), None, tab, hist_valid=False)
    assert np.isfinite(got).all() and np.array_equal(got, want)
    # and the C entry directly, scalar path included
    lib = _lib.lib()
    for n in (1024, 1023):
        xd, ed = x.reshape(-1)[:n].to(dev), e.reshape(-1)[:n].to(dev)
        hd = torch.full((n,), float("nan"), device=dev)
        out = torch.empty_like(xd)
        tabd = torch.from_numpy(tab).to(dev)
        _lib.check(lib.sdk_dpmpp_step(xd.data_ptr(), ed.data_ptr(), 0, 0.0, hd.data_ptr(), 0, out.data_ptr(), n, tabd.data_ptr(),
                                      s.noise_step, 0, t, 0, _lib.current_stream(dev)))
        assert np.array_equal(out.cpu().numpy(), want.reshape(-1)[:n]) and torch.isfinite(hd).all()


def test_out_of_range_timestep_poisons(dev):
    s = sampler(10)
    x = torch.ones(1, 4, 8, 8, device=dev)
    assert torch.isnan(s.reverse_process(x, torch.tensor([1000], device=dev), x)).all()
    assert torch.isnan(s.reverse_process(x, -1, x)).all()


@pytest.mark.parametrize("ptype", ["epsilon", "v_prediction"])
def test_inpaint_step_bit_exact(dev, ptype):
    s = sampler(20, ptype, strength=0.8)
    tab = s.coefficient_table().numpy()
    a_hat = s.alphas_hat.numpy()
    g = torch.Generator().manual_seed(14)
    lat = torch.randn((2, 4, 16, 24), generator=g)
    enc = torch.randn((1, 4, 16, 24), generator=g)
    mask = torch.rand((16, 24), generator=g) > 0.5
    hist = None
    for i in range(4):
        t = int(s.timesteps[i])
        pred2 = torch.randn((4, 4, 16, 24), generator=g)
        got = s.inpaint_step(lat.to(dev), torch.tensor([t], device=dev), pred2.to(dev), enc.to(dev), mask.to(dev), cfg_scale=7.5)
        want, hist = DO.dpmpp_inpaint_step(lat.numpy(), t, pred2.numpy(), enc.numpy(), mask.numpy(), 7.5, a_hat, hist, tab, ptype,
                                           hist_valid=i > 0)
        assert np.array_equal(got.cpu().numpy(), want), i
        lat = got.cpu()
    got = s.inpaint_step(lat.to(dev), int(s.timesteps[4]), pred2[:2].to(dev), enc.expand(2, -1, -1, -1).to(dev), mask.to(dev))
    want, _ = DO.dpmpp_inpaint_step(lat.numpy(), int(s.timesteps[4]), pred2[:2].numpy(), enc.numpy(), mask.numpy(), None, a_hat, hist,
                                    tab, ptype)
    assert np.array_equal(got.cpu().numpy(), want)


@pytest.fixture(scope="module")
def oracle_loop(golden_dir):
    """fp32 CPU loop: the oracle UNet + dpmpp_reverse, SD1.5-arch seed 0, 16x16, 10 steps, CFG 7.5."""
    g = np.load(os.path.join(golden_dir, "unet_sd15_golden.npz"))
    sd = UO.make_state_dict(0, **UO.SD15)
    s = sampler(10)
    tab = s.coefficient_table().numpy()
    x, ctx = torch.from_numpy(g["lat16"]), torch.from_numpy(g["ctx"])
    hist = None
    for i, t in enumerate(s.timesteps.tolist()):
        pred = UO.unet_forward(sd, x.repeat(2, 1, 1, 1), torch.tensor([t]), ctx, **UO.SD15).numpy()
        xn, hist = DO.dpmpp_reverse(x.numpy(), t, SO.cfg_combine(*SO.cfg_blend(pred), 7.5), hist, tab, hist_valid=i > 0)
        x = torch.from_numpy(xn)
    return x.numpy()


@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("bf16", 1e-2)])
def test_loop_matches_stepwise_and_oracle(net15, golden_dir, oracle_loop, dev, precision, tol):
    g = np.load(os.path.join(golden_dir, "unet_sd15_golden.npz"))
    net15.set_precision(precision)
    lat, ctx = torch.from_numpy(g["lat16"]).to(dev), torch.from_numpy(g["ctx"]).to(dev)
    smp = sampler(10)
    with torch.no_grad():
        final = denoise(net15, smp, lat, ctx, do_cfg=True, cfg_scale=7.5)
        x = lat.clone()
        for ts in smp.timesteps.to(dev):
            ts = ts.unsqueeze(0)
            x = smp.reverse_process(x, ts, net15(x.repeat(2, 1, 1, 1), ts, ctx), cfg_scale=7.5)
        assert torch.isfinite(final).all() and torch.equal(x, final)
        loop = DenoiseLoop(net15, smp, 1, 16, 16)
        a = loop.run(lat, ctx)
        b = loop.run(lat, ctx)
        assert torch.equal(a, final) and torch.equal(b, final)
    e = rel_l2(final.cpu().numpy(), oracle_loop)
    print(f"DPM-Solver++ loop {precision} vs oracle loop: rel-L2 {e:.3e}")
    assert e < tol


def test_img2img_and_inpaint_loops(net15, dev):
    net15.set_precision("fp32")
    B, h, w = 1, 16, 16
    g = torch.Generator().manual_seed(21)
    lat = torch.randn((B, 4, h, w), generator=g).to(dev)
    ctx = torch.randn((2 * B, 77, 768), generator=g).to(dev)
    enc = torch.randn((1, 4, h, w), generator=g).to(dev)
    mask = (torch.rand((1, 1, h, w), generator=g) > 0.5).to(dev)
    noise = torch.randn((B, 4, h, w), generator=g).to(dev)
    with torch.no_grad():
        got = img2img(net15, sampler(10), enc, noise, ctx, 0.6)
        s = sampler(10, strength=0.6)
        x, _ = s.forward_process(enc, s.timesteps[0].unsqueeze(0), noise)
        for ts in s.timesteps.to(dev):
            ts = ts.unsqueeze(0)
            x = s.reverse_process(x, ts, net15(x.repeat(2, 1, 1, 1), ts, ctx), cfg_scale=7.5)
        assert len(s.timesteps) == 6 and torch.isfinite(got).all() and torch.equal(got, x)
        s = sampler(10, strength=0.6)
        got = inpaint(net15, s, lat, ctx, enc, mask, do_cfg=True, cfg_scale=7.5)
        x = lat
        for ts in s.timesteps.to(dev):
            ts = ts.unsqueeze(0)
            x = s.inpaint_step(x, ts, net15(x.repeat(2, 1, 1, 1), ts, ctx), enc, mask, cfg_scale=7.5)
        assert torch.isfinite(got).all() and torch.equal(got, x)


def test_engine_c_host_and_reload(net15, dev, tmp_path):
    """An exported DPM-Solver++ loop engine, run by tools/c_host/denoise.c and reloaded in-process, == DenoiseLoop.run."""
    if shutil.disk_usage(str(tmp_path)).free < 4 * (1 << 30):
        pytest.skip("needs 4 GiB of scratch space for the engine file")
    net15.set_precision("bf16")
    g = torch.Generator().manual_seed(7)
    lat = torch.randn((1, 4, 16, 16), generator=g)
    ctx = torch.randn((2, 77, 768), generator=g)
    smp = sampler(10, "v_prediction")
    steps = 10
    with torch.no_grad():
        loop = DenoiseLoop(net15, smp, 1, 16, 16, do_cfg=True, cfg_scale=7.5)
        ref = loop.run(lat.to(dev), ctx.to(dev)).cpu()
        loop.reset(lat.to(dev), ctx.to(dev))
        eng = str(tmp_path / "loop.engine")
        loop.export_engine(eng)
    assert torch.isfinite(ref).all()
    lib = _lib.lib()
    h = C.c_void_p()
    _lib.check(lib.sdk_plan_load(eng.encode(), C.byref(h)))
    try:
        st = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        xs, cs, zero = lat.contiguous(), ctx.contiguous(), torch.zeros(1, dtype=torch.int32)
        nan = torch.full_like(xs, float("nan"))
        _lib.check(lib.sdk_plan_upload(h, b"x", xs.data_ptr(), xs.numel() * 4, st))
        _lib.check(lib.sdk_plan_upload(h, b"context", cs.data_ptr(), cs.numel() * 4, st))
        _lib.check(lib.sdk_plan_upload(h, b"history", nan.data_ptr(), nan.numel() * 4, st))     # stale history is never read
        _lib.check(lib.sdk_plan_upload(h, b"counter", zero.data_ptr(), 4, st))
        _lib.check(lib.sdk_plan_launch(h, 1, st))
        for _ in range(steps):
            _lib.check(lib.sdk_plan_launch(h, 4, st))
        out = torch.empty_like(xs)
        _lib.check(lib.sdk_plan_download(h, b"x", out.data_ptr(), out.numel() * 4, st))
        torch.cuda.synchronize()
        assert torch.equal(out, ref)
    finally:
        _lib.check(lib.sdk_plan_destroy(h))
    if shutil.which("gcc") is None:
        pytest.skip("no C compiler on this box (the in-process reload above covers the engine format)")
    exe = str(tmp_path / "denoise")
    libdir = os.path.join(ROOT, "stable-diffusion-pytorch_b200")
    cc = subprocess.run(["gcc", "-O2", "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tools", "c_host", "denoise.c"), "-o", exe,
                         "-L", libdir, "-lsdb200", f"-Wl,-rpath,{libdir}"], capture_output=True, text=True)
    assert cc.returncode == 0, cc.stderr
    lat.numpy().tofile(str(tmp_path / "lat.f32"))
    ctx.numpy().tofile(str(tmp_path / "ctx.f32"))
    r = subprocess.run([exe, eng, "loop", str(tmp_path / "lat.f32"), str(tmp_path / "ctx.f32"), str(steps), str(tmp_path / "out.f32")],
                       capture_output=True, text=True, timeout=600)
    print(r.stdout, r.stderr)
    os.remove(eng)
    assert r.returncode == 0, r.stderr
    got = torch.from_numpy(np.fromfile(str(tmp_path / "out.f32"), dtype=np.float32).reshape(1, 4, 16, 16))
    assert torch.equal(got, ref)
