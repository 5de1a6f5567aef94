"""Benchmark of the denoising hot path (BASELINE.json metric: SD1.5 UNet ms/step & images/sec, 512^2,
DDIM-50, CFG 7.5) on N B200s of one node.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config 2|3|4]
                    [--batch-per-gpu B] [--precision bf16|fp32] [--no-cpu-baseline] [--dump-outputs DIR]

A "step" is one pass of the loop body of models/diffusion.py:223-236 over one batch of synthetic input:
UNet forward on the CFG-doubled batch + guidance blend + DDIM update.  With N GPUs every rank runs its own
shard (data parallel, no collective inside a step; one all-gather of the final latents after the timed
region is checked but not timed).  Rank 0 prints ONE JSON line.  See DESIGN.md §Measurement.

--dump-outputs DIR writes the latents the timed path returned after its last step as DIR/latent.npy (float32;
inputs and weights are seeded, so two builds run with the same arguments can be compared output for output).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

# SURVEY.md §8(d): algorithmic GFLOP per UNet sample (2*MACs of conv/linear + 4*B*H*Sq*Sk*D attention)
GFLOP_PER_SAMPLE = {("sd15", 64): 803.25, ("sd15", 32): 180.08, ("sd21", 64): 804.26, ("sd21", 96): 2149.08}
# dense-contraction part executed by the tcgen05 implicit-GEMM kernel (conv3x3 + s2 + conv1x1 + q/k/v/out proj
# + GEGLU-in + FFN-out), GFLOP per step at UNet batch 2, SD1.5 64x64 (SURVEY.md §8(d) breakdown)
GEMM_GFLOP_B2_SD15_64 = 789.3 + 11.3 + 87.2 + 159.4 + 204.7 + 102.3

CONFIGS = {
    2: dict(arch="sd15", hw=64, steps=50, cfg=True, batch=1, ptype="epsilon", dctx=768,
            name="SD1.5-arch UNet 512^2 (64x64 latent), DDIM-50, CFG 7.5, batch 1 per GPU"),
    3: dict(arch="sd15", hw=64, steps=50, cfg=True, batch=8, ptype="epsilon", dctx=768,
            name="SD1.5-arch UNet 512^2, DDIM-50, CFG 7.5, batch 64 over 8 GPUs (8 per GPU)"),
    4: dict(arch="sd21", hw=96, steps=50, cfg=True, batch=2, ptype="v_prediction", dctx=1024,
            name="SD2.1-arch UNet 768^2 (96x96 latent), DDIM-50, v-prediction, batch 16 over 8 GPUs (2 per GPU)"),
    5: dict(arch="sd21", hw=64, steps=1, cfg=False, batch=32, ptype="epsilon", dctx=1024,
            name="SwiftBrush one-step: SD2.1-arch UNet 512^2, ONE forward at t=999, no CFG, batch 256 over 8 GPUs (32 per GPU)"),
}


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(path, arrays):
    """Write each tensor as `path/<name>.npy` in float32.  A tensor over its share of DUMP_MAX_BYTES is replaced by a fixed,
    seeded sample of its flattened elements (same indices in every run of the same shape)."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    cap = DUMP_MAX_BYTES // (4 * len(arrays))
    for name, t in arrays.items():
        a = t.detach().float().cpu().numpy()
        if a.size > cap:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, cap, replace=False))]
        np.save(os.path.join(path, f"{name}.npy"), a)


def split_steps(k, regions):
    """`k` steps as `regions` (at most k) runs of near-equal length."""
    n = max(1, min(regions, k))
    return [k // n + (i < k % n) for i in range(n)]


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return float(p["hbm_gbs"]), float(p["bf16_tflops"]), float(p.get("bf16_tflops_sustained", p["bf16_tflops"])), "measured"
    except Exception:
        return 6650.0, 1590.0, 1400.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def build_oracle_inputs(cfg, total_batch):
    from oracle import unet_oracle as UO          # synthetic-input recipe + weights (checker infrastructure)
    arch = UO.SD15 if cfg["arch"] == "sd15" else UO.SD21
    sd = UO.make_state_dict(0 if cfg["arch"] == "sd15" else 1, **arch)
    g = torch.Generator().manual_seed(1234)
    latent = torch.randn((total_batch, 4, cfg["hw"], cfg["hw"]), generator=g)
    ctx = torch.randn(((2 if cfg["cfg"] else 1) * total_batch, 77, cfg["dctx"]), generator=g)
    return arch, sd, latent, ctx


# --------------------------------------------------------------------------------------------------
def cpu_loop_body_seconds(cfg, sd, arch, hw, n_timed, budget_s):
    """Seconds per loop-body step of the ORACLE port on the host cores (UNet batch 2B=2 + CFG + DDIM), the number of timed
    steps, and the latent after the last step."""
    from oracle import sampler_oracle as SO
    from oracle import unet_oracle as UO
    UO.USE_SDPA = True                                     # the reference's stock attention path (models/unet/attention.py:37-43)
    torch.set_num_threads(os.cpu_count())
    g = torch.Generator().manual_seed(1234)
    lat = torch.randn((1, 4, hw, hw), generator=g)
    nctx = 2 if cfg["cfg"] else 1
    ctx = torch.randn((nctx, 77, cfg["dctx"]), generator=g)
    _, alphas, a_hat = SO.schedule_fp32()
    ts = SO.ddim_timesteps(1000, 50)
    times = []
    t_start = time.time()
    with torch.no_grad():
        for i in range(n_timed + 1):                       # first iteration = warm-up
            t0 = time.time()
            t = int(ts[min(i, len(ts) - 1)])
            out = UO.unet_forward(sd, lat.repeat(nctx, 1, 1, 1), torch.tensor([t]), ctx, **arch)
            if cfg["cfg"]:
                u, c = SO.cfg_blend(out.numpy())
                eps = SO.cfg_combine(u, c, 7.5)
            else:
                eps = out.numpy()
            lat = torch.from_numpy(SO.ddim_reverse(lat.numpy(), t, eps, alphas, a_hat, 1000, 50, cfg["ptype"]))
            dt = time.time() - t0
            if i > 0:
                times.append(dt)
            if time.time() - t_start > budget_s and len(times) >= 1:
                break
    UO.USE_SDPA = False
    return sum(times) / len(times), len(times), lat


def run_reference_arm(args, cfg):
    """--impl reference: the reference's CPU path (oracle port; the Python reference cannot travel to the GPU box)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    arch, sd, _, _ = build_oracle_inputs(cfg, 1)
    total = args.steps + args.warmup
    hw = cfg["hw"]
    est_full = 6.0 * (GFLOP_PER_SAMPLE[(cfg["arch"], hw)] / 803.25)
    sample = f"full loop-body steps (oracle port, SDPA attention) at {hw}x{hw} latent, UNet batch {2 if cfg['cfg'] else 1}"
    scale = 1.0
    if total * est_full > 240 and (cfg["arch"], 32) in GFLOP_PER_SAMPLE:
        scale = GFLOP_PER_SAMPLE[(cfg["arch"], hw)] / GFLOP_PER_SAMPLE[(cfg["arch"], 32)]
        hw = 32
        sample = f"loop-body steps on a 32x32 latent, time scaled x{scale:.2f} by algorithmic FLOPs to {cfg['hw']}x{cfg['hw']}"
    torch.set_num_threads(os.cpu_count())
    n = max(1, min(args.steps, int(240 / max(est_full / scale, 0.5))))
    sec, used, lat = cpu_loop_body_seconds(cfg, sd, arch, hw, n, budget_s=240)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"latent": lat})
    sec *= scale
    img_s = 1.0 / (cfg["steps"] * sec)
    line = {"impl": "reference", "metric": "images_per_sec", "value": img_s, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": make_config(cfg, cfg["batch"], (2 if cfg["cfg"] else 1) * cfg["batch"]), "timed_steps": used,
            "cpu_baseline": {"value": img_s, "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port", "sample": sample},
            "e2e": {"value": img_s, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


# --------------------------------------------------------------------------------------------------
def time_gemm_family(loop, iters=5, fns=None):
    """Average device time of ALL tcgen05 implicit-GEMM launches of one step, replayed back to back as a graph."""
    lib = loop.prog.lib
    names = fns or ["sdk_tc_gemm_launch"]
    targets = [getattr(lib, n) for n in names]
    ops = [(fn, a) for fn, a in loop.prog.ops if any(fn is t for t in targets)]
    if not ops:
        return None, 0
    g = torch.cuda.CUDAGraph()
    loop.prog.launch(ops)
    torch.cuda.synchronize()
    with torch.cuda.graph(g):
        loop.prog.launch(ops)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g.replay()
    torch.cuda.synchronize()
    e0.record()
    for _ in range(iters):
        g.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters, len(ops)


def torch_eager_on_gpu(cfg, sd, arch, dev, steps=8):
    """The reference's op sequence (oracle port, SDPA attention as in attention.py:37-43) executed by STOCK PyTorch eager
    kernels (cuDNN / cuBLAS / SDPA) on the same GPU: the 'library kernels on the same box' comparator of SURVEY 8(d)."""
    from oracle import unet_oracle as UO
    UO.USE_SDPA = True
    out = {}
    sd_d = {k: v.to(dev) for k, v in sd.items()}
    g = torch.Generator().manual_seed(1234)
    lat = torch.randn((1, 4, cfg["hw"], cfg["hw"]), generator=g).to(dev)
    ctx = torch.randn((2, 77, cfg["dctx"]), generator=g).to(dev)
    t = torch.tensor([981], device=dev)
    for name, ac in (("fp32_tf32", None), ("autocast_bf16", torch.bfloat16)):
        torch.backends.cuda.matmul.allow_tf32 = True
        torch.backends.cudnn.allow_tf32 = True
        def step():
            with torch.no_grad():
                if ac is None:
                    o = UO.unet_forward(sd_d, lat.repeat(2, 1, 1, 1), t, ctx, **arch)
                else:
                    with torch.autocast("cuda", dtype=ac):
                        o = UO.unet_forward(sd_d, lat.repeat(2, 1, 1, 1), t, ctx, **arch)
                u, c = o.float().chunk(2)
                return u + 7.5 * (c - u)
        for _ in range(3):
            step()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        out[name] = {"ms_per_step": ms, "images_per_s": 1.0 / (cfg["steps"] * ms * 1e-3)}
    UO.USE_SDPA = False
    del sd_d
    torch.cuda.empty_cache()
    return out


def run_one_step(args, cfg):
    """BASELINE config 5 (models/diffusion.py:106-113): images/s of UNet forward (no CFG, context batch 1 broadcast) + x0 update."""
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from stable_diffusion_pytorch_b200 import DDIMSampler, UNet
    from stable_diffusion_pytorch_b200.pipeline import one_step
    B = cfg["batch"]
    arch, sd, latent_all, ctx_all = build_oracle_inputs(cfg, B * world)
    net = UNet(attention_head_dim=arch["attention_head_dim"], cross_attention_dim=arch["cross_attention_dim"])
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval().set_precision(args.precision)
    lat = latent_all[rank * B:(rank + 1) * B].to(dev)
    ctx = ctx_all[:1].to(dev)                                # one prompt, broadcast (diffusion.py:102)
    smp = DDIMSampler()
    K, Wm = args.steps, max(args.warmup, 3)
    with torch.no_grad():
        for _ in range(Wm):
            out = one_step(net, smp, lat, ctx)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        sampler = ClockSampler(local_rank)
        sampler.start()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            out = one_step(net, smp, lat, ctx)
        e1.record()
        torch.cuda.synchronize()
        sampler.stop_flag = True
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_step = float(t.item()) / K
        finite = bool(torch.isfinite(out).all().item())
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"latent": out})             # rank 0's images: this path has no gather
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    _, _, tf_sus, peak_src = peaks()
    gf = GFLOP_PER_SAMPLE[(cfg["arch"], cfg["hw"])] * B
    print(json.dumps({
        "metric": "images_per_sec", "value": B * world / (ms_step * 1e-3), "unit": "images/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": args.precision, "data": "synthetic",
        "config": {"workload": cfg["name"], "images_per_gpu": B, "unet_batch_per_gpu": B, "latent": [cfg["hw"], cfg["hw"]], "finite": finite,
                   "l2_policy": "inputs larger than L2: each forward streams 1.73 GB of bf16 weights", "api": "pipeline.one_step (UNet.forward + x0 kernel)"},
        "step_tflops": gf / ms_step, "step_frac_of_peak": gf / ms_step / tf_sus, "peak_source": peak_src,
        "clocks": sampler.summary()}))


def time_vae_decode(dev, B, hw, reps=10):
    """VAE.decode (models/vae/vae.py:270-274) of a (B,4,hw,hw) latent on random-init weights: device time per decode (CUDA events,
    graph replay) and end to end with the latent in pinned host memory and the image copied back to the host."""
    from oracle import vae_oracle as VO          # synthetic weights recipe only (checker infrastructure, outside the timed region)
    from stable_diffusion_pytorch_b200 import VAE
    vae = VAE()
    vae.load_state_dict(VO.make_state_dict(3), strict=True)
    vae = vae.to(dev).eval()
    g = torch.Generator().manual_seed(77)
    z_h = (torch.randn((B, 4, hw, hw), generator=g) * 0.18215 * 4.0).pin_memory()
    z = z_h.to(dev)
    with torch.no_grad():
        for _ in range(3):
            img = vae.decode(z)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            img = vae.decode(z)
        e1.record()
        torch.cuda.synchronize()
        dev_ms = e0.elapsed_time(e1) / reps
        out_h = torch.empty(img.shape, dtype=img.dtype).pin_memory()
        t0 = time.perf_counter()
        for _ in range(reps):
            out_h.copy_(vae.decode(z_h.to(dev, non_blocking=True)), non_blocking=True)
            torch.cuda.current_stream().synchronize()
        e2e_ms = (time.perf_counter() - t0) * 1e3 / reps
    gflop = 2514.5 * B * (hw / 64.0) ** 2            # 2*MACs of every conv / linear + 4*S*S*C of the attention, per 512^2 image (un-folded upsample convs)
    res = {"workload": f"VAE.decode, latent ({B},4,{hw},{hw}) -> image ({B},3,{8 * hw},{8 * hw}), bf16 tensor-core path, random-init weights",
           "ms_per_decode": dev_ms, "images_per_s": B / (dev_ms * 1e-3), "approx_tflops": gflop / dev_ms,
           "e2e_ms_per_decode": e2e_ms, "h2d_bytes": z_h.numel() * 4, "d2h_bytes": out_h.numel() * 4,
           "finite": bool(torch.isfinite(img).all().item())}
    del vae
    torch.cuda.empty_cache()
    return res


def make_config(cfg, B, ub):
    """The `config` object of the JSON line: the workload only, IDENTICAL for our arm and for the reference arm."""
    return {"workload": cfg["name"], "images_per_gpu": B, "unet_batch_per_gpu": ub, "latent": [cfg["hw"], cfg["hw"]],
            "sampler_steps_per_image": cfg["steps"], "cfg_scale": 7.5 if cfg["cfg"] else None,
            "l2_policy": "inputs larger than L2: each step streams 1.72 GB of bf16 weights (L2 = 126 MB)"}


def timed_steps(loop, smp, K, Wm, repeats, dev, world, dist, lat_d, ctx_d):
    """W warm-up steps, then EXACTLY K timed steps split into `repeats` regions (at most K), every region bracketed by
    barrier + synchronize and timed with CUDA events; per-region time = MAX over ranks.  Returns the sorted per-step times
    (ms) of the regions."""
    n_grid = len(smp.timesteps)
    pos = [0]

    def run_steps(n):
        done = 0
        while done < n:                                      # walk the sampler grid; restart the walk when it ends
            m = min(n - done, n_grid - pos[0])
            for _ in range(m):
                loop.step()
            pos[0] += m
            done += m
            if pos[0] >= n_grid:
                loop.counter.zero_()
                pos[0] = 0

    loop.reset(lat_d, ctx_d)
    run_steps(Wm)
    out = []
    for n in split_steps(K, repeats):
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        run_steps(n)
        e1.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out.append(float(t.item()) / n)
    return sorted(out)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50, help="timed steps")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--repeats", type=int, default=5, help="timed regions the --steps steps are split into; the median is reported")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=sorted(CONFIGS))
    ap.add_argument("--batch-per-gpu", type=int, default=0)
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--breakdown", action="store_true", help="also time each kernel class of one step as its own graph")
    ap.add_argument("--no-torch-eager", action="store_true", help="skip timing the reference op sequence in stock PyTorch eager on this GPU")
    ap.add_argument("--no-config3", action="store_true", help="N > 1: skip the batch-64-sharded (BASELINE config 3) measurement")
    ap.add_argument("--no-fp32", action="store_true", help="N = 1: skip the one-off fp32-mode ms/step figure")
    ap.add_argument("--no-vae", action="store_true", help="N = 1: skip the VAE-decode (latent -> image) figure")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the latents of the last timed step as DIR/latent.npy (float32)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    cfg = dict(CONFIGS[args.config])
    if args.batch_per_gpu:
        cfg["batch"] = args.batch_per_gpu
    if args.impl == "reference":
        return run_reference_arm(args, cfg)
    if args.config == 5:
        return run_one_step(args, cfg)
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    import torch.distributed as dist
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from stable_diffusion_pytorch_b200 import DDIMSampler, UNet
    from stable_diffusion_pytorch_b200.dist import gather_latents, shard_inputs
    from stable_diffusion_pytorch_b200.pipeline import DenoiseLoop

    B = cfg["batch"]
    arch, sd, latent_all, ctx_all = build_oracle_inputs(cfg, B * world)
    net = UNet(attention_head_dim=arch["attention_head_dim"], cross_attention_dim=arch["cross_attention_dim"])
    net.load_state_dict(sd, strict=True)
    net = net.to(dev).eval().set_precision(args.precision)
    lat, ctx = shard_inputs(latent_all, ctx_all, rank, world, do_cfg=cfg["cfg"])
    lat_d, ctx_d = lat.to(dev), ctx.to(dev)
    smp = DDIMSampler(prediction_type=cfg["ptype"])
    smp._set_inference_steps(50)
    loop = DenoiseLoop(net, smp, B, cfg["hw"], cfg["hw"], do_cfg=cfg["cfg"], cfg_scale=7.5, use_cuda_graph=not args.no_graph)
    K, Wm = args.steps, args.warmup
    n_grid = len(smp.timesteps)

    with torch.no_grad():
        sampler = ClockSampler(local_rank)
        sampler.start()
        regions = timed_steps(loop, smp, K, Wm, max(1, args.repeats), dev, world, dist, lat_d, ctx_d)
        sampler.stop_flag = True
        ms_step = regions[len(regions) // 2]                  # median region
        last = loop.latent.clone()                            # the loop state after the last timed step
        finite = bool(torch.isfinite(last).all().item())

        # ---- e2e through the public drop-in API with HOST buffers (UNet.forward + sampler.reverse_process)
        ub = 2 * B if cfg["cfg"] else B
        lat_h = lat.clone().pin_memory()
        ctx_h = ctx.clone().pin_memory()
        res_h = torch.empty_like(lat_h).pin_memory()
        ts_list = smp.timesteps.tolist()

        def e2e_step(i):
            x = lat_h.to(dev, non_blocking=True)
            c = ctx_h.to(dev, non_blocking=True)
            tt = torch.tensor([ts_list[i % n_grid]], dtype=torch.int64).to(dev, non_blocking=True)
            xin = x.repeat(2, 1, 1, 1) if cfg["cfg"] else x
            o = net(xin, tt, c)
            y = smp.reverse_process(x, tt, o, cfg_scale=7.5) if cfg["cfg"] else smp.reverse_process(x, tt, o)
            res_h.copy_(y, non_blocking=True)
            torch.cuda.current_stream().synchronize()         # the caller reads the step's result on the host
            lat_h.copy_(res_h)

        for i in range(3):
            e2e_step(i)
        e2e_regions = []
        for k2 in split_steps(K, max(1, min(args.repeats, 3))):
            torch.cuda.synchronize()
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            for i in range(k2):
                e2e_step(3 + i)
            torch.cuda.synchronize()
            t = torch.tensor([(time.perf_counter() - t0) * 1e3 / k2], device=dev)
            if world > 1:
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
            e2e_regions.append(float(t.item()))
        e2e_regions.sort()
        e2e_ms = e2e_regions[len(e2e_regions) // 2]
        h2d = lat_h.numel() * 4 + ctx_h.numel() * 4 + 8
        d2h = res_h.numel() * 4

        # ---- roofline of the dominant kernel family (tcgen05 implicit GEMM), rank 0
        gemm_ms, gemm_launches = (None, 0)
        lln_ms, lln_launches, lln_gflop = (None, 0, 0.0)
        breakdown = None
        if rank == 0 and args.precision == "bf16":
            gemm_ms, gemm_launches = time_gemm_family(loop)
            # projection + LayerNorm cluster launches (sdk_linear_ln): their matmuls are part of the step's conv / linear FLOPs but
            # the kernel also does the LayerNorm, so it is timed and reported on its own
            lln_ms, lln_launches = time_gemm_family(loop, fns=["sdk_linear_ln_launch"])
            from stable_diffusion_pytorch_b200._lib import LinearLnDesc
            lln_gflop = sum(2.0 * d.M * d.K * d.N for d in loop.prog.keep if isinstance(d, LinearLnDesc)) / 1e9
            if args.breakdown:
                breakdown = {}
                for label, fns in (("tc_gemm", ["sdk_tc_gemm_launch"]), ("linear_ln", ["sdk_linear_ln_launch"]), ("attention", ["sdk_attention_bf16", "sdk_attention_tc_launch"]),
                                   ("groupnorm", ["sdk_groupnorm_stats", "sdk_groupnorm_apply", "sdk_groupnorm_fused", "sdk_groupnorm_apply_cs", "sdk_channel_stats"]),
                                   ("layernorm", ["sdk_layernorm"]),
                                   ("other", ["sdk_cast_upsample", "sdk_im2col_s2", "sdk_nchw_to_nhwc", "sdk_gemv", "sdk_time_sinusoid", "sdk_conv_gemm_f32", "sdk_conv_in"])):
                    ms, n = time_gemm_family(loop, fns=fns)
                    breakdown[label] = {"ms": ms, "launches": n}

        # the path's only collective: ONE all-gather of the final latents per generation -- timed once, outside the step loop
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        final = gather_latents(last.clone(), B * world)
        g1.record()
        torch.cuda.synchronize()
        gather_ms = g0.elapsed_time(g1)
        assert final.shape[0] == B * world
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"latent": final})
        launches_per_step = loop.launches_per_step

        # ---- N > 1: BASELINE config 3 (batch 64 SHARDED over the N GPUs: strong scaling) in the same run
        config3 = None
        if world > 1 and args.config == 2 and not args.no_config3 and 64 % world == 0:
            try:
                del loop
                net.invalidate()
                torch.cuda.empty_cache()
                c3 = dict(CONFIGS[3])
                B3 = 64 // world
                _, _, lat3_all, ctx3_all = build_oracle_inputs(c3, 64)          # full batch from ONE generator, then sliced
                l3, x3 = shard_inputs(lat3_all, ctx3_all, rank, world, do_cfg=True)
                loop3 = DenoiseLoop(net, smp, B3, 64, 64, do_cfg=True, cfg_scale=7.5, use_cuda_graph=not args.no_graph)
                k3 = max(3, min(K, 10))
                reg3 = timed_steps(loop3, smp, k3, 3, max(1, min(args.repeats, 3)), dev, world, dist, l3.to(dev), x3.to(dev))
                ms3 = reg3[len(reg3) // 2]
                fin3 = bool(torch.isfinite(loop3.latent).all().item())
                torch.cuda.synchronize()
                dist.barrier()
                g0.record()
                final3 = gather_latents(loop3.latent.clone(), 64)
                g1.record()
                torch.cuda.synchronize()
                _, _, tf_sus3, _ = peaks()
                gf3 = GFLOP_PER_SAMPLE[("sd15", 64)] * 2 * B3                     # per GPU per step
                config3 = {"workload": "SD1.5-arch UNet 512^2, DDIM-50, CFG 7.5, batch 64 sharded over %d GPUs (%d images, UNet batch %d per GPU)" % (world, B3, 2 * B3),
                           "scaling": "strong", "ms_per_step": ms3, "ms_per_step_min": reg3[0], "ms_per_step_max": reg3[-1], "timed_steps": k3,
                           "images_per_s": 64 / (50 * ms3 * 1e-3), "step_tflops_per_gpu": gf3 / ms3, "frac": gf3 / ms3 / tf_sus3,
                           "gather_latents_ms": g0.elapsed_time(g1), "gathered": list(final3.shape), "finite": fin3}
                del loop3
            except Exception as ex:                                               # never take the headline line down
                config3 = {"error": repr(ex)}

        # ---- N = 1: what the exact-fp32 mode (the 1e-4 parity gate) costs per step, reported once
        fp32_ms = None
        if world == 1 and args.precision == "bf16" and not args.no_fp32 and args.config == 2:
            try:
                if "loop" in dir():
                    del loop
                net.invalidate()
                torch.cuda.empty_cache()
                net.set_precision("fp32")
                loopf = DenoiseLoop(net, smp, B, cfg["hw"], cfg["hw"], do_cfg=cfg["cfg"], cfg_scale=7.5, use_cuda_graph=not args.no_graph)
                regf = timed_steps(loopf, smp, 3, 3, 1, dev, 1, dist, lat_d, ctx_d)
                fp32_ms = regf[0]
                del loopf
                net.invalidate()
                net.set_precision(args.precision)
                torch.cuda.empty_cache()
            except Exception as ex:
                fp32_ms = repr(ex)

        # ---- N = 1: the stage after the loop (SURVEY 8(f) rank 1): VAE.decode, latent -> 512^2 image, device-timed and end to end
        vae_line = None
        if world == 1 and args.precision == "bf16" and not args.no_vae and args.config == 2:
            try:
                vae_line = time_vae_decode(dev, B, cfg["hw"])
            except Exception as ex:
                vae_line = {"error": repr(ex)}

    if world > 1:
        dist.barrier()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    hbm, tf_burst, tf_sus, peak_src = peaks()
    imgs_per_s = (B * world) / (cfg["steps"] * ms_step * 1e-3)
    e2e_imgs = (B * world) / (cfg["steps"] * e2e_ms * 1e-3)
    gf_sample = GFLOP_PER_SAMPLE[(cfg["arch"], cfg["hw"])]
    step_gflop = gf_sample * ub
    roof = None
    if gemm_ms:
        gemm_gflop = GEMM_GFLOP_B2_SD15_64 * (ub / 2.0) if (cfg["arch"], cfg["hw"]) == ("sd15", 64) else None
        if gemm_gflop:
            # dominant kernel = conv_gemm_tc_kernel: the FLOPs of ITS launches (all conv / linear FLOPs of the step minus the
            # matmuls that run inside the projection + LayerNorm kernel) over the device time of ITS launches
            ach = (gemm_gflop - lln_gflop) / gemm_ms            # GFLOP / ms == TFLOP/s
            traffic, traffic_src = None, None
            for name in ("r02b_gemm_traffic.json", "r02_gemm_traffic.json", "r01_gemm_traffic.json"):
                try:
                    with open(os.path.join(ROOT, "profiles", name)) as f:
                        tj = json.load(f)
                    if ub == 2:                       # captured for UNet batch 2 only
                        traffic, traffic_src = tj["dram_bytes_read"] + tj["dram_bytes_write"], name
                    break
                except Exception:
                    continue
            roof = {"bound": "tensor", "achieved": ach, "peak": tf_sus, "unit": "TFLOP/s", "frac": ach / tf_sus, "traffic": traffic,
                    "traffic_note": f"DRAM bytes of all launches of the kernel in one step (ncu, cold L2 per launch): profiles/{traffic_src}",
                    "kernel": "conv_gemm_tc_kernel (tcgen05 implicit GEMM), all launches of one step",
                    "gflop_per_step_in_kernel": gemm_gflop - lln_gflop,
                    "launches_per_step": gemm_launches, "ms_per_step_in_kernel": gemm_ms, "share_of_step": gemm_ms / ms_step,
                    "peak_source": f"MEASURED_PEAKS.json bf16_tflops_sustained ({peak_src})"}
            if lln_ms:
                roof["linear_ln"] = {"kernel": "linear_ln_kernel (tcgen05 projection + bias + residual + LayerNorm, one cluster launch)",
                                     "launches_per_step": lln_launches, "ms_per_step_in_kernel": lln_ms, "gflop_per_step_in_kernel": lln_gflop,
                                     "achieved": lln_gflop / lln_ms, "share_of_step": lln_ms / ms_step,
                                     "note": "latency-bound: 48 launches of 1.3-25 GFLOP matmul + the LayerNorm of their rows"}
                roof["family_frac"] = gemm_gflop / (gemm_ms + lln_ms) / tf_sus
    line = {
        "metric": "images_per_sec", "value": imgs_per_s, "unit": "images/s", "n_gpus": world, "steps": K, "warmup": Wm,
        "ms_per_step": ms_step, "ms_per_step_min": regions[0], "ms_per_step_max": regions[-1], "repeats": len(regions),
        "timing": "`steps` steps split into `repeats` CUDA-event-timed regions; median of the regions' per-step times (max over ranks per region)",
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": args.precision, "data": "synthetic",
        "config": make_config(cfg, B, ub), "cuda_graph": not args.no_graph, "finite": finite,
        "step_tflops": step_gflop / ms_step, "step_frac_of_peak": step_gflop / ms_step / tf_sus,
        "clocks": sampler.summary(),
        "e2e": {"value": e2e_imgs, "unit": "images/s", "ms_per_step": e2e_ms, "ms_per_step_min": e2e_regions[0], "ms_per_step_max": e2e_regions[-1],
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "api": "UNet.forward + DDIMSampler.reverse_process, pinned host buffers in and out every step"},
        "gpu_launches": launches_per_step * K,
        "gather_latents_ms": gather_ms,
        "roofline": roof,
    }
    if config3 is not None:
        line["config3"] = config3
    if fp32_ms is not None:
        line["fp32_mode_ms_per_step"] = fp32_ms
    if vae_line is not None:
        line["vae_decode"] = vae_line
    if breakdown:
        line["breakdown_ms_per_step"] = breakdown
    if not args.no_torch_eager and cfg["cfg"] and world == 1:
        try:
            line["torch_eager_same_gpu"] = torch_eager_on_gpu(cfg, sd, arch, dev)
        except Exception as ex:
            line["torch_eager_same_gpu"] = {"error": repr(ex)}
    if not args.no_cpu_baseline and world >= 1:
        try:
            sec, used, _ = cpu_loop_body_seconds(cfg, sd, arch, cfg["hw"], 2, budget_s=45)
            line["cpu_baseline"] = {"value": 1.0 / (cfg["steps"] * sec), "unit": "images/s", "cores": torch.get_num_threads(), "kind": "port",
                                    "sample": f"{used} loop-body steps (after 1 warm-up) of the oracle port (SDPA attention as attention.py:37-43) at {cfg['hw']}x{cfg['hw']}, extrapolated x{cfg['steps']}",
                                    "s_per_step": sec}
        except Exception as ex:                               # the baseline must never take the bench line down
            line["cpu_baseline"] = {"error": repr(ex)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
