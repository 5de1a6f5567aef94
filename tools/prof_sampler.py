"""Cost of the DPM-Solver++(2M) sampler next to DDIM; prints one JSON line.

    python tools/prof_sampler.py [--launches 200] [--repeats 7] [--steps 20]

* kernel: device time of one sdk_dpmpp_step against one sdk_ddim_step (CFG on, order-2 row with the history read) at
  the latents of BASELINE configs 2 (1 x 4 x 64 x 64), 3 per GPU (8 x 4 x 64 x 64) and 4 per GPU (2 x 4 x 96 x 96).  Each is a
  CUDA graph of --launches back-to-back launches, timed with CUDA events; median and spread over --repeats replays.  Bytes moved:
  DDIM reads x, u, c and writes x (16 B per element); DPM-Solver++ also reads and writes the history (24 B).  The working sets fit
  the 126 MB L2, as they do inside the sampling loop.
* loop: DenoiseLoop ms/step at config 2 (SD1.5-arch UNet, seeded default init, bf16, CFG 7.5) for DDIM and for DPM-Solver++,
  alternated in one process: warm-up steps, then --repeats regions of --steps steps each, CUDA events; median and spread.
* images/s of DPM-Solver++ at 20 steps next to DDIM at 50, from those step times.
* the card's name and power limit, read in the same run (read-only query).
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from stable_diffusion_pytorch_b200 import DDIMSampler, DPMSolverSampler, UNet, _lib  # noqa: E402
from stable_diffusion_pytorch_b200.pipeline import DenoiseLoop  # noqa: E402
from stable_diffusion_pytorch_b200.scheduler import PRED_EPS  # noqa: E402

LATENTS = {"config2": (1, 4, 64, 64), "config3_per_gpu": (8, 4, 64, 64), "config4_per_gpu": (2, 4, 96, 96)}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip() if q.returncode == 0 else None}


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1]}


def time_graph(fn, launches, repeats):
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        fn()                                                   # warm: module load, table upload
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=s):
            for _ in range(launches):
                fn()
    g.replay()
    torch.cuda.synchronize()
    out = []
    for _ in range(repeats):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) * 1e3 / launches)      # us per launch
    return stats(out)


def kernel_times(dev, launches, repeats):
    lib = _lib.lib()
    ddim, dpm = DDIMSampler(), DPMSolverSampler()
    for s in (ddim, dpm):
        s._set_inference_steps(20)
    t = int(dpm.timesteps[5])                                  # an order-2 row: the history is read
    tab_ddim, tab_dpm = ddim._coef_table(dev, 0.0), dpm._coef_table(dev, 0.0)
    res = {}
    for name, shape in LATENTS.items():
        g = torch.Generator(device=dev).manual_seed(0)
        x = torch.randn(shape, device=dev, generator=g)
        mo = torch.randn((2 * shape[0],) + shape[1:], device=dev, generator=g) * 1e-3
        hist, out = x.clone(), torch.empty_like(x)                # out of place: x stays the same over the repeats
        n = x.numel()
        eu, ec = mo.data_ptr(), mo.data_ptr() + 4 * n

        def run_ddim():
            _lib.check(lib.sdk_ddim_step(x.data_ptr(), eu, ec, 7.5, 0, out.data_ptr(), n, tab_ddim.data_ptr(), ddim.noise_step, 0, t,
                                         PRED_EPS, C.c_void_p(torch.cuda.current_stream().cuda_stream)))

        def run_dpm():
            _lib.check(lib.sdk_dpmpp_step(x.data_ptr(), eu, ec, 7.5, hist.data_ptr(), 1, out.data_ptr(), n, tab_dpm.data_ptr(),
                                          dpm.noise_step, 0, t, PRED_EPS, C.c_void_p(torch.cuda.current_stream().cuda_stream)))

        a = time_graph(run_ddim, launches, repeats)
        b = time_graph(run_dpm, launches, repeats)
        assert torch.isfinite(out).all()
        res[name] = {"elements": n, "ddim_us": a, "dpmpp_us": b, "ddim_bytes": 16 * n, "dpmpp_bytes": 24 * n,
                     "ddim_GBps": 16 * n / a["median"] / 1e3, "dpmpp_GBps": 24 * n / b["median"] / 1e3}
    return res


def loop_times(dev, steps, repeats, warmup):
    torch.manual_seed(0)
    net = UNet().to(dev).eval().set_precision("bf16")
    g = torch.Generator().manual_seed(1)
    lat = torch.randn((1, 4, 64, 64), generator=g).to(dev)
    ctx = torch.randn((2, 77, 768), generator=g).to(dev)
    loops = {}
    for name, cls in (("ddim", DDIMSampler), ("dpmpp", DPMSolverSampler)):
        s = cls()
        s._set_inference_steps(steps)
        loops[name] = DenoiseLoop(net, s, 1, 64, 64, do_cfg=True, cfg_scale=7.5)
    times = {k: [] for k in loops}
    with torch.no_grad():
        for loop in loops.values():
            loop.reset(lat, ctx)
            for _ in range(warmup):
                loop.step()
        for _ in range(repeats):
            for name, loop in loops.items():                  # alternate the two in the same process
                loop.reset(lat, ctx)
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(steps):
                    loop.step()
                e1.record()
                torch.cuda.synchronize()
                times[name].append(e0.elapsed_time(e1) / steps)
        finite = all(bool(torch.isfinite(loop.latent).all()) for loop in loops.values())
    return {k: stats(v) for k, v in times.items()}, finite


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--launches", type=int, default=200)
    ap.add_argument("--repeats", type=int, default=7)
    ap.add_argument("--steps", type=int, default=20, help="steps per timed loop region (one full grid)")
    ap.add_argument("--warmup", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("prof_sampler.py measures on a CUDA device; none is visible")
    dev = torch.device("cuda:0")
    kern = kernel_times(dev, args.launches, args.repeats)
    loop, finite = loop_times(dev, args.steps, args.repeats, args.warmup)
    ms_ddim, ms_dpm = loop["ddim"]["median"], loop["dpmpp"]["median"]
    print(json.dumps({
        "card": card(),
        "kernel": kern,
        "loop_config2_ms_per_step": loop,
        "loop_finite": finite,
        "images_per_s": {"ddim_50": 1e3 / (50 * ms_ddim), "dpmpp_20": 1e3 / (20 * ms_dpm)},
        "method": f"kernel: CUDA graph of {args.launches} launches x {args.repeats} replays; loop: {args.warmup} warm-up steps, "
                  f"{args.repeats} alternating regions of {args.steps} steps, CUDA events",
    }))


if __name__ == "__main__":
    main()
