"""LoRA merge cost at config 2 (SD1.5 architecture, bf16, 64x64 latent, UNet batch 2 = CFG over one image), one JSON line.

    python tools/prof_lora.py [--steps 20] [--out FILE]

Two seeded synthetic adapters: rank 64 on every transformer Linear, rank 32 LoCon on every conv.  Reports the device time of the
merge launches (CUDA events) with bytes/s and FLOP/s and which bound applies; host time of load_lora / set_lora_scale / unload_lora,
each ending in a synchronise; the path without this feature (merge into the parameters with torch, invalidate(), first forward
re-packs, re-plans and re-captures), timed the same way; and ms/step of the DenoiseLoop with and without the adapters, alternated.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from stable_diffusion_pytorch_b200 import DDIMSampler, DenoiseLoop, UNet, _lib, lora  # noqa: E402
from stable_diffusion_pytorch_b200.arch import param_spec  # noqa: E402

HBM_BPS, FFMA_FLOPS = 7.7e12, 2 * 148 * 128 * 1.965e9      # B200 data sheet bandwidth; fp32 FFMA peak at the 1965 MHz boost clock


def adapter(arch, rank, convs, seed):
    """kohya state dict: rank-``rank`` factors on every transformer Linear (convs=False) or LoCon on every conv (convs=True)."""
    g = torch.Generator().manual_seed(seed)
    shapes, sd = dict(param_spec(arch)), {}
    for dpath, ref in lora.targets(arch).items():
        shape = shapes[ref]
        is_conv = len(shape) == 4 and not dpath.endswith(("proj_in", "proj_out"))
        if is_conv != convs:
            continue
        k = 1
        for d in shape[1:]:
            k *= d
        stem = "lora_unet_" + dpath.replace(".", "_")
        sd[f"{stem}.lora_down.weight"] = torch.randn((rank,) + tuple(shape[1:]), generator=g) / k ** 0.5
        up = torch.randn((shape[0], rank), generator=g) * 0.01
        sd[f"{stem}.lora_up.weight"] = up[:, :, None, None] if is_conv else up
        sd[f"{stem}.alpha"] = torch.tensor(float(rank))
    return sd


def timed(fn, dev):
    torch.cuda.synchronize(dev)
    t0 = time.perf_counter()
    fn()
    torch.cuda.synchronize(dev)
    return (time.perf_counter() - t0) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "prof_lora.py measures on the GPU"
    dev = torch.device("cuda:0")
    torch.manual_seed(0)
    net = UNet().to(dev).eval().set_precision("bf16")
    a_lin, a_conv = adapter(net.arch, 64, False, 1), adapter(net.arch, 32, True, 2)
    smp = DDIMSampler()
    smp._set_inference_steps(50)
    g = torch.Generator().manual_seed(3)
    lat, ctx = torch.randn((1, 4, 64, 64), generator=g).to(dev), torch.randn((2, 77, 768), generator=g).to(dev)
    lib = _lib.lib()
    res = {"config": "SD1.5 bf16 64x64 latent, UNet batch 2", "adapters": "rank 64 on every transformer Linear + rank 32 LoCon on every conv"}
    with torch.no_grad():
        loop = DenoiseLoop(net, smp, 1, 64, 64, do_cfg=True, cfg_scale=7.5)
        loop.run(lat, ctx, steps=3)
        # ---- host time of the API calls
        res["load_lora_ms"] = timed(lambda: (net.load_lora(a_lin, name="lin"), net.load_lora(a_conv, name="conv")), dev)
        res["set_lora_scale_ms"] = timed(lambda: (net.set_lora_scale("lin", 0.5), net.set_lora_scale("conv", 0.5)), dev)
        res["unload_lora_ms"] = timed(lambda: net.unload_lora(), dev)
        # ---- device time of the merge launches alone
        net.load_lora(a_lin, name="lin")
        net.load_lora(a_conv, name="conv")
        pw = net._weights(dev)
        params = dict(net.named_parameters())
        ops, nbytes, flops = [], 0, 0
        for ref in sorted({r for _, m in net._lora.values() for r in m}):
            mods = [(m[ref], s) for _, (s, m) in sorted(net._lora.items()) if ref in m]
            for op in lora.merge_ops(net.arch, pw, ref, params[ref], mods):
                n, k = op["base"].shape
                r = op["up"].shape[1]
                code = _lib.BF16_T if op["dst"].dtype == torch.bfloat16 else _lib.F32_T
                ops.append((op, (op["base"].data_ptr(), k, op["up"].data_ptr(), op["down"].data_ptr(), r,
                                 op["dst"].data_ptr() + op["offset"] * op["dst"].element_size(), code, op["layout"], op["dst_rows"],
                                 op["row_off"], op["row_step"], n, k)))
                nbytes += n * k * (4 + op["dst"].element_size()) + 4 * r * (n + k)
                flops += 2 * n * k * r
        stream = C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 5
        for _ in range(2):
            for _, a in ops:
                _lib.check(lib.sdk_lora_merge(*a, stream))
        e0.record()
        for _ in range(reps):
            for _, a in ops:
                _lib.check(lib.sdk_lora_merge(*a, stream))
        e1.record()
        e1.synchronize()
        t = e0.elapsed_time(e1) / reps * 1e-3
        res["merge_launches"] = len(ops)
        res["merge_device_ms"] = t * 1e3
        res["merge_bytes"], res["merge_flops"] = nbytes, flops
        res["merge_GBps"], res["merge_TFLOPs"] = nbytes / t / 1e9, flops / t / 1e12
        res["merge_bound"] = "memory" if nbytes / HBM_BPS > flops / FFMA_FLOPS else "fp32 FFMA"
        res["merge_share_of_bound"] = max(nbytes / HBM_BPS, flops / FFMA_FLOPS) / t
        del ops
        # ---- ms/step with and without the adapters, alternated (the launch list is the same)
        x, tt = lat.repeat(2, 1, 1, 1), torch.tensor([481], device=dev)

        def ms_per_step():
            loop.reset(lat, ctx)
            loop.step()
            e0.record()
            for _ in range(args.steps):
                loop.step()
            e1.record()
            e1.synchronize()
            return e0.elapsed_time(e1) / args.steps

        with_a, without = [], []
        for _ in range(3):
            with_a.append(ms_per_step())
            net.unload_lora()
            without.append(ms_per_step())
            net.load_lora(a_lin, name="lin")
            net.load_lora(a_conv, name="conv")
        res["ms_per_step_with_adapters"], res["ms_per_step_without"] = min(with_a), min(without)
        res["ms_per_step_samples"] = {"with": with_a, "without": without}
        net.unload_lora()
        # ---- the path without this feature: merge into the parameters, invalidate, re-pack / re-plan / re-capture on first use
        loop = None
        net(x, tt, ctx)
        net(x, tt, ctx)
        net(x, tt, ctx)
        mods = {**lora.read_adapter(a_lin, net.arch)[0], **lora.read_adapter(a_conv, net.arch)[0]}
        saved = {ref: params[ref].detach().clone() for ref in mods}

        def today():
            for ref, m in mods.items():
                w = params[ref]
                w.add_((m.mult * (m.up.to(dev) @ m.down.to(dev).reshape(m.down.shape[0], -1))).reshape(w.shape))
            net.invalidate()
            for _ in range(3):                                  # eager run, capture, replay
                net(x, tt, ctx)

        res["torch_merge_invalidate_first_forward_ms"] = timed(today, dev)
        for ref, w in saved.items():
            params[ref].copy_(w)
        net.invalidate()
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    res["gpu"] = q.stdout.strip().splitlines()[0] if q.returncode == 0 else torch.cuda.get_device_name(dev)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
