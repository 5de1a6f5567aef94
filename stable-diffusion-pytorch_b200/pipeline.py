"""The denoising loop as ONE replayable device program — drop-in for the loop body of the
reference's ``StableDiffusion.generate`` (models/diffusion.py:223-236) and for the one-step path
(models/diffusion.py:106-113).

Per step the reference does: ``latent.repeat(2,...)`` -> UNet -> ``chunk(2)`` -> ``u + s*(c-u)`` ->
``sampler.reverse_process`` with three host syncs.  Here a step is a single CUDA-graph replay:

    next_timestep (device walk of the host-built grid)  ->  UNet step program (batch 2B, the repeat is
    folded into the NCHW->NHWC gather)  ->  fused CFG + DDIM/DDPM update, in place on the latent state

so the host enqueues one graph launch per step and never synchronises.  The timestep grid, the
coefficient tables and all index bookkeeping are the sampler's (bit-exact with the reference).
"""
from __future__ import annotations

import ctypes as C
from typing import Optional

import torch

from . import _lib
from .program import GraphRunner
from .scheduler import PRED_EPS, PRED_V, DDIMSampler, DDPMSampler, x0_from_eps
from .unet import StepProgram, UNet, same_context, tensor_version


class DenoiseLoop:
    """Sampler loop for a fixed problem shape.

    loop = DenoiseLoop(unet, sampler, batch=B, height=h, width=w, do_cfg=True, cfg_scale=7.5)
    latent = loop.run(latent, context)          # context rows [uncond ; cond] when do_cfg
    """

    def __init__(self, unet: UNet, sampler, batch: int, height: int, width: int, *, do_cfg: bool = True,
                 cfg_scale: float = 7.5, context_len: int = 77, context_batch: Optional[int] = None,
                 device=None, use_cuda_graph: Optional[bool] = None):
        if not isinstance(sampler, (DDIMSampler, DDPMSampler)):
            raise TypeError("sampler must be a stable_diffusion_pytorch_b200 DDIMSampler/DDPMSampler")
        self.unet, self.sampler = unet, sampler
        self.device = torch.device(device) if device is not None else next(unet.parameters()).device
        if self.device.type != "cuda":
            raise RuntimeError("DenoiseLoop needs the UNet on a CUDA device; there is no CPU fallback")
        self.B, self.H, self.W = batch, height, width
        self.do_cfg, self.cfg_scale = do_cfg, float(cfg_scale)
        ub = 2 * batch if do_cfg else batch
        bc = ub if context_batch is None else context_batch
        self.lib = _lib.lib()
        pw = unet._weights(self.device)
        self.prog = StepProgram(unet, pw, ub, height, width, 1, bc, context_len, b_src=batch)
        self.runner = GraphRunner(self.prog, unet.use_cuda_graph if use_cuda_graph is None else use_cuda_graph, self._enqueue_step)
        self.latent = self.prog.x_in                         # the loop state IS the UNet's input staging buffer
        with torch.inference_mode(False), torch.no_grad():     # loop state stays writable when built under inference_mode
            self.noise = torch.empty_like(self.latent) if isinstance(sampler, DDPMSampler) else None
            self.counter = torch.zeros(1, dtype=torch.int32, device=self.device)
        self.ts_table = None
        self.tb_table = None
        self.hoist_time = True                                # precompute the time-embedding rows of the grid (exactly the per-step values)
        self._grid_key = None
        self._cond_ref, self._cond_version = None, -1
        self.launches_per_step = len(self.prog.body_ops) + 3
        self.inpaint_orig, self.inpaint_mask = None, None     # set_inpaint(): the step becomes the inpainting loop body

    def set_inpaint(self, encoded_img: Optional[torch.Tensor], mask: Optional[torch.Tensor]):
        """Turn the loop into the inpainting loop of models/diffusion.py:379-398 (context rows [cond ; uncond], CFG form
        s*(c-u)+c, known region re-noised from ``encoded_img`` every step); ``None, None`` restores plain sampling."""
        if encoded_img is None:
            self.inpaint_orig, self.inpaint_mask = None, None
        else:
            o = encoded_img.to(self.device, torch.float32).contiguous()
            if o.shape[0] not in (1, self.B) or tuple(o.shape[1:]) != tuple(self.latent.shape[1:]):
                raise RuntimeError(f"encoded_img {tuple(o.shape)} does not broadcast against the latent {tuple(self.latent.shape)}")
            if mask.numel() != self.H * self.W:
                raise RuntimeError(f"mask must hold one value per latent pixel ({self.H}x{self.W})")
            self.inpaint_orig = o
            self.inpaint_mask = mask.to(self.device).reshape(self.H * self.W).ne(0).to(torch.uint8).contiguous()
        self.runner.graph = None                               # pointers are baked into the captured launches

    # ---- one step = [next timestep] + UNet program + [CFG + scheduler update in place] -------------------
    def _enqueue_step(self):
        s, p, lib = self.sampler, self.prog, self.lib
        stream = C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(lib.sdk_next_timestep(self.ts_table.data_ptr(), self.ts_table.numel(), self.counter.data_ptr(),
                                         p.t_in.data_ptr(), stream))
        if self.tb_table is not None:
            # the time-embedding projections of the whole grid were computed in _prepare: fetch this step's row (counter was
            # advanced by next_timestep) and run the step without the 4-launch time-embedding chain
            _lib.check(lib.sdk_gather_row(self.tb_table.data_ptr(), p.tb.shape[1], self.tb_table.shape[0], self.counter.data_ptr(), -1,
                                          p.tb.data_ptr(), stream))
            p.launch(p.body_ops)
        else:
            p.launch(p.ops)
        n = self.latent.numel()
        out = p.out
        eps_u = out.data_ptr()
        eps_c = out.data_ptr() + 4 * n if self.do_cfg else 0
        if isinstance(s, DDPMSampler) and self.inpaint_orig is not None:
            ch = self.latent.shape[1]                  # rows are [cond ; uncond] in the inpaint loop: eps_u / eps_c name the halves
            _lib.check(lib.sdk_ddpm_inpaint_step(self.latent.data_ptr(), eps_u, eps_c, self.cfg_scale, self.inpaint_orig.data_ptr(),
                                                 self.inpaint_orig.shape[0], self.inpaint_mask.data_ptr(), self.noise.data_ptr(),
                                                 self.latent.data_ptr(), self.B, ch, self.H * self.W, self.coef.data_ptr(), s.noise_step,
                                                 p.t_in.data_ptr(), 0, stream))
        elif isinstance(s, DDPMSampler):
            _lib.check(lib.sdk_ddpm_step(self.latent.data_ptr(), eps_u, eps_c, self.cfg_scale, self.noise.data_ptr(),
                                         self.latent.data_ptr(), n, self.coef.data_ptr(), s.noise_step, p.t_in.data_ptr(), 0, stream))
        elif self.inpaint_orig is not None:
            pred = PRED_V if s.prediction_type == "v_prediction" else PRED_EPS
            ch = self.latent.shape[1]
            _lib.check(lib.sdk_ddim_inpaint_step(self.latent.data_ptr(), eps_u, eps_c, self.cfg_scale, self.inpaint_orig.data_ptr(),
                                                 self.inpaint_orig.shape[0], self.inpaint_mask.data_ptr(), self.latent.data_ptr(),
                                                 self.B, ch, self.H * self.W, self.coef.data_ptr(), s.noise_step, p.t_in.data_ptr(), 0,
                                                 pred, stream))          # rows are [cond ; uncond] here: eps_u/eps_c name the halves
        else:
            pred = PRED_V if s.prediction_type == "v_prediction" else PRED_EPS
            _lib.check(lib.sdk_ddim_step(self.latent.data_ptr(), eps_u, eps_c, self.cfg_scale, 0, self.latent.data_ptr(), n,
                                         self.coef.data_ptr(), s.noise_step, p.t_in.data_ptr(), 0, pred, stream))

    def export_engine(self, path: str):
        """Engine file of the WHOLE sampling loop for a host without Python (sdk_plan_load; tools/c_host/denoise.c): programs 0-3 of
        the UNet plan plus program 4 = one sampler step (next timestep -> time-embedding row -> UNet -> CFG + DDIM/DDPM update in
        place).  Call after ``reset`` (the timestep grid, coefficient and time-embedding tables are baked in as constants).
        Named regions: "x" (the latent state, NCHW fp32), "context", "counter" (int32 grid position: zero it to restart), "out",
        and "noise" for DDPM."""
        s, p = self.sampler, self.prog
        if self.ts_table is None:
            raise RuntimeError("export_engine: call reset(latent, context) first (the timestep grid is part of the engine)")
        if self.inpaint_orig is not None:
            raise RuntimeError("export_engine: the inpainting loop is not exportable (its image / mask are per-call inputs)")
        pid = StepProgram.PROGRAM_LOOP_STEP
        if self.lib.sdk_plan_num_launches(p._ensure_plan(), pid) == 0:
            p.plan_add(pid, "sdk_next_timestep", (self.ts_table.data_ptr(), self.ts_table.numel(), self.counter.data_ptr(), p.t_in.data_ptr()))
            body = p.ops
            if self.tb_table is not None:
                p.plan_add(pid, "sdk_gather_row", (self.tb_table.data_ptr(), p.tb.shape[1], self.tb_table.shape[0], self.counter.data_ptr(),
                                                   -1, p.tb.data_ptr()))
                body = p.body_ops
            for fn, args in body:
                p.plan_add(pid, fn.__name__, args)
            n = self.latent.numel()
            eps_u = p.out.data_ptr()
            eps_c = p.out.data_ptr() + 4 * n if self.do_cfg else 0
            if isinstance(s, DDPMSampler):
                p.plan_add(pid, "sdk_ddpm_step", (self.latent.data_ptr(), eps_u, eps_c, self.cfg_scale, self.noise.data_ptr(),
                                                  self.latent.data_ptr(), n, self.coef.data_ptr(), s.noise_step, p.t_in.data_ptr(), 0))
            else:
                pred = PRED_V if s.prediction_type == "v_prediction" else PRED_EPS
                p.plan_add(pid, "sdk_ddim_step", (self.latent.data_ptr(), eps_u, eps_c, self.cfg_scale, 0, self.latent.data_ptr(), n,
                                                  self.coef.data_ptr(), s.noise_step, p.t_in.data_ptr(), 0, pred))
        extra = [(self.ts_table, 0, ""), (self.coef, 0, ""), (self.counter, 2, "counter")]
        if self.tb_table is not None:
            extra.append((self.tb_table, 0, ""))
        if self.noise is not None:
            extra.append((self.noise, 2, "noise"))
        p.export_engine(path, extra_regions=extra)

    def _prepare(self, context: torch.Tensor):
        s, p = self.sampler, self.prog
        key = (tuple(s.timesteps.tolist()), s._stride())
        if key != self._grid_key:
            self.ts_table = s.timesteps.to(self.device, torch.int64).contiguous()
            self.coef = s._coef_table(self.device, 0.0)
            self._grid_key = key
            self.runner.graph = None                           # tables are baked into the captured launches
            # time embedding -> 22 ResBlock projections depend only on t: run that chain once per grid point, keep the rows
            self.tb_table = None
            if self.hoist_time and p.nt == 1:
                rows = []
                for tv in self.ts_table.tolist():
                    p.t_in.fill_(tv)
                    p.launch(p.time_ops)
                    rows.append(p.tb[0].clone())
                self.tb_table = torch.stack(rows).contiguous()
        if not same_context(context, self._cond_ref, self._cond_version):
            if tuple(context.shape) != tuple(p.cond_in.shape):
                raise RuntimeError(f"context shape {tuple(context.shape)} != {tuple(p.cond_in.shape)}")
            p.cond_in.copy_(context, non_blocking=True)
            p.launch(p.ctx_ops)                                # cross-attention K/V once per generation (loop-invariant)
            self._cond_ref, self._cond_version = context, tensor_version(context)

    def step(self):
        """Advance the latent state by one sampler step (device-side timestep walk)."""
        if isinstance(self.sampler, DDPMSampler):
            # same global-RNG draw as ddpm.py:80, outside the graph so torch's generator state advances normally
            self.noise.copy_(torch.randn(self.latent.shape, dtype=self.latent.dtype, device=self.device))
        self.runner.run()

    def reset(self, latent: torch.Tensor, context: torch.Tensor):
        if tuple(latent.shape) != tuple(self.latent.shape):
            raise RuntimeError(f"latent shape {tuple(latent.shape)} != {tuple(self.latent.shape)}")
        self._prepare(context)
        self.latent.copy_(latent, non_blocking=True)
        self.counter.zero_()

    def run(self, latent: torch.Tensor, context: torch.Tensor, steps: Optional[int] = None) -> torch.Tensor:
        """Full loop over ``sampler.timesteps`` (or the first ``steps`` of them); returns the final latent."""
        self.reset(latent, context)
        n = len(self.sampler.timesteps) if steps is None else steps
        for _ in range(n):
            self.step()
        return self.latent.clone()


@torch.no_grad()
def denoise(unet: UNet, sampler, latent: torch.Tensor, context: torch.Tensor, *, do_cfg: bool = True,
            cfg_scale: float = 7.5) -> torch.Tensor:
    """Functional form of the loop body of models/diffusion.py:223-236 (sampler._set_inference_steps first)."""
    b, _, h, w = latent.shape
    loop = DenoiseLoop(unet, sampler, b, h, w, do_cfg=do_cfg, cfg_scale=cfg_scale, context_len=context.shape[1],
                       context_batch=context.shape[0], device=latent.device)
    return loop.run(latent, context)


@torch.no_grad()
def img2img(unet: UNet, sampler, encoded_img: torch.Tensor, noise: torch.Tensor, context: torch.Tensor, strength: float, *,
            do_cfg: bool = True, cfg_scale: float = 7.5) -> torch.Tensor:
    """Image-to-image loop of models/diffusion.py:204-236 after the VAE encode: ``set_strength`` shortens the grid, the
    encoded image is noised to its first timestep (forward_process), then the ordinary loop runs."""
    sampler.set_strength(strength=strength)
    latent, _ = sampler.forward_process(encoded_img, sampler.timesteps[0].unsqueeze(0), noise)
    return denoise(unet, sampler, latent, context, do_cfg=do_cfg, cfg_scale=cfg_scale)


@torch.no_grad()
def inpaint(unet: UNet, sampler, latent: torch.Tensor, context: torch.Tensor, encoded_img: torch.Tensor, mask: torch.Tensor, *,
            do_cfg: bool = True, cfg_scale: float = 7.5) -> torch.Tensor:
    """Inpainting loop of models/diffusion.py:379-398 (``latent`` = the already masked/noised start of :365-369; context rows
    [cond ; uncond]); one CUDA-graph replay per step like ``denoise``."""
    b, _, h, w = latent.shape
    loop = DenoiseLoop(unet, sampler, b, h, w, do_cfg=do_cfg, cfg_scale=cfg_scale, context_len=context.shape[1],
                       context_batch=context.shape[0], device=latent.device)
    loop.set_inpaint(encoded_img, mask)
    return loop.run(latent, context)


@torch.no_grad()
def one_step(unet: UNet, sampler, latent: torch.Tensor, context: torch.Tensor) -> torch.Tensor:
    """SwiftBrush one-step generation (models/diffusion.py:106-113): t = sampler.timesteps[0], no CFG,
    context batch 1 broadcast, x0 = (x - sigma_T*eps)/alpha_T."""
    t = sampler.timesteps[0].to(latent.device).unsqueeze(0)
    pred = unet(latent, t, context)
    return x0_from_eps(latent, pred)
