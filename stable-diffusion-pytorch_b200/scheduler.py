"""DDIM / DDPM / DPM-Solver++(2M) samplers for the B200 denoising path.

Drop-in for the reference's ``models/scheduler`` classes (reference:
models/scheduler/ddim.py:7-96, models/scheduler/ddpm.py:10-89): same
constructor arguments, same attributes (``timesteps``, ``alphas_hat``,
``noise_step``, ``inference_steps``, ``prediction_type``) and same method
names.  ``step`` is an alias of ``reverse_process``.  ``DPMSolverSampler`` adds the
multistep DPM-Solver++ of order 2 (diffusers' ``DPMSolverMultistepScheduler``,
"DPM++ 2M") with DDIM's constructor, grid and calling convention.

Split of responsibilities
  * timestep / index bookkeeping stays on the host and is bit-exact with the
    reference (it is produced by the same numpy/torch integer expressions);
  * the latent update runs as ONE fused sm_100a kernel per step
    (csrc/sampler_kernels.cu) that looks its per-timestep scalars up in a small
    device-resident coefficient table, so there is no host sync in the loop
    (the reference does three per step: ddim.py:64,66,74);
  * there is NO CPU implementation of the update here: a CPU tensor or a
    missing extension raises.
"""
from __future__ import annotations

import json
import os
from typing import Optional

import numpy as np
import torch

from . import _lib

# coefficient-table column indices (must match csrc/sampler_kernels.cu)
COEF_COLS = 8
_C_S1, _C_S2, _C_SQRT_PREV, _C_DIR, _C_STD = 0, 1, 2, 3, 4          # DDIM
_P_INV_SQRT_CUR, _P_EPS_COEF, _P_STD = 0, 1, 2                      # DDPM
_F_SQRT_A, _F_SQRT_1MA = 5, 6                                       # forward_process (all)
_D_A, _D_B, _D_C, _D_ORDER2 = 2, 3, 4, 7                            # DPM-Solver++(2M); columns 0-1 are DDIM's

PRED_EPS, PRED_V = 0, 1


def _beta_tables(noise_step, beta_start, beta_end, use_cosine_schedule, device, explicit_f32):
    """Schedule tables (reference: ddim.py:9-23 / ddpm.py:12-26).

    The values have to be bit-identical to the reference's, so they are built
    from the same torch primitives (linspace -> square -> cumprod, fp32)."""
    kw = dict(dtype=torch.float32) if explicit_f32 else {}
    betas = torch.linspace(beta_start ** 0.5, beta_end ** 0.5, noise_step, device=device, **kw) ** 2
    alphas = 1.0 - betas
    alphas_hat = torch.cumprod(alphas, dim=0)
    if use_cosine_schedule:
        s = 0.008

        def f_t(t):
            return np.cos((t / noise_step + s) / (1 + s) * np.pi / 2) ** 2

        alphas_hat = f_t(torch.arange(0, noise_step + 1)) / f_t(0)
        alphas_hat = alphas_hat.to(device)
        betas = torch.clip(1 - alphas_hat[1:] / alphas_hat[:-1], 0, 0.999)
        alphas = torch.clip(1. - betas, 0, 0.999)
        alphas_hat = torch.clip(alphas_hat[1:], 0, 0.999)
    return betas, alphas, alphas_hat


class _SamplerBase:
    _timestep_offset = 0      # DDIM grids carry a +1 (ddim.py:31), DDPM grids do not (ddpm.py:32)
    _explicit_f32 = True

    def _init_tables(self, noise_step, beta_start, beta_end, use_cosine_schedule, device):
        self.betas, self.alphas, self.alphas_hat = _beta_tables(
            noise_step, beta_start, beta_end, use_cosine_schedule, device, self._explicit_f32)
        self.noise_step = noise_step
        self.timesteps = torch.from_numpy(np.arange(0, noise_step)[::-1].copy()).to(device)
        self._coef_cache = {}

    # ---- host bookkeeping (bit-exact with the reference) -----------------
    def _set_inference_steps(self, inference_steps=50):
        """reference: ddim.py:28-31 / ddpm.py:29-32."""
        self.inference_steps = inference_steps
        stride = self.noise_step // self.inference_steps
        grid = np.arange(0, self.inference_steps) * stride + self._timestep_offset
        self.timesteps = torch.from_numpy(grid.round()[::-1].copy().astype(np.int64))

    def _get_prev_timestep(self, timestep):
        """reference: ddim.py:37-39 / ddpm.py:38-40."""
        return timestep - self.noise_step // self.inference_steps

    def set_strength(self, strength: float = 0.8):
        """reference: ddim.py:41-43 / ddpm.py:42-44."""
        start_t = self.inference_steps - int(self.inference_steps * strength)
        self.timesteps = self.timesteps[start_t:]

    # ---- device coefficient tables -----------------------------------------
    def _host_tables(self):
        return (self.alphas.detach().to("cpu", torch.float32),
                self.alphas_hat.detach().to("cpu", torch.float32))

    def _stride(self):
        if not hasattr(self, "inference_steps"):
            # the reference raises AttributeError here too (ddpm.py:39)
            raise AttributeError(f"{type(self).__name__} has no inference_steps; call _set_inference_steps first")
        return self.noise_step // self.inference_steps

    def _table_key(self):
        return ()

    def _coef_table(self, device, eta: float) -> torch.Tensor:
        key = (str(device), self._stride(), float(eta), self.prediction_type if hasattr(self, "prediction_type") else "") + self._table_key()
        tab = self._coef_cache.get(key)
        if tab is None:
            tab = self._build_coef(float(eta)).to(device).contiguous()
            self._coef_cache = {key: tab}      # one live table; rebuilt when the step grid changes
        return tab

    def coefficient_table(self, eta: float = 0.0) -> torch.Tensor:
        """Host copy of the per-timestep scalar table the kernel reads ([noise_step, 8] fp32)."""
        return self._build_coef(float(eta))

    @staticmethod
    def _x0_cols(tab, a_hat):
        """DDIM's x0-prediction scalars s1 = fp32((1 - a_t)**0.5), s2 = fp32(a_t**0.5), a_t the python double of the fp32
        table entry (ddim.py:64-66, .item())."""
        a_list = a_hat.tolist()
        tab[:, _C_S1] = torch.tensor([(1 - a) ** 0.5 for a in a_list], dtype=torch.float64).to(torch.float32)
        tab[:, _C_S2] = torch.tensor([a ** 0.5 for a in a_list], dtype=torch.float64).to(torch.float32)

    def _forward_cols(self, tab, a_hat):
        tab[:, _F_SQRT_A] = torch.sqrt(a_hat)
        tab[:, _F_SQRT_1MA] = torch.sqrt(1 - a_hat)

    # ---- shared device entry points ------------------------------------
    @staticmethod
    def _check_cuda(x: torch.Tensor, what: str):
        if not isinstance(x, torch.Tensor) or not x.is_cuda:
            raise RuntimeError(
                f"{what}: the B200 sampler only runs on CUDA tensors (got {getattr(x, 'device', type(x))}); "
                "there is no CPU fallback")

    @staticmethod
    def _timestep_args(timestep, device):
        """-> (device_ptr_or_0, host_value, keepalive)"""
        if isinstance(timestep, torch.Tensor):
            if timestep.numel() != 1:
                raise ValueError("reverse_process takes a single timestep (the reference calls .item() on it, ddim.py:64)")
            if timestep.is_cuda:
                t = timestep.reshape(1).to(torch.int64)
                return t.data_ptr(), 0, t
            return 0, int(timestep.reshape(()).item()), None
        return 0, int(timestep), None

    def forward_process(self, x_0: torch.Tensor, timestep, noise: Optional[torch.Tensor] = None):
        """x_t = sqrt(a_hat[t]) * x_0 + sqrt(1 - a_hat[t]) * noise, per-sample t (n,).

        reference: ddim.py:46-55 / ddpm.py:47-57."""
        self._check_cuda(x_0, "forward_process")
        x0 = x_0.contiguous().float()
        if noise is None:
            noise = torch.randn(x0.shape, dtype=x0.dtype, device=x0.device)
        nz = noise.to(x0.device, torch.float32).contiguous()
        if not isinstance(timestep, torch.Tensor):
            timestep = torch.tensor([int(timestep)], dtype=torch.int64)
        t = timestep.reshape(-1).to(x0.device, torch.int64)
        n = x0.shape[0]
        if t.numel() not in (1, n):
            raise RuntimeError(f"forward_process: {t.numel()} timesteps for batch {n}")
        if t.numel() == 1 and n > 1:
            t = t.expand(n).contiguous()
        tab = self._forward_table(x0.device)
        out = torch.empty_like(x0)
        with torch.cuda.device(x0.device):              # launches go to the tensor's device, not the caller's current one
            _lib.check(_lib.lib().sdk_forward_process(
                x0.data_ptr(), nz.data_ptr(), out.data_ptr(), n, x0.numel() // max(n, 1),
                tab.data_ptr(), self.noise_step, t.data_ptr(), _lib.current_stream(x0.device)))
        return out, noise

    def _forward_table(self, device):
        key = ("fwd", str(device))
        tab = self._coef_cache.get(key)
        if tab is None:
            host = torch.zeros(self.noise_step, COEF_COLS, dtype=torch.float32)
            self._forward_cols(host, self._host_tables()[1])
            tab = host.to(device)
            self._coef_cache[key] = tab
        return tab


    def inpaint_step(self, x_t: torch.Tensor, timestep, model_output: torch.Tensor, encoded_img: torch.Tensor, mask: torch.Tensor,
                     *, cfg_scale: Optional[float] = None, out: Optional[torch.Tensor] = None,
                     noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Everything the inpainting loop does after the UNet call (models/diffusion.py:387-398), fused:

            cond, uncond = model_output.chunk(2); pred = cfg_scale * (cond - uncond) + cond      (only with cfg_scale)
            noised, _ = forward_process(encoded_img, timestep, pred)
            x = torch.where(~mask, noised, x_t)                   # mask: (1, 1, h, w) or (h, w) bool, True = repaint
            return reverse_process(x, timestep, pred)

        Note the inpaint loop's own CFG convention: rows ordered [cond ; uncond] and pred = s*(c-u) + c.
        Every sampler (the reference's inpaint takes sampler='ddim' or 'ddpm', diffusion.py:314-320) launches its own update in
        ``_inpaint_update``; with DDPM the update draws fresh N(0,1) noise from torch's global generator like ddpm.py:80 unless
        ``noise`` is given, and DPM-Solver++ reads and replaces its history like ``reverse_process``."""
        self._check_cuda(x_t, "inpaint_step")
        x = x_t.contiguous().float()
        b, ch, h, w = x.shape
        mo = model_output.to(x.device, torch.float32).contiguous()
        n = x.numel()
        if cfg_scale is None:
            if mo.shape != x.shape:
                raise RuntimeError(f"model_output {tuple(mo.shape)} vs x_t {tuple(x.shape)}")
            eps_c, eps_u, scale = mo.data_ptr(), 0, 0.0
        else:
            if mo.shape[0] != 2 * b or mo.shape[1:] != x.shape[1:]:
                raise RuntimeError(f"CFG model_output must be (2B, ...) = {(2 * b,) + tuple(x.shape[1:])}, got {tuple(mo.shape)}")
            eps_c, eps_u, scale = mo.data_ptr(), mo.data_ptr() + n * 4, float(cfg_scale)
        orig = encoded_img.to(x.device, torch.float32).contiguous()
        if orig.shape[0] not in (1, b) or tuple(orig.shape[1:]) != (ch, h, w):
            raise RuntimeError(f"encoded_img {tuple(orig.shape)} does not broadcast against x_t {tuple(x.shape)}")
        if mask.numel() != h * w:
            raise RuntimeError(f"mask must hold one value per latent pixel ({h}x{w}), got {tuple(mask.shape)}")
        m8 = mask.to(x.device).reshape(h * w).ne(0).to(torch.uint8).contiguous()
        tab = self._coef_table(x.device, 0.0)
        t_ptr, t_host, keep = self._timestep_args(timestep, x.device)
        res = torch.empty_like(x) if out is None else out
        if n == 0:
            return res
        with torch.cuda.device(x.device):              # launches go to the tensor's device, not the caller's current one
            self._inpaint_update(x_t, x, eps_c, eps_u, scale, orig, m8, res, tab, t_ptr, t_host, noise)
        return res


class DDIMSampler(_SamplerBase):
    """reference: models/scheduler/ddim.py:7-96."""
    _timestep_offset = 1

    def __init__(self, noise_step: int = 1000, beta_start: float = 0.00085, beta_end: float = 0.012,
                 use_cosine_schedule: bool = False, device: str = 'cpu', prediction_type: str = "epsilon"):
        self._init_tables(noise_step, beta_start, beta_end, use_cosine_schedule, device)
        self.inference_steps = self.noise_step
        self.prediction_type = prediction_type

    def _sample_timestep(self, n, device):
        return torch.randint(low=0, high=self.noise_step, size=(n,), device=device)

    def _build_coef(self, eta: float) -> torch.Tensor:
        """Per-timestep scalars of the DDIM update, laid out [noise_step, 8].

        Mirrors the scalar arithmetic of ddim.py:60-81 for every t at once:
          s1 = fp32( (1 - a_t)**0.5 ), s2 = fp32( a_t**0.5 ) with a_t the python
          double of the fp32 table entry (ddim.py:64-66, .item());
          a_prev = alphas_hat[t - stride] or exactly 1.0 when t - stride < 0 (:74);
          variance uses self.alphas[t] (the reference's quirk, :73-76);
          std = sqrt(eta * variance); dir = sqrt(1 - a_prev - std**2) in fp32 (:77,79)."""
        alphas, a_hat = self._host_tables()
        T, stride = self.noise_step, self._stride()
        tab = torch.zeros(T, COEF_COLS, dtype=torch.float32)
        self._x0_cols(tab, a_hat)
        prev_idx = torch.arange(T) - stride
        a_prev = torch.where(prev_idx >= 0, a_hat[prev_idx.clamp(min=0)], torch.tensor(1.0))
        variance = (1 - a_prev) / (1 - alphas) * (1 - alphas / a_prev)
        std = torch.sqrt(eta * variance)
        tab[:, _C_SQRT_PREV] = torch.sqrt(a_prev)
        tab[:, _C_DIR] = torch.sqrt(1 - a_prev - std ** 2)
        tab[:, _C_STD] = std
        self._forward_cols(tab, a_hat)
        return tab

    def _inpaint_update(self, x_t, x, eps_c, eps_u, scale, orig, m8, res, tab, t_ptr, t_host, noise):
        b, ch, h, w = x.shape
        _lib.check(_lib.lib().sdk_ddim_inpaint_step(
            x.data_ptr(), eps_c, eps_u, scale, orig.data_ptr(), orig.shape[0], m8.data_ptr(), res.data_ptr(), b, ch, h * w,
            tab.data_ptr(), self.noise_step, t_ptr, t_host, PRED_V if self.prediction_type == "v_prediction" else PRED_EPS,
            _lib.current_stream(x.device)))

    def reverse_process(self, x_t: torch.Tensor, timestep, model_output: torch.Tensor, eta: float = 0.0,
                        *, cfg_scale: Optional[float] = None) -> torch.Tensor:
        """One DDIM update (reference: ddim.py:58-87).

        With ``cfg_scale`` given, ``model_output`` is the (2B, ...) UNet output
        ordered [uncond ; cond] and the guidance blend u + s*(c-u)
        (reference: models/diffusion.py:233-235) is fused into the same kernel."""
        self._check_cuda(x_t, "reverse_process")
        if self.prediction_type not in ("epsilon", "v_prediction"):
            raise ValueError(f"unknown prediction_type {self.prediction_type!r}")
        x = x_t.contiguous().float()
        mo = model_output.to(x.device, torch.float32).contiguous()
        n = x.numel()
        if cfg_scale is None:
            if mo.shape != x.shape:
                raise RuntimeError(f"model_output {tuple(mo.shape)} vs x_t {tuple(x.shape)}")
            eps_u, eps_c, scale = mo.data_ptr(), 0, 0.0
        else:
            if mo.shape[0] != 2 * x.shape[0] or mo.shape[1:] != x.shape[1:]:
                raise RuntimeError(f"CFG model_output must be (2B, ...) = {(2 * x.shape[0],) + tuple(x.shape[1:])}, got {tuple(mo.shape)}")
            eps_u, eps_c, scale = mo.data_ptr(), mo.data_ptr() + n * 4, float(cfg_scale)
        noise = None
        if eta > 0:
            noise = torch.randn_like(x)              # same RNG draw as ddim.py:84
        tab = self._coef_table(x.device, eta)
        t_ptr, t_host, keep = self._timestep_args(timestep, x.device)
        out = torch.empty_like(x)
        if n == 0:
            return out
        with torch.cuda.device(x.device):              # launches go to the tensor's device, not the caller's current one
            _lib.check(_lib.lib().sdk_ddim_step(
                x.data_ptr(), eps_u, eps_c, scale, noise.data_ptr() if noise is not None else 0,
                out.data_ptr(), n, tab.data_ptr(), self.noise_step, t_ptr, t_host,
                PRED_V if self.prediction_type == "v_prediction" else PRED_EPS,
                _lib.current_stream(x.device)))
        return out

    step = reverse_process

    @staticmethod
    def from_config(cfg_path: str, use_cosine_schedule: bool = False, device: str = 'cpu'):
        """reference: ddim.py:89-96 (reads <cfg_path>/scheduler_config.json)."""
        with open(os.path.join(cfg_path, "scheduler_config.json"), 'r') as f:
            config = json.load(f)
        return DDIMSampler(noise_step=config["num_train_timesteps"], beta_start=config["beta_start"],
                           beta_end=config["beta_end"], use_cosine_schedule=use_cosine_schedule, device=device,
                           prediction_type=config.get("prediction_type", "epsilon"))


class DDPMSampler(_SamplerBase):
    """reference: models/scheduler/ddpm.py:10-89.

    ``inference_steps`` is deliberately NOT set by the constructor (ddpm.py:11-27):
    like the reference, ``reverse_process`` before ``_set_inference_steps`` raises
    AttributeError."""
    _timestep_offset = 0
    _explicit_f32 = False     # ddpm.py:12 builds linspace in the default dtype
    prediction_type = "epsilon"

    def __init__(self, noise_step: int = 1000, beta_start: float = 0.00085, beta_end: float = 0.0120,
                 use_cosine_schedule: bool = False, device: str = 'cpu'):
        self._init_tables(noise_step, beta_start, beta_end, use_cosine_schedule, device)

    def _sample_timestep(self, n):
        return torch.randint(low=0, high=self.noise_step, size=(n,))

    def _build_coef(self, eta: float = 0.0) -> torch.Tensor:
        """Per-timestep scalars of the ancestral update (ddpm.py:62-82), fp32 tensor math:
          cur_a = clip(a_hat[t] / a_prev, 0, 0.999); inv = 1/sqrt(cur_a);
          ce = (1 - cur_a)/sqrt(1 - a_hat[t]);
          std = sqrt(clamp((1 - a_prev)/(1 - a_hat[t]) * (1 - cur_a), 1e-20)) for t > 0, 0 for t == 0."""
        _, a_hat = self._host_tables()
        T, stride = self.noise_step, self._stride()
        tab = torch.zeros(T, COEF_COLS, dtype=torch.float32)
        prev_idx = torch.arange(T) - stride
        a_prev = torch.where(prev_idx >= 0, a_hat[prev_idx.clamp(min=0)], torch.tensor(1.0))
        cur_a = torch.clip(a_hat / a_prev, 0, 0.999)
        cur_b = 1 - cur_a
        tab[:, _P_INV_SQRT_CUR] = 1 / torch.sqrt(cur_a)
        tab[:, _P_EPS_COEF] = (1 - cur_a) / torch.sqrt(1 - a_hat)
        std = torch.sqrt(torch.clamp((1 - a_prev) / (1 - a_hat) * cur_b, min=1e-20))
        std[0] = 0.0
        tab[:, _P_STD] = std
        self._forward_cols(tab, a_hat)
        return tab

    def _inpaint_update(self, x_t, x, eps_c, eps_u, scale, orig, m8, res, tab, t_ptr, t_host, noise):
        b, ch, h, w = x.shape
        if noise is None:
            noise = torch.randn(x_t.shape, dtype=x_t.dtype, device=x_t.device)
        nz = noise.to(x.device, torch.float32).contiguous()
        _lib.check(_lib.lib().sdk_ddpm_inpaint_step(
            x.data_ptr(), eps_c, eps_u, scale, orig.data_ptr(), orig.shape[0], m8.data_ptr(), nz.data_ptr(), res.data_ptr(), b, ch,
            h * w, tab.data_ptr(), self.noise_step, t_ptr, t_host, _lib.current_stream(x.device)))

    def reverse_process(self, x_t: torch.Tensor, timestep, model_output: torch.Tensor,
                        *, cfg_scale: Optional[float] = None, noise: Optional[torch.Tensor] = None) -> torch.Tensor:
        """One ancestral DDPM update (reference: ddpm.py:62-82).

        Fresh N(0,1) noise is drawn from torch's global generator on x_t's device on every
        call, including t == 0 where it is multiplied by zero, exactly like ddpm.py:80.
        ``noise`` lets a data-parallel caller pass its slice of a full-batch draw."""
        self._check_cuda(x_t, "reverse_process")
        x = x_t.contiguous().float()
        mo = model_output.to(x.device, torch.float32).contiguous()
        n = x.numel()
        if cfg_scale is None:
            if mo.shape != x.shape:
                raise RuntimeError(f"model_output {tuple(mo.shape)} vs x_t {tuple(x.shape)}")
            eps_u, eps_c, scale = mo.data_ptr(), 0, 0.0
        else:
            if mo.shape[0] != 2 * x.shape[0] or mo.shape[1:] != x.shape[1:]:
                raise RuntimeError("CFG model_output must be (2B, ...)")
            eps_u, eps_c, scale = mo.data_ptr(), mo.data_ptr() + n * 4, float(cfg_scale)
        tab = self._coef_table(x.device, 0.0)
        if noise is None:
            noise = torch.randn(x_t.shape, dtype=x_t.dtype, device=x_t.device)
        nz = noise.to(x.device, torch.float32).contiguous()
        t_ptr, t_host, keep = self._timestep_args(timestep, x.device)
        out = torch.empty_like(x)
        if n == 0:
            return out
        with torch.cuda.device(x.device):              # launches go to the tensor's device, not the caller's current one
            _lib.check(_lib.lib().sdk_ddpm_step(
                x.data_ptr(), eps_u, eps_c, scale, nz.data_ptr(), out.data_ptr(), n,
                tab.data_ptr(), self.noise_step, t_ptr, t_host, _lib.current_stream(x.device)))
        return out

    step = reverse_process

    @staticmethod
    def from_config(cfg_path: str, use_cosine_schedule: bool = False, device: str = 'cpu'):
        """reference: ddpm.py:84-89.  The reference forwards ``prediction_type`` to a constructor
        that does not take it and crashes; here the key is read and ignored (DDPM is eps-only)."""
        with open(os.path.join(cfg_path, "scheduler_config.json"), 'r') as f:
            config = json.load(f)
        return DDPMSampler(noise_step=config["num_train_timesteps"], beta_start=config["beta_start"],
                           beta_end=config["beta_end"], use_cosine_schedule=use_cosine_schedule, device=device)


def dpmpp_coefficients(a_path, schedule_steps: Optional[int] = None) -> np.ndarray:
    """float64 [N, 4] = (A, B, C, order-2 flag) of N DPM-Solver++(2M) steps along a path of N + 1 alpha-bar values.

    diffusers' DPMSolverMultistepScheduler with algorithm_type="dpmsolver++", solver_type="midpoint": with
    alpha = sqrt(a), sigma = sqrt(1 - a), lambda = log(alpha) - log(sigma) and h = lambda_t - lambda_s for step s -> t,
        x_t = A*x_s + B*m0 + C*(m0 - m1),   A = sigma_t/sigma_s,  B = -alpha_t*expm1(-h),  C = B/(2r),
    r = (lambda_s - lambda_prev)/h, m0 / m1 the x0 predictions at s and at the step before.  A step to a = 1 (sigma = 0, the
    last step of a sampling grid) has A = 0, B = 1: it returns m0.  Steps are first order (C = 0, flag 0) on the first step,
    the last step, and the second-to-last step when the schedule has fewer than 15 steps.  ``schedule_steps`` is the length of
    the whole schedule (default N): a path that is the tail of a longer schedule (img2img strength) counts the whole schedule,
    as diffusers does when it starts a pipeline part-way through its timesteps."""
    a = np.asarray(a_path, dtype=np.float64)
    n = len(a) - 1
    short = (n if schedule_steps is None else schedule_steps) < 15
    alpha, sigma = np.sqrt(a), np.sqrt(1.0 - a)
    with np.errstate(divide="ignore"):
        lam = np.log(alpha) - np.log(sigma)                  # +inf where sigma == 0
    out = np.zeros((n, 4), dtype=np.float64)
    for i in range(n):
        if sigma[i + 1] == 0.0:
            out[i, 0], out[i, 1] = 0.0, 1.0
        else:
            h = lam[i + 1] - lam[i]
            out[i, 0] = sigma[i + 1] / sigma[i]
            out[i, 1] = -alpha[i + 1] * np.expm1(-h)
        order2 = 0 < i < n - 1 and not (i == n - 2 and short)
        if order2:
            r = (lam[i] - lam[i - 1]) / (lam[i + 1] - lam[i])
            out[i, 2] = out[i, 1] / (2.0 * r)
            out[i, 3] = 1.0
    return out


class DPMSolverSampler(_SamplerBase):
    """Multistep DPM-Solver++ of order 2 ("DPM++ 2M"; diffusers' DPMSolverMultistepScheduler defaults: dpmsolver++,
    midpoint, lower_order_final, final sigma zero) on DDIM's timestep grid, commonly run at 20-25 steps.

    Same constructor, ``from_config``, grid (bit for bit), ``set_strength`` and ``forward_process`` as ``DDIMSampler``; the
    final step goes to alpha-bar = 1 and returns the x0 prediction.  The update needs the previous step's x0 prediction: the
    sampler keeps it in a device tensor per shape and device.  A host flag says whether that history belongs to the current
    sequence; ``_set_inference_steps``, ``set_strength``, ``reset()`` and a change of shape or device clear it, so a sequence
    that starts anywhere takes a first-order step instead of reading stale history.  The coefficient table depends on the
    whole grid; a timestep off the grid poisons the update with NaN, like an out-of-range one."""
    _timestep_offset = 1

    def __init__(self, noise_step: int = 1000, beta_start: float = 0.00085, beta_end: float = 0.012,
                 use_cosine_schedule: bool = False, device: str = 'cpu', prediction_type: str = "epsilon"):
        self._init_tables(noise_step, beta_start, beta_end, use_cosine_schedule, device)
        self.inference_steps = self.noise_step
        self.prediction_type = prediction_type
        self._hist, self._hist_valid = None, False

    def _sample_timestep(self, n, device):
        return torch.randint(low=0, high=self.noise_step, size=(n,), device=device)

    def reset(self):
        """Forget the history: the next step is first order."""
        self._hist_valid = False

    def _set_inference_steps(self, inference_steps=50):
        super()._set_inference_steps(inference_steps)
        self.reset()

    def set_strength(self, strength: float = 0.8):
        super().set_strength(strength)
        self.reset()

    def _history(self, x: torch.Tensor):
        """-> (history tensor for x's shape and device, hist_valid for this step).  The caller marks the history valid
        (``_hist_valid = True``) once the step that fills it has been launched."""
        if self._hist is None or self._hist.shape != x.shape or self._hist.device != x.device:
            with torch.inference_mode(False), torch.no_grad():
                self._hist = torch.empty_like(x)
            self._hist_valid = False
        return self._hist, int(self._hist_valid)

    def _inpaint_update(self, x_t, x, eps_c, eps_u, scale, orig, m8, res, tab, t_ptr, t_host, noise):
        b, ch, h, w = x.shape
        hist, valid = self._history(x)
        _lib.check(_lib.lib().sdk_dpmpp_inpaint_step(
            x.data_ptr(), eps_c, eps_u, scale, orig.data_ptr(), orig.shape[0], m8.data_ptr(), res.data_ptr(), b, ch, h * w,
            tab.data_ptr(), self.noise_step, t_ptr, t_host, PRED_V if self.prediction_type == "v_prediction" else PRED_EPS,
            hist.data_ptr(), valid, _lib.current_stream(x.device)))
        self._hist_valid = True

    def _table_key(self):
        return (self.inference_steps,) + tuple(self.timesteps.tolist())

    def _build_coef(self, eta: float = 0.0) -> torch.Tensor:
        """[noise_step, 8] fp32: columns 0-1 and 5-6 are DDIM's (bit for bit); on the rows of the current grid t_0 > ... > t_N-1,
        columns 2-4 = A, B, C and 7 = the order-2 flag of ``dpmpp_coefficients`` along alpha-bar[t_0], ..., alpha-bar[t_N-1], 1.0,
        computed in float64 and rounded to fp32 once; the lower-order-final rule counts the whole ``inference_steps`` schedule, so
        a ``set_strength`` tail keeps the flags it has in the full grid except on its first row.  Other rows are NaN in columns 2-4."""
        _, a_hat = self._host_tables()
        T = self.noise_step
        tab = torch.zeros(T, COEF_COLS, dtype=torch.float32)
        self._x0_cols(tab, a_hat)
        self._forward_cols(tab, a_hat)
        tab[:, _D_A:_D_C + 1] = float("nan")
        grid = [int(t) for t in self.timesteps.tolist()]
        if any(t < 0 or t >= T for t in grid):
            raise ValueError(f"timestep grid {grid} outside [0, {T})")
        a_path = a_hat.to(torch.float64)[grid].tolist() + [1.0]
        k = torch.from_numpy(dpmpp_coefficients(a_path, self.inference_steps)).to(torch.float32)
        rows = torch.tensor(grid, dtype=torch.int64)
        tab[rows, _D_A], tab[rows, _D_B], tab[rows, _D_C], tab[rows, _D_ORDER2] = k[:, 0], k[:, 1], k[:, 2], k[:, 3]
        return tab

    def reverse_process(self, x_t: torch.Tensor, timestep, model_output: torch.Tensor, *,
                        cfg_scale: Optional[float] = None) -> torch.Tensor:
        """One DPM-Solver++(2M) update from ``timestep`` to the next point of the grid (alpha-bar = 1 after the last).

        Calling convention of ``DDIMSampler.reverse_process``: host or device timestep, no host sync, and with ``cfg_scale``
        given ``model_output`` is the (2B, ...) UNet output ordered [uncond ; cond], blended as u + s*(c-u) in the same kernel.
        Reads the previous step's x0 prediction from the sampler's history and replaces it with this step's."""
        self._check_cuda(x_t, "reverse_process")
        if self.prediction_type not in ("epsilon", "v_prediction"):
            raise ValueError(f"unknown prediction_type {self.prediction_type!r}")
        x = x_t.contiguous().float()
        mo = model_output.to(x.device, torch.float32).contiguous()
        n = x.numel()
        if cfg_scale is None:
            if mo.shape != x.shape:
                raise RuntimeError(f"model_output {tuple(mo.shape)} vs x_t {tuple(x.shape)}")
            eps_u, eps_c, scale = mo.data_ptr(), 0, 0.0
        else:
            if mo.shape[0] != 2 * x.shape[0] or mo.shape[1:] != x.shape[1:]:
                raise RuntimeError(f"CFG model_output must be (2B, ...) = {(2 * x.shape[0],) + tuple(x.shape[1:])}, got {tuple(mo.shape)}")
            eps_u, eps_c, scale = mo.data_ptr(), mo.data_ptr() + n * 4, float(cfg_scale)
        tab = self._coef_table(x.device, 0.0)
        t_ptr, t_host, keep = self._timestep_args(timestep, x.device)
        out = torch.empty_like(x)
        if n == 0:
            return out
        hist, valid = self._history(x)
        with torch.cuda.device(x.device):              # launches go to the tensor's device, not the caller's current one
            _lib.check(_lib.lib().sdk_dpmpp_step(
                x.data_ptr(), eps_u, eps_c, scale, hist.data_ptr(), valid, out.data_ptr(), n, tab.data_ptr(), self.noise_step,
                t_ptr, t_host, PRED_V if self.prediction_type == "v_prediction" else PRED_EPS, _lib.current_stream(x.device)))
        self._hist_valid = True
        return out

    step = reverse_process

    @staticmethod
    def from_config(cfg_path: str, use_cosine_schedule: bool = False, device: str = 'cpu'):
        """Reads <cfg_path>/scheduler_config.json like DDIMSampler.from_config."""
        with open(os.path.join(cfg_path, "scheduler_config.json"), 'r') as f:
            config = json.load(f)
        return DPMSolverSampler(noise_step=config["num_train_timesteps"], beta_start=config["beta_start"],
                                beta_end=config["beta_end"], use_cosine_schedule=use_cosine_schedule, device=device,
                                prediction_type=config.get("prediction_type", "epsilon"))


def x0_from_eps(latent: torch.Tensor, pred_noise: torch.Tensor, alpha_T: float = 0.0047 ** 0.5,
                sigma_T: float = (1 - 0.0047) ** 0.5) -> torch.Tensor:
    """One-step (SwiftBrush) update x0 = (x - sigma_T*eps)/alpha_T (reference: models/diffusion.py:111-113)."""
    _SamplerBase._check_cuda(latent, "x0_from_eps")
    x = latent.contiguous().float()
    e = pred_noise.to(x.device, torch.float32).contiguous()
    if e.shape != x.shape:
        raise RuntimeError(f"pred_noise {tuple(e.shape)} vs latent {tuple(x.shape)}")
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):              # launches go to the tensor's device, not the caller's current one
        _lib.check(_lib.lib().sdk_x0_from_eps(x.data_ptr(), e.data_ptr(), float(sigma_T), float(alpha_T),
                                              out.data_ptr(), x.numel(), _lib.current_stream(x.device)))
    return out
