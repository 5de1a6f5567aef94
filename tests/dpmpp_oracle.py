"""ORACLE (test infrastructure, not product code) for the DPM-Solver++(2M) sampler: the coefficients in float64, derived
from lambda = log(alpha/sigma) without the product's host code, and the update in numpy fp32 in the kernel's op order
with every rounding explicit (the style of oracle/sampler_oracle.py, which it builds on).

The method is diffusers' DPMSolverMultistepScheduler with algorithm_type="dpmsolver++", solver_order=2,
solver_type="midpoint", lower_order_final=True, final_sigmas_type="zero".  For a step s -> t with h = lambda_t - lambda_s and
h_prev = lambda_s - lambda_prev, data prediction m0 at s and m1 at the step before:

    x_t = (alpha_t/alpha_s) e^-h x_s + alpha_t (1 - e^-h) m0 + alpha_t (1 - e^-h) h/(2 h_prev) (m0 - m1)
"""
from __future__ import annotations

import numpy as np

from oracle import sampler_oracle as SO

F = np.float32


def dpmpp_coefficients(a_path, schedule_steps=None):
    """float64 [N, 4] (A, B, C, order-2 flag) for the N steps along the alpha-bar path a_path[0..N].  A step to alpha-bar 1
    (sigma 0) returns the data prediction: A = 0, B = 1.  First order on the first and last steps and, when the whole
    schedule (``schedule_steps``, default N; longer when the path is a strength-shortened tail) has fewer than 15 steps,
    on the second-to-last step (diffusers' lower_order_final with len(timesteps) of the full schedule)."""
    a = np.asarray(a_path, dtype=np.float64)
    n = len(a) - 1
    m = n if schedule_steps is None else schedule_steps
    out = np.zeros((n, 4))
    lam = [0.5 * (np.log(v) - np.log1p(-v)) if v < 1.0 else np.inf for v in a]
    for i in range(n):
        if a[i + 1] == 1.0:
            out[i, :2] = (0.0, 1.0)
        else:
            h = lam[i + 1] - lam[i]
            out[i, 0] = np.sqrt(a[i + 1] / a[i]) * np.exp(-h)
            out[i, 1] = np.sqrt(a[i + 1]) * (1.0 - np.exp(-h))
        first_order = i == 0 or i == n - 1 or (m < 15 and i == n - 2)
        if not first_order:
            h, h_prev = lam[i + 1] - lam[i], lam[i] - lam[i - 1]
            out[i, 2] = out[i, 1] * h / (2.0 * h_prev)
            out[i, 3] = 1.0
    return out


def dpmpp_reverse(x_t, t, model_output, hist, table, prediction_type="epsilon", hist_valid=True):
    """One update from the fp32 [T][8] table at timestep t -> (x', m0): m0 is what the kernel writes to the history.

    model_output is the (already CFG-blended) prediction.  Op order of dpmpp_step_kernel, one fp32 rounding per op:
      eps: m0 = (x - s1*e)/s2     v: m0 = s2*x - s1*e
      x'  = (A*x + B*m0) + C*(m0 - m1)      the C term only when column 7 is set and hist_valid"""
    x = np.asarray(x_t, F)
    e = np.asarray(model_output, F)
    T = table.shape[0]
    if not 0 <= t < T:
        nan = np.full(x.shape, np.nan, F)
        return nan, nan.copy()
    s1, s2, A, B, C, flag = (F(table[t, j]) for j in (0, 1, 2, 3, 4, 7))
    if prediction_type == "epsilon":
        m0 = ((x - (s1 * e).astype(F)).astype(F) / s2).astype(F)
    elif prediction_type == "v_prediction":
        m0 = ((s2 * x).astype(F) - (s1 * e).astype(F)).astype(F)
    else:
        raise ValueError(prediction_type)
    r = ((A * x).astype(F) + (B * m0).astype(F)).astype(F)
    if hist_valid and flag != 0:
        r = (r + (C * (m0 - np.asarray(hist, F)).astype(F)).astype(F)).astype(F)
    return r, m0


def dpmpp_inpaint_step(x_t, t, pred_2b, orig, mask, cfg_scale, a_hat, hist, table, prediction_type="epsilon", hist_valid=True):
    """The inpainting loop body of oracle/sampler_oracle.inpaint_step (inpaint CFG form, re-noise, mask select) with the
    DPM-Solver++(2M) update -> (x', m0)."""
    if cfg_scale is None:
        e = pred_2b.astype(F)
    else:
        c, u = np.split(pred_2b.astype(F), 2, axis=0)
        e = (F(cfg_scale) * (c - u)).astype(F) + c
    noised = SO.forward_process(np.broadcast_to(orig, e.shape).astype(F), np.array([t]), e, a_hat)
    x = np.where(mask[None, None].astype(bool), x_t.astype(F), noised)
    return dpmpp_reverse(x, t, e, hist, table, prediction_type, hist_valid)
