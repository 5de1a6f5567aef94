"""CPU suite for the DPM-Solver++(2M) sampler: its timestep grid, its coefficient table against an independent float64
derivation, the placement of the order-2 rows, the first-order and last-step special cases, the convergence order of the
method on a problem with a closed-form solution, and the absence of a CPU fallback."""
import numpy as np
import pytest
import torch

import dpmpp_oracle as DO
from stable_diffusion_pytorch_b200 import DDIMSampler, DPMSolverSampler
from stable_diffusion_pytorch_b200.scheduler import dpmpp_coefficients


def grids(n, strength=None):
    d, p = DDIMSampler(), DPMSolverSampler()
    for s in (d, p):
        s._set_inference_steps(n)
        if strength is not None:
            s.set_strength(strength)
    return d, p


@pytest.mark.parametrize("n,strength", [(10, None), (20, None), (50, None), (10, 0.6), (50, 0.6)])
def test_grid_equals_ddim(n, strength):
    d, p = grids(n, strength)
    assert p.timesteps.dtype == d.timesteps.dtype and torch.equal(p.timesteps, d.timesteps)


@pytest.mark.parametrize("n,strength,ptype", [(10, None, "epsilon"), (20, None, "v_prediction"), (50, None, "epsilon"),
                                              (10, 0.6, "epsilon"), (25, 0.6, "v_prediction")])
def test_table_matches_oracle(n, strength, ptype):
    d, p = grids(n, strength)
    p.prediction_type = d.prediction_type = ptype
    td, tp = d.coefficient_table(), p.coefficient_table()
    for col in (0, 1, 5, 6):                                  # x0 prediction and forward_process: DDIM's, bit for bit
        assert torch.equal(tp[:, col], td[:, col]), col
    grid = p.timesteps.tolist()
    a_path = p.alphas_hat.to(torch.float64)[grid].tolist() + [1.0]
    want = DO.dpmpp_coefficients(a_path, n)
    got = tp[grid][:, [2, 3, 4, 7]].numpy()
    np.testing.assert_allclose(got, want.astype(np.float32), rtol=2e-7, atol=0)
    assert np.array_equal(got[:, 3], want[:, 3])
    off = np.setdiff1d(np.arange(p.noise_step), grid)          # rows off the grid poison the update
    assert torch.isnan(tp[off][:, 2:5]).all() and (tp[off][:, 7] == 0).all()


@pytest.mark.parametrize("n", [2, 3, 10, 14, 15, 20, 50])
def test_order2_rows(n):
    p = DPMSolverSampler()
    p._set_inference_steps(n)
    flags = p.coefficient_table()[p.timesteps, 7].tolist()
    first = {0, n - 1} | ({n - 2} if n < 15 else set())
    assert flags == [0.0 if i in first else 1.0 for i in range(n)]
    p.set_strength(0.6)                                        # the shortened grid starts first order again
    m = len(p.timesteps)
    flags = p.coefficient_table()[p.timesteps, 7].tolist()
    first = {0, m - 1} | ({m - 2} if n < 15 else set())        # lower-order-final counts the whole n-step schedule
    assert flags == [0.0 if i in first else 1.0 for i in range(m)]


def test_strength_tail_counts_the_whole_schedule():
    """20 steps at strength 0.6 keep 12: the tail's second-to-last step stays second order, as in diffusers' img2img, which
    starts part-way through the full 20-step schedule."""
    p = DPMSolverSampler()
    p._set_inference_steps(20)
    p.set_strength(0.6)
    assert len(p.timesteps) == 12
    flags = p.coefficient_table()[p.timesteps, 7].tolist()
    assert flags == [0.0] + [1.0] * 10 + [0.0]


def test_table_cache_follows_the_grid():
    p = DPMSolverSampler()
    p._set_inference_steps(10)
    a = p._coef_table("cpu", 0.0)
    p.set_strength(0.6)
    b = p._coef_table("cpu", 0.0)
    assert b[p.timesteps[0], 7] == 0 and a[p.timesteps[0], 7] == 1      # same stride, different grid: rebuilt


def test_first_order_row_is_ddim():
    """DPM-Solver++(1) is DDIM with eta = 0: A*x + B*x0 == sqrt(a_prev)*x0 + sqrt(1 - a_prev)*eps, in float64."""
    rng = np.random.default_rng(0)
    a = np.sort(rng.uniform(0.01, 0.99, 12))
    k = dpmpp_coefficients(list(a) + [1.0])
    x, x0 = rng.standard_normal(64), rng.standard_normal(64)
    for i in range(len(a) - 1):
        A, B = k[i, 0], k[i, 1]
        eps = (x - np.sqrt(a[i]) * x0) / np.sqrt(1 - a[i])
        want = np.sqrt(a[i + 1]) * x0 + np.sqrt(1 - a[i + 1]) * eps
        got = A * x + B * x0
        assert np.max(np.abs(got - want)) <= 1e-12 * np.max(np.abs(want))


def test_last_row_returns_x0():
    p = DPMSolverSampler()
    p._set_inference_steps(20)
    row = p.coefficient_table()[p.timesteps[-1]]
    assert row[2] == 0 and row[3] == 1 and row[4] == 0 and row[7] == 0
    tab = p.coefficient_table().numpy()
    rng = np.random.default_rng(1)
    x, e, h = (rng.standard_normal(37).astype(np.float32) for _ in range(3))
    out, m0 = DO.dpmpp_reverse(x, int(p.timesteps[-1]), e, h, tab)
    assert np.array_equal(out, m0)


def _solve(lams, mu, s, x_start, order2):
    """float64 sampling along a path uniform in lambda with the exact eps-predictor of N(mu, s^2) data."""
    lam = np.asarray(lams)
    a = 1.0 / (1.0 + np.exp(-2.0 * lam))                      # alpha-bar from lambda = log(alpha/sigma)
    k = DO.dpmpp_coefficients(a)
    x, m1 = x_start.copy(), None
    for i in range(len(a) - 1):
        al, sg = np.sqrt(a[i]), np.sqrt(1 - a[i])
        eps = sg * (x - al * mu) / (al * al * s * s + sg * sg)
        m0 = (x - sg * eps) / al
        nx = k[i, 0] * x + k[i, 1] * m0
        if order2 and k[i, 3]:
            nx = nx + k[i, 2] * (m0 - m1)
        x, m1 = nx, m0
    return x, a[-1]


def test_convergence_order():
    """On N(mu, s^2) data the probability-flow ODE has the solution x = alpha*mu + sqrt(alpha^2 s^2 + sigma^2)*z, z constant.
    DPM-Solver++(2M) converges at second order, its first-order form (DDIM) at first order."""
    mu, s = 0.7, 0.5
    z = np.random.default_rng(2).standard_normal(256)

    def err(n, order2):
        lams = np.linspace(-3.0, 3.0, n + 1)
        a0 = 1.0 / (1.0 + np.exp(6.0))
        x_start = np.sqrt(a0) * mu + np.sqrt(a0 * s * s + 1 - a0) * z
        x, a1 = _solve(lams, mu, s, x_start, order2)
        exact = np.sqrt(a1) * mu + np.sqrt(a1 * s * s + 1 - a1) * z
        return np.linalg.norm(x - exact) / np.linalg.norm(exact)

    dpm = {n: err(n, True) for n in (20, 40, 80)}
    ddim = {n: err(n, False) for n in (40, 80)}
    print("rel err DPM++2M", dpm, "DDIM", ddim)
    assert dpm[40] / dpm[80] >= 3.5
    assert 1.8 <= ddim[40] / ddim[80] <= 2.2
    assert dpm[20] < ddim[80]


def test_cpu_tensor_raises():
    p = DPMSolverSampler()
    p._set_inference_steps(10)
    x = torch.zeros(1, 4, 8, 8)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        p.reverse_process(x, 901, x)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        p.inpaint_step(x, 901, x, x, torch.ones(8, 8, dtype=torch.bool))


def test_history_flag():
    """reset, _set_inference_steps and set_strength make the next step first order (hist_valid = 0)."""
    p = DPMSolverSampler()
    p._set_inference_steps(10)
    x = torch.zeros(2, 3)
    h, v = p._history(x)
    assert v == 0 and p._history(x) == (h, 0)                  # valid only once a step that fills it has been launched
    p._hist_valid = True
    assert p._history(x) == (h, 1)
    p.reset()
    assert p._history(x)[1] == 0
    for change in (lambda: p._set_inference_steps(20), lambda: p.set_strength(0.5)):
        p._hist_valid = True
        change()
        assert p._history(x)[1] == 0
    p._hist_valid = True
    h2, v2 = p._history(torch.zeros(4, 3))                     # new shape: new buffer, first order
    assert v2 == 0 and h2.shape == (4, 3)


def test_failed_launch_leaves_history_invalid(monkeypatch):
    """A step whose launch fails has written no history: the flag must not claim otherwise."""
    from stable_diffusion_pytorch_b200 import _lib

    class Failing:
        def __getattr__(self, name):
            return lambda *a: -1

        def sdk_last_error(self):
            return b"launch failed"
    monkeypatch.setattr(_lib, "lib", lambda: Failing())
    monkeypatch.setattr(DPMSolverSampler, "_check_cuda", staticmethod(lambda x, what: None))
    monkeypatch.setattr(torch.cuda, "device", lambda d: __import__("contextlib").nullcontext())
    monkeypatch.setattr(_lib, "current_stream", lambda d: 0)
    p = DPMSolverSampler()
    p._set_inference_steps(10)
    x = torch.zeros(1, 4, 8, 8)
    with pytest.raises(RuntimeError, match="launch failed"):
        p.reverse_process(x, int(p.timesteps[0]), x)
    assert p._history(x)[1] == 0
    with pytest.raises(RuntimeError, match="launch failed"):
        p.inpaint_step(x, int(p.timesteps[0]), x, x, torch.ones(8, 8, dtype=torch.bool))
    assert p._history(x)[1] == 0
