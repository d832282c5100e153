"""CPU: DPM-Solver++ multistep host logic -- the grid, the per-step coefficient table against the float64 D-form of
oracle/dpm_solver_oracle.py, and the solver's convergence order on the analytic model."""
import math

import numpy as np
import pytest
import torch

import fidm_b200 as F
from fidm_b200 import _lib, dpm_solver
from oracle import dpm_solver_oracle as O


@pytest.mark.parametrize("T,N", [(1000, 2), (1000, 20), (1000, 25), (1000, 999), (1000, 1000), (100, 100), (7, 3)])
def test_grid_is_distinct_descending_and_spans_the_table(T, N):
    g = dpm_solver.timestep_grid(T, N)
    assert g.dtype == np.int64 and len(g) == N
    assert g[0] == T - 1 and g[-1] == 0
    assert (np.diff(g) < 0).all()
    assert g.tolist() == O.grid(T, N)


@pytest.mark.parametrize("steps", [0, 1, 1001, 2.0, "20", True, None])
def test_grid_rejects_bad_step_counts(steps):
    with pytest.raises(ValueError):
        dpm_solver.timestep_grid(1000, steps)


@pytest.mark.parametrize("order", [0, 3, 1.5, None])
def test_order_outside_one_two_raises(order):
    with pytest.raises(ValueError):
        dpm_solver.step_orders(20, order)


def test_public_loop_validates_before_drawing_or_touching_the_gpu():
    d = F.create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="quadratic")
    fn = lambda x, t, **k: torch.zeros(1, 6, 8, 8)  # noqa: E731
    with pytest.raises(ValueError):
        d.dpm_solver_sample_loop(fn, (1, 3, 8, 8), steps=1, device="cpu")
    with pytest.raises(ValueError):
        d.dpm_solver_sample_loop(fn, (1, 3, 8, 8), steps=20, order=3, device="cpu")
    with pytest.raises(_lib.FidmError):         # no CPU fallback
        d.dpm_solver_sample_loop(fn, (1, 3, 8, 8), steps=20, device="cpu")
    d_prev = F.GaussianDiffusion(betas=d.betas, model_mean_type=F.ModelMeanType.PREVIOUS_X,
                                 model_var_type=F.ModelVarType.FIXED_LARGE, loss_type=F.LossType.MSE)
    with pytest.raises(NotImplementedError):
        d_prev.dpm_solver_sample_loop(fn, (1, 3, 8, 8), steps=20, device="cpu")


@pytest.mark.parametrize("sched", ["linear", "cosine", "quadratic"])
@pytest.mark.parametrize("N,order", [(2, 2), (3, 2), (20, 1), (20, 2), (100, 2), (1000, 2)])
def test_update_rows_equal_float64_d_form(sched, N, order):
    d = F.create_gaussian_diffusion(steps=1000, noise_schedule=sched)
    ab = d.alphas_cumprod
    g = dpm_solver.timestep_grid(1000, N)
    rows = dpm_solver.update_rows(ab, g, order)
    orders = dpm_solver.step_orders(N, order)
    assert orders[0] == 1 and orders[-1] == 1
    gen = torch.Generator().manual_seed(N)
    x, m, mp = (torch.randn(64, generator=gen, dtype=torch.float64) for _ in range(3))
    for k in range(N - 1):
        second = orders[k] == 2
        want = O.d_form_update(ab[g[k]], ab[g[k + 1]], ab[g[k - 1]] if second else None, x, m, mp if second else None)
        A, B0, B1 = rows[k]
        got = A * x + B0 * m + B1 * mp
        assert ((got - want).abs().max() / want.abs().max()).item() < 1e-12, (k, orders[k])
        if not second:
            assert B1 == 0.0
    assert (rows[-1] == 0).all()


@pytest.mark.parametrize("cumulative", [True, False])
def test_table_reuses_the_class_path_fp32_values(cumulative):
    d = F.create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="quadratic")
    tab = dpm_solver.coefficient_table(d, 20, 2, cumulative)
    cls = d.coefficient_table(0.0)
    g = torch.from_numpy(dpm_solver.timestep_grid(1000, 20))
    assert tab.dtype == torch.float32 and tab.shape == (20, _lib.MS_COLS)
    assert torch.equal(tab[:, _lib.MS_X0_C1], cls[g, 4]) and torch.equal(tab[:, _lib.MS_X0_C2], cls[g, 5])
    ia, is_ = (0, 1) if cumulative else (2, 3)
    assert torch.equal(tab[:-1, _lib.MS_INJ_A], cls[g[1:], ia]) and torch.equal(tab[:-1, _lib.MS_INJ_S], cls[g[1:], is_])
    rows = dpm_solver.update_rows(d.alphas_cumprod, g.numpy(), 2)
    assert torch.equal(tab[:, _lib.MS_A:_lib.MS_B1 + 1], torch.from_numpy(rows).float())


def _rms_errors(sched, order, Ns):
    ab = F.create_gaussian_diffusion(steps=1000, noise_schedule=sched).alphas_cumprod
    shape = (4, 3, 32, 32)
    model = O.AnalyticGaussian(ab, shape, seed=1)
    x_T = torch.randn(*shape, generator=torch.Generator().manual_seed(2), dtype=torch.float64)
    ref = model.reference(x_T)
    return [((O.sample_loop(ab, model.eps, x_T, N, order) - ref) ** 2).mean().sqrt().item() for N in Ns]


@pytest.mark.parametrize("sched", ["linear", "cosine"])
def test_convergence_order_on_the_analytic_model(sched):
    """2M converges at second order on the time-uniform grid of a 1000-step table, order 1 (DDIM) at first order, and
    2M at N = 40 beats order 1 at N = 80."""
    Ns = (10, 20, 40, 80, 160)
    e1, e2 = _rms_errors(sched, 1, Ns), _rms_errors(sched, 2, Ns)
    slope = lambda e, i: math.log2(e[i] / e[i + 1])  # noqa: E731
    print(sched, "order 1", ["%.2e" % v for v in e1], "2M", ["%.2e" % v for v in e2])
    assert slope(e2, 2) >= 1.8, e2
    assert 0.9 <= slope(e1, 2) <= 1.1, e1
    assert e2[2] < e1[3], (e2, e1)
