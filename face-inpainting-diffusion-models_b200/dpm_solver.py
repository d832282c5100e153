"""DPM-Solver++ multistep (Lu et al. 2022, "DPM-Solver++: Fast Solver for Guided Sampling of Diffusion Probabilistic
Models", the multistep data-prediction solver 2M) on the integer timesteps of a `GaussianDiffusion` table: the grid
and the per-step fp32 coefficient rows of K6 (`fidm_multistep_step`, csrc/sampler_multistep.cu).

With alpha_t = sqrt(ab_t), sigma_t = sqrt(1 - ab_t), lambda_t = log(alpha_t) - log(sigma_t), the update from s = t_k to
t = t_{k+1} with h = lambda_t - lambda_s and phi = expm1(-h) is

    order 1:  x <- (sigma_t / sigma_s) x - alpha_t phi m_k                                  (= DDIM, eta = 0)
    order 2:  x <- (sigma_t / sigma_s) x - alpha_t phi [(1 + 1/2r) m_k - (1/2r) m_{k-1}],  r = (lambda_s - lambda_{t_{k-1}}) / h

where m_k is the model's x0 prediction at t_k.  Each update is stored as the row x' = A x + B0 m_k + B1 m_{k-1},
computed in float64 and rounded to fp32 once.  The first update has no history and the update into t = 0 is first
order: with a second-order step into t = 0 the solver is less accurate than DDIM at 20 steps.
"""
import numbers

import numpy as np
import torch

from . import _lib as L


def timestep_grid(num_timesteps, steps):
    """t_k = round(linspace(T - 1, 0, steps)): `steps` distinct integer timesteps, one model evaluation each."""
    T = int(num_timesteps)
    if isinstance(steps, bool) or not isinstance(steps, numbers.Integral) or not 2 <= steps <= T:
        raise ValueError(f"steps must be an integer in [2, {T}] for a {T}-step diffusion, got {steps!r}")
    return np.round(np.linspace(T - 1, 0, int(steps))).astype(np.int64)


def step_orders(steps, order):
    """Order of the update out of t_k, k = 0 .. steps - 2: min(order, k + 1), and 1 into the last grid point."""
    if isinstance(order, bool) or order not in (1, 2):
        raise ValueError(f"order must be 1 or 2, got {order!r}")
    return [1 if k == steps - 2 else min(order, k + 1) for k in range(steps - 1)]


def update_rows(alphas_cumprod, grid, order):
    """float64 [steps, 3]: (A, B0, B1) of the update out of each grid point; the last row (no update) is zero."""
    ab = np.asarray(alphas_cumprod, dtype=np.float64)[grid]
    alpha, sigma = np.sqrt(ab), np.sqrt(1.0 - ab)
    lam = np.log(alpha) - np.log(sigma)
    rows = np.zeros((len(grid), 3), dtype=np.float64)
    for k, o in enumerate(step_orders(len(grid), order)):
        h = lam[k + 1] - lam[k]
        w = -alpha[k + 1] * np.expm1(-h)
        if o == 1:
            rows[k] = (sigma[k + 1] / sigma[k], w, 0.0)
        else:
            half_inv_r = 0.5 * h / (lam[k] - lam[k - 1])
            rows[k] = (sigma[k + 1] / sigma[k], w * (1.0 + half_inv_r), -w * half_inv_r)
    return rows


def coefficient_table(diffusion, steps, order, cumulative=True):
    """fp32 CPU tensor [steps, FIDM_MS_COLS] (column meaning in include/fidm_b200.h).  The x0-prediction and injection
    columns are the class path's own fp32 values (GaussianDiffusion.coefficient_table), so m_k and the injected pixels
    are bit-identical to its pred_xstart and injection for the same inputs."""
    grid = timestep_grid(diffusion.num_timesteps, steps)
    rows = update_rows(diffusion.alphas_cumprod, grid, order)
    cls = diffusion.coefficient_table(0.0)
    tab = torch.zeros(len(grid), L.MS_COLS, dtype=torch.float32)
    g = torch.from_numpy(grid)
    tab[:, L.MS_X0_C1] = cls[g, 4]
    tab[:, L.MS_X0_C2] = cls[g, 5]
    tab[:, L.MS_A:L.MS_B1 + 1] = torch.from_numpy(rows).float()
    ia, is_ = (0, 1) if cumulative else (2, 3)
    tab[:-1, L.MS_INJ_A] = cls[g[1:], ia]
    tab[:-1, L.MS_INJ_S] = cls[g[1:], is_]
    return tab
