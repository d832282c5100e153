"""RePaint resampling (Lugmayr et al. 2022, "RePaint: Inpainting using Denoising Diffusion Probabilistic Models",
Algorithm 1 and its jump schedule): the time walk and the per-evaluation work of
`GaussianDiffusion.repaint_sample_loop`, host only.

The walk goes down one timestep per model evaluation.  At every jump point it goes back up `jump_length` levels by
re-noising the state with the forward process, `jump_n_sample - 1` times per jump point, so that the hole and the
injected known region can agree before the walk goes further down.

The paper's code re-noises one level at a time, x <- sqrt(1 - beta_s) x + sqrt(beta_s) z, s = t .. t_up.  Here the
`jump_length` steps of one jump are collapsed into ONE draw: x <- a_u x + s_u u with a_u = sqrt(ab[t_up] / ab[t-1]),
s_u = sqrt(1 - ab[t_up] / ab[t-1]).  The result has the same distribution (the composition of Gaussian steps is
Gaussian with exactly these moments) but consumes one randn per jump instead of `jump_length`, so the RNG stream
differs from the paper's code.  It saves jump_length - 1 draws and launches per jump.
"""
import numbers
from collections import namedtuple

import numpy as np

# t: the evaluation's timestep; t_up: the level the state is re-noised to after it (None: no jump follows);
# undo_a / undo_s: a_u and s_u rounded to fp32 (0.0 when no jump follows)
Evaluation = namedtuple("Evaluation", "t t_up undo_a undo_s")


def _check(T, jump_length, jump_n_sample):
    T = int(T)
    if isinstance(jump_length, bool) or not isinstance(jump_length, numbers.Integral) or not 1 <= jump_length <= T - 1:
        raise ValueError(f"jump_length must be an integer in [1, {T - 1}] for a {T}-step diffusion, got {jump_length!r}")
    if isinstance(jump_n_sample, bool) or not isinstance(jump_n_sample, numbers.Integral) or jump_n_sample < 1:
        raise ValueError(f"jump_n_sample must be an integer >= 1, got {jump_n_sample!r}")
    return T, int(jump_length), int(jump_n_sample)


def jump_schedule(T, jump_length, jump_n_sample):
    """RePaint's time list (its get_schedule_jump with n_sample = 1): starts at T - 1, ends at -1; a step down is one
    model evaluation, a step up one level of re-noising."""
    T, jl, jn = _check(T, jump_length, jump_n_sample)
    jumps = {j: jn - 1 for j in range(0, T - jl, jl)}
    t, ts = T, []
    while t >= 1:
        t -= 1
        ts.append(t)
        if jumps.get(t, 0) > 0:
            jumps[t] -= 1
            for _ in range(jl):
                t += 1
                ts.append(t)
    ts.append(-1)
    return ts


def undo_coefficients(alphas_cumprod, t, t_up):
    """float64 (a_u, s_u) of the collapsed re-noising from level t - 1 to t_up."""
    ab = np.asarray(alphas_cumprod, dtype=np.float64)
    r = ab[t_up] / ab[t - 1]
    return float(np.sqrt(r)), float(np.sqrt(1.0 - r))


def evaluation_plan(alphas_cumprod, jump_length, jump_n_sample):
    """One Evaluation per model evaluation of the walk; consecutive steps up collapse into one undo."""
    ts = jump_schedule(len(alphas_cumprod), jump_length, jump_n_sample)
    plan = []
    i = 0
    while ts[i] >= 0:
        t = ts[i]
        assert ts[i + 1] == t - 1
        i += 1
        up = i
        while up + 1 < len(ts) and ts[up + 1] == ts[up] + 1:
            up += 1
        if up == i:
            plan.append(Evaluation(t, None, 0.0, 0.0))
            continue
        t_up = ts[up]
        a, s = undo_coefficients(alphas_cumprod, t, t_up)
        plan.append(Evaluation(t, t_up, float(np.float32(a)), float(np.float32(s))))
        i = up
    return plan
