"""CPU ORACLE (test infrastructure only) -- DPM-Solver++ multistep inpainting sampler.

Checker only: imported by `tests/` and `tools/dpm_solver_probe.py`, never by the product path.  Two restatements of
`GaussianDiffusion.dpm_solver_sample_loop`, written from the paper (Lu et al. 2022, "DPM-Solver++: Fast Solver for
Guided Sampling of Diffusion Probabilistic Models", Algorithm 2 / eq. (13) and the multistep 2M update), not from
`dpm_solver.py`:

  * `sample_loop`: float64 loop in the paper's D-form  x_t = (s_t/s_s) x - a_t (e^{-h} - 1) D,
    D = (1 + 1/2r) x0_s - (1/2r) x0_{s'}  (first order: D = x0_s), with the package's grid, order rule and injection.
  * `mirror_step`: an fp32 op-order mirror of one launch of K6 (csrc/sampler_multistep.cu) on torch CPU tensors, one
    IEEE rounding per op in the kernel's order, given the kernel's fp32 coefficient row.

and the analytic model the accuracy checks use: per-pixel Gaussian data x0 ~ N(mu, s^2), for which the exact eps
predictor and the exact probability-flow ODE solution are closed-form.
"""
import numpy as np
import torch


# ------------------------------------------------------------------------------------------ float64 loop (D-form)
def grid(T, steps):
    """The integer timesteps the sampler evaluates at: T-1 .. 0, evenly spaced, rounded."""
    return [int(v) for v in np.round(np.linspace(T - 1, 0, steps))]


def _alpha_sigma_lambda(ab):
    a, s = np.sqrt(ab), np.sqrt(1.0 - ab)
    return a, s, np.log(a) - np.log(s)


def d_form_update(ab_s, ab_t, ab_prev, x, m, m_prev):
    """One update from s to t in float64.  m_prev None: first order; else second order with the history point at
    alphas_cumprod = ab_prev."""
    a_s, s_s, l_s = _alpha_sigma_lambda(ab_s)
    a_t, s_t, l_t = _alpha_sigma_lambda(ab_t)
    h = l_t - l_s
    if m_prev is None:
        D = m
    else:
        _, _, l_p = _alpha_sigma_lambda(ab_prev)
        r = (l_s - l_p) / h
        D = (1.0 + 1.0 / (2.0 * r)) * m - (1.0 / (2.0 * r)) * m_prev
    return (s_t / s_s) * x - a_t * np.expm1(-h) * D


def sample_loop(alphas_cumprod, model, x_T, steps, order, *, clip=False, mean_type="epsilon", gt=None, keep=None,
                noise_fn=None, schedule="all", trace=None):
    """float64 loop.  model(x_float64, t_int) -> model output (first C channels used).  noise_fn(t) -> injection noise
    at t (the same tensor every time it is asked for the same t when the noise is cumulative).  Returns the x0
    prediction at t = 0."""
    ab = np.asarray(alphas_cumprod, dtype=np.float64)
    T = len(ab)
    ts = grid(T, steps)
    C = x_T.shape[1]

    def inject(x, t):
        gated = (schedule == "high" and t < T // 2) or (schedule == "low" and t >= T // 2)
        if gt is None or gated:
            return x
        wg = np.sqrt(ab[t]) * gt.double() + np.sqrt(1.0 - ab[t]) * noise_fn(t).double()
        m = keep.double().expand_as(x)
        return m * wg + (1 - m) * x

    x = inject(x_T.double(), ts[0])
    hist = []
    for k, t in enumerate(ts):
        out = model(x, t).double()[:, :C]
        if mean_type == "start_x":
            m = out
        else:
            m = np.sqrt(1.0 / ab[t]) * x - np.sqrt(1.0 / ab[t] - 1.0) * out
        if clip:
            m = m.clamp(-1, 1)
        if trace is not None:
            trace.append({"t": t, "x": x.clone(), "pred_xstart": m.clone()})
        if k == steps - 1:
            return m
        o = 1 if (k == 0 or k == steps - 2) else order
        x = d_form_update(ab[t], ab[ts[k + 1]], ab[ts[k - 1]] if k > 0 else None, x, m, hist[-1] if o == 2 else None)
        hist.append(m)
        x = inject(x, ts[k + 1])


# ------------------------------------------------------------------------------------------ fp32 op-order mirror of K6
def mirror_step(row, x, model_out, *, m_prev=None, update=True, clip=True, mean_type="epsilon", gt=None, keep=None,
                noise=None):
    """One K6 launch on fp32 CPU tensors.  row: the kernel's fp32 coefficient row (c1, c2, A, B0, B1, ia, is).
    Returns (m_k, x_next or None)."""
    c1, c2, A, B0, B1, ia, is_ = (torch.tensor(float(v), dtype=torch.float32) for v in row)
    C = x.shape[1]
    mo = model_out[:, :C]
    m = mo.clone() if mean_type == "start_x" else c1 * x - c2 * mo
    if clip:
        m = m.clamp(-1, 1)
    if not update:
        return m, None
    xn = A * x + B0 * m
    if m_prev is not None:
        xn = xn + B1 * m_prev
    if gt is not None:
        k = keep.expand_as(x)
        wg = ia * gt + is_ * noise
        xn = k * wg + (1 - k) * xn
    return m, xn


# ------------------------------------------------------------------------------------------ analytic model
class AnalyticGaussian:
    """Data x0 ~ N(mu, s^2) independently per pixel, mu ~ U[-0.5, 0.5], s ~ U[0.1, 0.5] (seeded).  All float64."""

    def __init__(self, alphas_cumprod, shape, seed=0):
        g = torch.Generator().manual_seed(seed)
        self.ab = np.asarray(alphas_cumprod, dtype=np.float64)
        self.mu = torch.rand(*shape, generator=g, dtype=torch.float64) - 0.5
        self.s = torch.rand(*shape, generator=g, dtype=torch.float64) * 0.4 + 0.1

    def _as(self, t):
        return float(np.sqrt(self.ab[t])), float(np.sqrt(1.0 - self.ab[t]))

    def eps(self, x, t):
        """Exact eps predictor: sigma_t (x - alpha_t mu) / (alpha_t^2 s^2 + sigma_t^2)."""
        a, s = self._as(t)
        mu, sd = self.mu.to(x.device), self.s.to(x.device)
        return s * (x.double() - a * mu) / (a * a * sd * sd + s * s)

    def exact(self, x, t_a, t_b):
        """The probability-flow ODE solution from t_a to t_b (linear per pixel)."""
        (a_a, s_a), (a_b, s_b) = self._as(t_a), self._as(t_b)
        mu, sd = self.mu.to(x.device), self.s.to(x.device)
        scale = torch.sqrt(a_b * a_b * sd * sd + s_b * s_b) / torch.sqrt(a_a * a_a * sd * sd + s_a * s_a)
        return a_b * mu + scale * (x.double() - a_a * mu)

    def reference(self, x_T):
        """x0 prediction at t = 0 of the exact solution from t = T-1: what a converged sampler returns."""
        T = len(self.ab)
        x0 = self.exact(x_T, T - 1, 0)
        return np.sqrt(1.0 / self.ab[0]) * x0 - np.sqrt(1.0 / self.ab[0] - 1.0) * self.eps(x0, 0)
