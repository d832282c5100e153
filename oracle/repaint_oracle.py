"""CPU ORACLE (test infrastructure only) -- RePaint resampling.

Checker only: imported by `tests/`, never by the product path.  Written from the paper (Lugmayr et al. 2022, "RePaint:
Inpainting using Denoising Diffusion Probabilistic Models", Algorithm 1 and the jump schedule of its code), not from
`repaint.py`:

  * `schedule`: the time list (jumps of `jump_length` at every jump point, `jump_n_sample - 1` times each);
  * `sample_loop`: float64 loop over the time pairs of that list -- a step down is the class path's DDPM step with
    the known-region injection before the model call, a step up is ONE level of forward re-noising,
    x <- sqrt(1 - beta_s) x + sqrt(beta_s) z, with every noise taken from an injected provider;
  * `collapse_undo_noise`: the single undo draw u of the package's collapsed undo that reproduces given per-level draws
    exactly (sum_s w_s z_s / s_u with sum_s w_s^2 = s_u^2: standard normal when the z_s are);
  * `mirror_undo`: an fp32 op-order mirror of one launch of K7 (csrc/sampler_resample.cu), one IEEE rounding per op;
  * `CorrelatedGaussian`: Gaussian data with spatially correlated pixels, Sigma_ij = 0.25 exp(-|p_i - p_j| / 4)
    + 1e-4 delta_ij per channel (block-diagonal over channels), mean 0.  Its exact eps predictor and the exact
    conditional distribution of the hole given the known pixels are closed-form.
"""
import math

import numpy as np
import torch


# ------------------------------------------------------------------------------------------ the jump schedule
def schedule(T, jump_length, jump_n_sample):
    jumps = {}
    for j in range(0, T - jump_length, jump_length):
        jumps[j] = jump_n_sample - 1
    t = T
    ts = []
    while t >= 1:
        t = t - 1
        ts.append(t)
        if jumps.get(t, 0) > 0:
            jumps[t] = jumps[t] - 1
            for _ in range(jump_length):
                t = t + 1
                ts.append(t)
    ts.append(-1)
    return ts


# ------------------------------------------------------------------------------------------ float64 loop
def sample_loop(betas, model, x_T, jump_length, jump_n_sample, *, gt, keep, noise, var="small", clip=False,
                injection_schedule="all", cumulative=True, trace=None):
    """float64.  model(x, t) -> eps.  noise(kind, t, visit) -> float64 tensor shaped like x_T, kind in
    "inject" | "step" | "undo"; visit counts the earlier draws of the same (kind, t) and is 0 for every injection
    when the injection noise is cumulative (one noise per timestep).  Returns the sample at t = 0."""
    b = np.asarray(betas, dtype=np.float64)
    T = len(b)
    ab = np.cumprod(1.0 - b)
    abp = np.append(1.0, ab[:-1])
    post_var = b * (1.0 - abp) / (1.0 - ab)
    logvar = np.log(np.append(post_var[1], post_var[1:] if var == "small" else b[1:]))
    visits = {}

    def draw(kind, t):
        v = visits.get((kind, t), 0)
        visits[(kind, t)] = v + 1
        return noise(kind, t, 0 if (kind == "inject" and cumulative) else v).double()

    m = keep.double().expand_as(x_T)
    x = x_T.double()
    ts = schedule(T, jump_length, jump_n_sample)
    for t_last, t_cur in zip(ts[:-1], ts[1:]):
        if t_cur < t_last:                       # reverse step at t = t_last (Algorithm 1, lines 4-7)
            t = t_last
            gated = (injection_schedule == "high" and t < T // 2) or (injection_schedule == "low" and t >= T // 2)
            if not gated:
                known = math.sqrt(ab[t]) * gt.double() + math.sqrt(1.0 - ab[t]) * draw("inject", t)
                x = m * known + (1 - m) * x
            eps = model(x, t).double()
            x0 = math.sqrt(1.0 / ab[t]) * x - math.sqrt(1.0 / ab[t] - 1.0) * eps
            if clip:
                x0 = x0.clamp(-1, 1)
            c1 = b[t] * math.sqrt(abp[t]) / (1.0 - ab[t])
            c2 = (1.0 - abp[t]) * math.sqrt(1.0 - b[t]) / (1.0 - ab[t])
            z = draw("step", t)
            x = c1 * x0 + c2 * x + (math.exp(0.5 * logvar[t]) * z if t > 0 else 0.0)
            if trace is not None:
                trace.append({"t": t, "sample": x.clone()})
        else:                                    # one level up: q(x_{t_cur} | x_{t_cur - 1}) (line 9)
            s = t_cur
            x = math.sqrt(1.0 - b[s]) * x + math.sqrt(b[s]) * draw("undo", s)
    return x


def collapse_undo_noise(betas, t, t_up, zs):
    """The undo noise u of the collapsed re-noising from level t - 1 to t_up for which a_u x + s_u u equals the
    step-by-step re-noising with the per-level draws zs = [z_t, ..., z_{t_up}]."""
    b = np.asarray(betas, dtype=np.float64)
    levels = list(range(t, t_up + 1))
    acc = 0.0
    for s, z in zip(levels, zs):
        w = math.sqrt(b[s]) * math.prod(math.sqrt(1.0 - b[r]) for r in range(s + 1, t_up + 1))
        acc = acc + w * z.double()
    s_u = math.sqrt(1.0 - math.prod(1.0 - b[s] for s in levels))
    return acc / s_u


# ------------------------------------------------------------------------------------------ fp32 op-order mirror of K7
def mirror_undo(x, u, undo_a, undo_s, *, gt=None, keep=None, noise=None, inject_a=None, inject_s=None):
    """One K7 launch on fp32 CPU tensors: x' = undo_a*x + undo_s*u, then keep*(ia*gt + is*n) + (1-keep)*x'."""
    f = lambda v: torch.tensor(float(v), dtype=torch.float32)  # noqa: E731
    xn = f(undo_a) * x + f(undo_s) * u
    if gt is not None:
        k = keep.expand_as(x)
        wg = f(inject_a) * gt + f(inject_s) * noise
        xn = k * wg + (1 - k) * xn
    return xn


# ------------------------------------------------------------------------------------------ analytic model
class CorrelatedGaussian:
    """x0 ~ N(0, Sigma) over [channels][H][W], Sigma block-diagonal over channels.  All float64."""

    def __init__(self, alphas_cumprod, H, W, channels=1):
        self.ab = np.asarray(alphas_cumprod, dtype=np.float64)
        self.C, self.H, self.W = channels, H, W
        yy, xx = torch.meshgrid(torch.arange(H, dtype=torch.float64), torch.arange(W, dtype=torch.float64),
                                indexing="ij")
        p = torch.stack([yy.reshape(-1), xx.reshape(-1)], 1)
        dist = torch.cdist(p, p)
        self.sigma = 0.25 * torch.exp(-dist / 4.0) + 1e-4 * torch.eye(H * W, dtype=torch.float64)
        self.mu = torch.zeros(H * W, dtype=torch.float64)
        self._inv = {}

    def _m(self, t, device):
        key = (int(t), str(device))
        if key not in self._inv:
            a2, s2 = self.ab[t], 1.0 - self.ab[t]
            self._inv[key] = torch.linalg.inv(a2 * self.sigma + s2 * torch.eye(len(self.mu), dtype=torch.float64)).to(device)
        return self._inv[key]

    def eps(self, x, t):
        """Exact eps predictor: sigma_t (alpha_t^2 Sigma + sigma_t^2 I)^-1 (x - alpha_t mu), per channel."""
        a, s = math.sqrt(self.ab[t]), math.sqrt(1.0 - self.ab[t])
        xf = x.double().reshape(x.shape[0], self.C, -1) - a * self.mu.to(x.device)
        return (s * xf @ self._m(t, x.device)).reshape(x.shape)

    def sample_prior(self, n, generator):
        L = torch.linalg.cholesky(self.sigma)
        z = torch.randn(n, self.C, self.H * self.W, generator=generator, dtype=torch.float64)
        return (self.mu + z @ L.T).reshape(n, self.C, self.H, self.W)

    def hole_conditional(self, x0, keep):
        """Exact mean [n_hole] and covariance [n_hole, n_hole] of the hole pixels (keep == 0, flattened over channels
        and pixels) given the known pixels of the image x0 [C, H, W]."""
        full = torch.block_diag(*([self.sigma] * self.C))
        mu = self.mu.repeat(self.C)
        k = keep.expand(self.C, self.H, self.W).reshape(-1) == 1
        h = ~k
        s_hk, s_kk = full[h][:, k], full[k][:, k]
        mean = mu[h] + s_hk @ torch.linalg.solve(s_kk, x0.double().reshape(-1)[k] - mu[k])
        cov = full[h][:, h] - s_hk @ torch.linalg.solve(s_kk, s_hk.T)
        return mean, cov


def harmonization_errors(samples, keep, mean, cov):
    """(RMS error of the hole's sample mean, relative Frobenius error of its sample covariance) of samples [B, C, H, W]
    against the exact conditional."""
    B = samples.shape[0]
    h = keep.reshape(keep.shape[-3:]).expand(samples.shape[1:]).reshape(-1) == 0
    xs = samples.double().reshape(B, -1)[:, h].cpu()
    d = xs - xs.mean(0)
    emp = d.T @ d / (B - 1)
    return ((xs.mean(0) - mean) ** 2).mean().sqrt().item(), ((emp - cov).norm() / cov.norm()).item()
