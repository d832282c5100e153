"""`GaussianDiffusion`: the masked-inpainting reverse process on a B200.

Drop-in for the sampling half of the reference's class (`gaussian_diffusion.py:27-538, 640-700`):
same constructor, attribute names, method names, argument order and defaults, same RNG draw order
(`randn(shape)` once, then per step `randn_like(gt)` on an injection-cache miss and `randn_like(x)`),
so seeding torch's generator reproduces the reference's noise on the same device.  With `seeds=` the fused loops instead
generate every noise value inside the sampler kernels from per-image seeds (seeded.py), independent of the batch.

What differs is the execution.  Per step the reference launches ~40 elementwise ATen kernels,
re-uploads 14 coefficient tables and synchronises on `.item()` (`:131`); here a step is ONE fused
launch (`fidm_sampler_step`, K4) that applies the update at t and the known-region injection for
t-1, reading per-timestep coefficients from a device table built once.  The table is computed on
the host with the reference's own arithmetic (float64 entry rounded to fp32, `:12-24`; sigma and
the DDIM square roots in fp32, `:472-482`), so results are bit-identical on the DDIM path.

Training utilities (`training_losses`, `_vb_terms_bpd`, `:540-637`) are not part of the sampling
path and raise NotImplementedError.
"""
import ctypes as C
import os

import numpy as np
import torch

from . import _lib as L
from . import dpm_solver, repaint, seeded
from .losses import LossType, ModelMeanType, ModelVarType  # noqa: F401

try:  # tqdm is only used when progress=True, as in the reference
    from tqdm.auto import tqdm
except Exception:  # pragma: no cover
    tqdm = None


def _extract_into_tensor(arr, timesteps, broadcast_shape):
    """Same contract as the reference helper (`:12-24`): fp32 values of a float64 table at `timesteps`,
    broadcast to `broadcast_shape`.  Only used by the unfused compatibility paths."""
    vals = torch.from_numpy(np.asarray(arr)).to(device=timesteps.device)[timesteps].float()
    vals = vals.reshape(vals.shape + (1,) * (len(broadcast_shape) - vals.dim()))
    return vals.expand(broadcast_shape)


def _f32(t):
    """`t` detached, as the fp32 contiguous tensor the sampler kernels read (`t` itself when it already is one)."""
    if t is None:
        return None
    t = t.detach()
    if t.dtype != torch.float32 or not t.is_contiguous():
        t = t.to(torch.float32).contiguous()
    return t


def _set_injection(a, x, gt, keep, inject_noise):
    """Point the known-region fields of a sampler arg struct (StepArgs, MultistepArgs, ResampleArgs) at fp32 copies of
    gt, keep and inject_noise.  Returns the copies: the caller holds them until the launch."""
    gt, keep, inject_noise = _f32(gt), _f32(keep), _f32(inject_noise)
    assert gt.shape == x.shape and (inject_noise is None or inject_noise.shape == x.shape)
    assert keep.shape[0] == x.shape[0] and keep.shape[2:] == x.shape[2:], tuple(keep.shape)
    a.gt, a.keep_mask, a.inject_noise = L.ptr(gt), L.ptr(keep), L.ptr(inject_noise)
    a.mask_channels = keep.shape[1]
    return gt, keep, inject_noise


def _set_stem(a, stem, t_next):
    """Step-boundary fusion fields of a sampler arg struct: stem = (NHWC network input, timestep tensor) of an engine
    plan receives the new state and, when t_next is given, the next timestep."""
    if stem is not None:
        x_in, t_in = stem
        a.stem_out, a.stem_dtype, a.stem_ld = L.ptr(x_in), L.dtype_code(x_in.dtype), x_in.shape[-1]
        if t_next is not None:
            a.t_out, a.t_out_value = L.ptr(t_in), float(t_next)


def _known_region(model_kwargs, use_inpainting_injection):
    """(gt, gt_keep_mask) from model_kwargs when the injection is on and both are given, else (None, None)."""
    if use_inpainting_injection and model_kwargs:
        gt, keep = model_kwargs.get("gt"), model_kwargs.get("gt_keep_mask")
        if gt is not None and keep is not None:
            return gt, keep
    return None, None


class _TorchDraws:
    """The noise of one unseeded loop: torch's generator, in the reference's draw order (the injection noise through
    the per-timestep cache when cumulative, drawn like `gt`)."""

    def __init__(self, diffusion, gt, cumulative):
        self.diffusion, self.gt, self.cumulative = diffusion, gt, cumulative

    def inject(self, ts):
        return self.diffusion._cached_noise(self.gt, ts) if self.cumulative else torch.randn_like(self.gt)

    def step(self, x, k):
        return torch.randn_like(x)

    undo = step


_MEAN_CODE = {ModelMeanType.PREVIOUS_X: L.MEAN_PREVIOUS_X, ModelMeanType.START_X: L.MEAN_START_X,
              ModelMeanType.EPSILON: L.MEAN_EPSILON}
_VAR_CODE = {ModelVarType.LEARNED: L.VAR_LEARNED, ModelVarType.LEARNED_RANGE: L.VAR_LEARNED_RANGE,
             ModelVarType.FIXED_LARGE: L.VAR_FIXED, ModelVarType.FIXED_SMALL: L.VAR_FIXED}


class GaussianDiffusion:
    def __init__(self, *, betas, model_mean_type, model_var_type, loss_type, rescale_timesteps=False):
        self.model_mean_type = model_mean_type
        self.model_var_type = model_var_type
        self.loss_type = loss_type
        self.rescale_timesteps = rescale_timesteps

        betas = np.array(betas, dtype=np.float64)
        assert betas.ndim == 1, "betas must be 1-D"
        assert (betas > 0).all() and (betas <= 1).all()
        self.betas = betas
        self.num_timesteps = int(betas.shape[0])

        # float64 tables, named as in the reference (:53-83)
        ab = np.cumprod(1.0 - betas, axis=0)
        ab_prev = np.append(1.0, ab[:-1])
        self.alphas_cumprod = ab
        self.alphas_cumprod_prev = ab_prev
        self.alphas_cumprod_next = np.append(ab[1:], 0.0)
        self.sqrt_alphas_cumprod = np.sqrt(ab)
        self.sqrt_one_minus_alphas_cumprod = np.sqrt(1.0 - ab)
        self.log_one_minus_alphas_cumprod = np.log(1.0 - ab)
        self.sqrt_recip_alphas_cumprod = np.sqrt(1.0 / ab)
        self.sqrt_recipm1_alphas_cumprod = np.sqrt(1.0 / ab - 1)
        self.posterior_variance = betas * (1.0 - ab_prev) / (1.0 - ab)
        self.posterior_log_variance_clipped = np.log(
            np.append(self.posterior_variance[1], self.posterior_variance[1:]))
        self.posterior_mean_coef1 = betas * np.sqrt(ab_prev) / (1.0 - ab)
        self.posterior_mean_coef2 = (1.0 - ab_prev) * np.sqrt(1.0 - betas) / (1.0 - ab)

        self._gt_noises_cache = {}
        self._coef_cache = {}

    # ------------------------------------------------------------------ coefficient table (K4)
    def coefficient_table(self, eta=0.0):
        """[T, FIDM_COEF_COLS] fp32 CPU tensor; column meaning in include/fidm_b200.h."""
        T = self.num_timesteps

        def f(a):  # float64 table -> fp32, the rounding of _extract_into_tensor (:21)
            return torch.from_numpy(np.asarray(a, dtype=np.float64)).float()

        ab, abp = f(self.alphas_cumprod), f(self.alphas_cumprod_prev)
        tab = torch.zeros(T, L.COEF_COLS, dtype=torch.float32)
        tab[:, 0] = f(self.sqrt_alphas_cumprod)
        tab[:, 1] = f(self.sqrt_one_minus_alphas_cumprod)
        tab[:, 2] = torch.sqrt(ab)                       # :143-145, fp32 on device in the reference
        tab[:, 3] = torch.sqrt(1 - ab)
        tab[:, 4] = f(self.sqrt_recip_alphas_cumprod)
        tab[:, 5] = f(self.sqrt_recipm1_alphas_cumprod)
        tab[:, 6] = f(np.log(self.betas))
        tab[:, 7] = f(self.posterior_log_variance_clipped)
        tab[:, 8] = f(self.posterior_mean_coef1)
        tab[:, 9] = f(self.posterior_mean_coef2)
        if self.model_var_type == ModelVarType.FIXED_SMALL:
            tab[:, 10] = f(self.posterior_log_variance_clipped)
        else:                                            # FIXED_LARGE (:254-258)
            tab[:, 10] = f(np.log(np.append(self.posterior_variance[1], self.betas[1:])))
        sigma = eta * torch.sqrt((1 - abp) / (1 - ab)) * torch.sqrt(1 - ab / abp)       # :474-477
        tab[:, 11] = torch.sqrt(abp)
        tab[:, 12] = torch.sqrt(1 - abp - sigma ** 2)
        tab[:, 13] = sigma
        tab[:, 14] = (torch.arange(T) != 0).float()
        with np.errstate(divide="ignore", invalid="ignore"):
            tab[:, 15] = f(1.0 / self.posterior_mean_coef1)
            tab[:, 16] = f(self.posterior_mean_coef2 / self.posterior_mean_coef1)
        return tab

    def _coef(self, device, eta):
        key = (str(device), float(eta))
        if key not in self._coef_cache:
            self._coef_cache[key] = self.coefficient_table(eta).to(device)
        return self._coef_cache[key]

    # ------------------------------------------------------------------ K4 launcher
    def _step(self, mode, x, *, t=None, t_inject=None, t_dev=None, model_out=None, z=None, gt=None, keep=None,
              inject_noise=None, ddim=True, eta=0.0, clip=True, cumulative=True, want_sample=False,
              want_x0=False, want_next=False, want_mean=False, want_logvar=False, script_table=None,
              stem=None, t_next=None, next_buf=None):
        """One K4 launch.  stem = (NHWC network-input tensor, timestep tensor) of an engine plan: the state after this call
        is also written as the first channels of the stem input and `t_next` into the timestep tensor (step-boundary
        fusion); next_buf: preallocated fp32 tensor for x_next.  z / inject_noise may be seeded.Draw values: the launch is
        then the seeded entry, which generates them in the kernel."""
        sn = seeded.launch_args(z, inject_noise)
        if sn is not None:
            z = inject_noise = None
        L.require_cuda(x, model_out, z, gt, keep, inject_noise)
        B, Cn = x.shape[0], x.shape[1]
        hw = x.numel() // (B * Cn)
        a = L.StepArgs()
        a.batch, a.channels, a.hw = B, Cn, hw
        a.mode = mode
        a.sampler = L.SAMPLER_DDIM if ddim else L.SAMPLER_DDPM
        a.mean_type, a.var_type = _MEAN_CODE[self.model_mean_type], _VAR_CODE[self.model_var_type]
        if script_table is not None:      # per-step rows of the evaluation scripts' strided DDIM
            a.sampler = L.SAMPLER_DDIM_SCRIPT
        a.clip_denoised, a.cumulative = int(bool(clip)), int(bool(cumulative))
        a.num_timesteps = self.num_timesteps if script_table is None else script_table.shape[0]
        a.t_update = -1 if t is None else int(t)
        a.t_inject = -1 if t_inject is None else int(t_inject)
        coef = script_table if script_table is not None else self._coef(x.device, eta if ddim else 0.0)
        x = _f32(x)
        a.coef, a.x = L.ptr(coef), L.ptr(x)
        if t_dev is not None:
            t_dev = t_dev.detach().to(device=x.device, dtype=torch.int64).contiguous()
            # the kernel indexes the coefficient table with these: validate on the host (the reference raises
            # IndexError from its table gather, :21).  Only the single-step entry points pass per-sample tensors;
            # the fused loops pass scalars that the C ABI range-checks itself.
            lo, hi = (int(v) for v in torch.stack(torch.aminmax(t_dev)).tolist())
            if lo < (1 if mode == L.STEP_UPDATE_INJECT else 0) or hi >= a.num_timesteps:
                raise IndexError(f"timesteps [{lo}, {hi}] out of range for a {a.num_timesteps}-step table")
            a.t_dev = L.ptr(t_dev)
        if mode != L.STEP_INJECT_ONLY:
            model_out, z = _f32(model_out), _f32(z)
            want_ch = Cn if a.var_type == L.VAR_FIXED else 2 * Cn
            if script_table is not None and model_out.shape[1] == Cn:
                a.var_type = L.VAR_FIXED          # scripts accept 3- or 6-channel outputs (:515-520)
                want_ch = Cn
            assert model_out.shape == (B, want_ch) + tuple(x.shape[2:]), \
                f"model output shape {tuple(model_out.shape)} != {(B, want_ch) + tuple(x.shape[2:])}"
            a.model_out, a.z = L.ptr(model_out), L.ptr(z)
        a.mask_channels = 1
        if mode != L.STEP_UPDATE_ONLY:
            gt, keep, inject_noise = _set_injection(a, x, gt, keep, inject_noise)
            assert keep.shape[1] in (1, Cn), tuple(keep.shape)
        out = {}
        for flag, key, field in ((want_sample, "sample", "sample"), (want_x0, "pred_xstart", "pred_xstart"),
                                 (want_next, "x_next", "x_next"), (want_mean, "mean", "mean_out"),
                                 (want_logvar, "log_variance", "logvar_out")):
            if flag:
                out[key] = next_buf if (key == "x_next" and next_buf is not None) else torch.empty_like(x)
                setattr(a, field, L.ptr(out[key]))
        _set_stem(a, stem, t_next)
        if sn is None:
            L.check(L.lib().fidm_sampler_step(C.byref(a), L.stream()), "sampler_step")
        else:
            L.check(L.lib().fidm_sampler_step_seeded(C.byref(a), C.byref(sn), L.stream()), "sampler_step_seeded")
        return out

    # ------------------------------------------------------------------ forward process helpers
    def q_mean_variance(self, x_start, t):
        mean = _extract_into_tensor(self.sqrt_alphas_cumprod, t, x_start.shape) * x_start
        variance = _extract_into_tensor(1.0 - self.alphas_cumprod, t, x_start.shape)
        log_variance = _extract_into_tensor(self.log_one_minus_alphas_cumprod, t, x_start.shape)
        return mean, variance, log_variance

    def q_sample(self, x_start, t, noise=None):
        """Sample q(x_t | x_0) (`:172-189`)."""
        if noise is None:
            noise = torch.randn_like(x_start)
        assert noise.shape == x_start.shape
        return (_extract_into_tensor(self.sqrt_alphas_cumprod, t, x_start.shape) * x_start
                + _extract_into_tensor(self.sqrt_one_minus_alphas_cumprod, t, x_start.shape) * noise)

    def q_posterior_mean_variance(self, x_start, x_t, t):
        assert x_start.shape == x_t.shape
        mean = (_extract_into_tensor(self.posterior_mean_coef1, t, x_t.shape) * x_start
                + _extract_into_tensor(self.posterior_mean_coef2, t, x_t.shape) * x_t)
        var = _extract_into_tensor(self.posterior_variance, t, x_t.shape)
        logvar = _extract_into_tensor(self.posterior_log_variance_clipped, t, x_t.shape)
        return mean, var, logvar

    # ------------------------------------------------------------------ known-region injection
    def clear_gt_noise_cache(self):
        self._gt_noises_cache.clear()

    def _cached_noise(self, gt, timestep):
        key = (gt.shape, timestep, gt.device)                # same key as the reference (:94)
        if key not in self._gt_noises_cache:
            self._gt_noises_cache[key] = torch.randn_like(gt)
        return self._gt_noises_cache[key]

    def get_gt_noised(self, gt, timestep):
        """q_sample(gt, timestep) with the per-timestep cached noise (`:85-108`)."""
        noise = self._cached_noise(gt, timestep)
        zero_mask = torch.ones(gt.shape[0], 1, *gt.shape[2:], device=gt.device)
        return self._step(L.STEP_INJECT_ONLY, gt, t_inject=timestep, gt=gt, keep=zero_mask,
                          inject_noise=noise, want_next=True)["x_next"]

    def _injection_gated(self, timestep, schedule):
        # :132-135
        if schedule == "high" and timestep < self.num_timesteps // 2:
            return True
        if schedule == "low" and timestep >= self.num_timesteps // 2:
            return True
        return False

    def apply_inpainting_injection(self, x, t, gt, gt_keep_mask, use_cumulative_noise=True,
                                   injection_schedule="all"):
        """x <- m * q_sample(gt, t) + (1 - m) * x  (`:114-157`)."""
        if gt is None or gt_keep_mask is None:
            return x
        timestep = int(t[0].item())
        if self._injection_gated(timestep, injection_schedule):
            return x
        if use_cumulative_noise:
            noise = self._cached_noise(gt, timestep)
            return self._step(L.STEP_INJECT_ONLY, x, t_inject=timestep, gt=gt, keep=gt_keep_mask,
                              inject_noise=noise, cumulative=True, want_next=True)["x_next"]
        noise = torch.randn_like(gt)
        return self._step(L.STEP_INJECT_ONLY, x, t_dev=t, gt=gt, keep=gt_keep_mask, inject_noise=noise,
                          cumulative=False, want_next=True)["x_next"]

    # ------------------------------------------------------------------ model posterior
    def _scale_timesteps(self, t):
        if self.rescale_timesteps:
            return t.float() * (1000.0 / self.num_timesteps)
        return t

    def _t_value(self, ts):
        """What the model sees for the integer timestep ts: _scale_timesteps (:321-324) in fp32 arithmetic."""
        if self.rescale_timesteps:
            return float(np.float32(ts) * np.float32(1000.0 / self.num_timesteps))
        return float(ts)

    def _call_model(self, model, x, t, model_kwargs):
        out = model(x, self._scale_timesteps(t), **(model_kwargs or {}))
        return out

    def p_mean_variance(self, model, x, t, clip_denoised=True, denoised_fn=None, model_kwargs=None):
        """Model call + posterior statistics (`:213-298`); returns mean / variance / log_variance /
        pred_xstart."""
        B = x.shape[0]
        assert t.shape == (B,)
        model_output = self._call_model(model, x, t, model_kwargs)
        if denoised_fn is not None:
            return self._p_mean_variance_unfused(model_output, x, t, clip_denoised, denoised_fn)
        r = self._step(L.STEP_UPDATE_ONLY, x, t_dev=t, model_out=model_output, ddim=False, clip=clip_denoised,
                       want_x0=True, want_mean=True, want_logvar=True)
        if self.model_var_type in (ModelVarType.LEARNED, ModelVarType.LEARNED_RANGE):
            variance = torch.exp(r["log_variance"])
        else:
            table = (self.posterior_variance if self.model_var_type == ModelVarType.FIXED_SMALL
                     else np.append(self.posterior_variance[1], self.betas[1:]))
            variance = _extract_into_tensor(table, t, x.shape)
        return {"mean": r["mean"], "variance": variance, "log_variance": r["log_variance"],
                "pred_xstart": r["pred_xstart"]}

    def _p_mean_variance_unfused(self, model_output, x, t, clip_denoised, denoised_fn):
        """Compatibility path for a user `denoised_fn` (arbitrary Python between the x0 prediction and
        the clamp, `:267-271`): the same arithmetic as K4 spelled as tensor ops."""
        Cn = x.shape[1]
        if self.model_var_type in (ModelVarType.LEARNED, ModelVarType.LEARNED_RANGE):
            model_output, v = torch.split(model_output, Cn, dim=1)
            if self.model_var_type == ModelVarType.LEARNED:
                logvar = v
            else:
                lo = _extract_into_tensor(self.posterior_log_variance_clipped, t, x.shape)
                hi = _extract_into_tensor(np.log(self.betas), t, x.shape)
                frac = (v + 1) / 2
                logvar = frac * hi + (1 - frac) * lo
            var = torch.exp(logvar)
        else:
            small = self.model_var_type == ModelVarType.FIXED_SMALL
            vt = self.posterior_variance if small else np.append(self.posterior_variance[1], self.betas[1:])
            lt = self.posterior_log_variance_clipped if small else np.log(vt)
            var, logvar = _extract_into_tensor(vt, t, x.shape), _extract_into_tensor(lt, t, x.shape)

        def finish(v):
            v = denoised_fn(v) if denoised_fn is not None else v
            return v.clamp(-1, 1) if clip_denoised else v

        if self.model_mean_type == ModelMeanType.PREVIOUS_X:
            x0 = finish(self._predict_xstart_from_xprev(x, t, model_output))
            mean = model_output
        else:
            x0 = finish(model_output if self.model_mean_type == ModelMeanType.START_X
                        else self._predict_xstart_from_eps(x, t, model_output))
            mean, _, _ = self.q_posterior_mean_variance(x0, x, t)
        return {"mean": mean, "variance": var, "log_variance": logvar, "pred_xstart": x0}

    def _predict_xstart_from_eps(self, x_t, t, eps):
        assert x_t.shape == eps.shape
        return (_extract_into_tensor(self.sqrt_recip_alphas_cumprod, t, x_t.shape) * x_t
                - _extract_into_tensor(self.sqrt_recipm1_alphas_cumprod, t, x_t.shape) * eps)

    def _predict_xstart_from_xprev(self, x_t, t, xprev):
        assert x_t.shape == xprev.shape
        return (_extract_into_tensor(1.0 / self.posterior_mean_coef1, t, x_t.shape) * xprev
                - _extract_into_tensor(self.posterior_mean_coef2 / self.posterior_mean_coef1, t, x_t.shape) * x_t)

    def _predict_eps_from_xstart(self, x_t, t, pred_xstart):
        return ((_extract_into_tensor(self.sqrt_recip_alphas_cumprod, t, x_t.shape) * x_t - pred_xstart)
                / _extract_into_tensor(self.sqrt_recipm1_alphas_cumprod, t, x_t.shape))

    def condition_mean(self, cond_fn, p_mean_var, x, t, model_kwargs=None):
        grad = cond_fn(x, self._scale_timesteps(t), **(model_kwargs or {}))
        return p_mean_var["mean"].float() + p_mean_var["variance"] * grad.float()

    def condition_score(self, cond_fn, p_mean_var, x, t, model_kwargs=None):
        ab = _extract_into_tensor(self.alphas_cumprod, t, x.shape)
        eps = self._predict_eps_from_xstart(x, t, p_mean_var["pred_xstart"])
        eps = eps - (1 - ab).sqrt() * cond_fn(x, self._scale_timesteps(t), **(model_kwargs or {}))
        out = dict(p_mean_var)
        out["pred_xstart"] = self._predict_xstart_from_eps(x, t, eps)
        out["mean"], _, _ = self.q_posterior_mean_variance(out["pred_xstart"], x, t)
        return out

    # ------------------------------------------------------------------ single reverse steps
    def _maybe_inject(self, x, t, model_kwargs, on, schedule, cumulative):
        gt, keep = _known_region(model_kwargs, on)
        if gt is None:
            return x
        return self.apply_inpainting_injection(x, t, gt, keep, use_cumulative_noise=cumulative,
                                               injection_schedule=schedule)

    def p_sample(self, model, x, t, clip_denoised=True, denoised_fn=None, cond_fn=None, model_kwargs=None,
                 use_inpainting_injection=False, injection_schedule="all", use_cumulative_noise=True):
        """One DDPM step with optional pre-model injection (`:357-388`)."""
        x = self._maybe_inject(x, t, model_kwargs, use_inpainting_injection, injection_schedule,
                               use_cumulative_noise)
        if denoised_fn is not None or cond_fn is not None:
            out = self.p_mean_variance(model, x, t, clip_denoised, denoised_fn, model_kwargs)
            noise = torch.randn_like(x)
            nz = (t != 0).float().view(-1, *([1] * (x.dim() - 1)))
            if cond_fn is not None:
                out["mean"] = self.condition_mean(cond_fn, out, x, t, model_kwargs=model_kwargs)
            return {"sample": out["mean"] + nz * torch.exp(0.5 * out["log_variance"]) * noise,
                    "pred_xstart": out["pred_xstart"]}
        model_output = self._call_model(model, x, t, model_kwargs)
        noise = torch.randn_like(x)
        r = self._step(L.STEP_UPDATE_ONLY, x, t_dev=t, model_out=model_output, z=noise, ddim=False,
                       clip=clip_denoised, want_sample=True, want_x0=True)
        return {"sample": r["sample"], "pred_xstart": r["pred_xstart"]}

    def ddim_sample(self, model, x, t, clip_denoised=True, denoised_fn=None, cond_fn=None, model_kwargs=None,
                    eta=0.0, use_inpainting_injection=False, injection_schedule="all",
                    use_cumulative_noise=True):
        """One DDIM step with optional pre-model injection (`:447-485`)."""
        x = self._maybe_inject(x, t, model_kwargs, use_inpainting_injection, injection_schedule,
                               use_cumulative_noise)
        if denoised_fn is not None or cond_fn is not None:
            out = self.p_mean_variance(model, x, t, clip_denoised, denoised_fn, model_kwargs)
            if cond_fn is not None:
                out = self.condition_score(cond_fn, out, x, t, model_kwargs=model_kwargs)
            eps = self._predict_eps_from_xstart(x, t, out["pred_xstart"])
            ab = _extract_into_tensor(self.alphas_cumprod, t, x.shape)
            abp = _extract_into_tensor(self.alphas_cumprod_prev, t, x.shape)
            sigma = eta * torch.sqrt((1 - abp) / (1 - ab)) * torch.sqrt(1 - ab / abp)
            noise = torch.randn_like(x)
            mean_pred = out["pred_xstart"] * torch.sqrt(abp) + torch.sqrt(1 - abp - sigma ** 2) * eps
            nz = (t != 0).float().view(-1, *([1] * (x.dim() - 1)))
            return {"sample": mean_pred + nz * sigma * noise, "pred_xstart": out["pred_xstart"]}
        model_output = self._call_model(model, x, t, model_kwargs)
        noise = torch.randn_like(x)                      # always drawn, even for eta = 0 (:478)
        r = self._step(L.STEP_UPDATE_ONLY, x, t_dev=t, model_out=model_output, z=noise if eta != 0.0 else None,
                       ddim=True, eta=eta, clip=clip_denoised, want_sample=True, want_x0=True)
        return {"sample": r["sample"], "pred_xstart": r["pred_xstart"]}

    # ------------------------------------------------------------------ loops
    def _x_T(self, model, shape, noise, device, seeds=None):
        """The device default and x_T of every loop: `noise`, or one randn(shape) draw, or with `seeds` (checked CPU
        tensor) the seeded draw (XT, 0); FidmError for a CPU x_T.  Returns (device, x_T, seeds on the device)."""
        if device is None:
            device = next(model.parameters()).device
        assert isinstance(shape, (tuple, list))
        if seeds is not None:
            seeds = seeds.to(device)
        if noise is not None:
            img = noise
        elif seeds is None:
            img = torch.randn(*shape, device=device)
        else:
            img = seeded.randn(seeds, shape, L.NOISE_XT, 0)
        L.require_cuda(img)
        return device, img, seeds

    def _loop_start(self, model, shape, noise, device, mk, gt, keep, t_first, injection_schedule, cumulative, seeds):
        """Prologue of the fused loops (K4, K6, K7).  gt / keep: the known region, None without injection; the
        injection noise is drawn like `gt` as given.  Returns (x, rng, evaluate, stem, bufs):
        x, the fp32 contiguous state the first evaluation (at t_first) sees, after the injection on x_T;
        rng, the loop's noise: rng.inject(ts) at timestep ts, rng.step(x, k) and rng.undo(x, k) of evaluation k -- torch
        tensors, or with `seeds` seeded.Draw values that the launchers turn into seeded launches;
        evaluate(x, t), the model output at t; stem, the engine plan's (network input, timestep tensor) or None;
        bufs, two state buffers to alternate between on the plan, or None (x is bufs[0] after an injection on the plan)."""
        if seeds is not None:
            seeds = seeded.check_seeds(seeds, shape[0])
        device, img, seeds = self._x_T(model, shape, noise, device, seeds)
        rng = _TorchDraws(self, gt, cumulative) if seeds is None else seeded.SeededDraws(seeds, cumulative)

        # Step-boundary fusion: when `model` is this package's model_fn (train_inpainting.InpaintingModelFn around a
        # DiffusionInpaintingModel), the step kernels write the next evaluation's stem channels and timestep themselves
        # and the UNet output is read where the head left it: a step is [graph replay, randn, kernel] -- no pack, no
        # copies, no clone.
        plan = None
        fused_plan = getattr(model, "fused_plan", None)
        if fused_plan is not None and os.environ.get("FIDM_FUSED_STEP", "1") != "0":
            plan = fused_plan(tuple(shape), img, self._t_value(t_first), mk)

        def evaluate(x, t):
            if plan is not None:
                return plan.run()                            # stem input and timestep are already in place
            return self._call_model(model, x, torch.full((shape[0],), t, device=device, dtype=torch.long), mk)

        # the kernels write the state in NCHW order: buffers allocated like a channels_last x_T would scramble it
        img = _f32(img)
        stem = (plan.x_in, plan.t_in) if plan is not None else None
        bufs = [torch.empty_like(img), torch.empty_like(img)] if plan is not None else None
        if gt is None or self._injection_gated(t_first, injection_schedule):
            return img, rng, evaluate, stem, bufs
        x = self._step(L.STEP_INJECT_ONLY, img, t_inject=t_first, gt=gt, keep=keep, inject_noise=rng.inject(t_first),
                       cumulative=cumulative, want_next=True, stem=stem, next_buf=bufs[0] if bufs else None)["x_next"]
        return x, rng, evaluate, stem, bufs

    def _update_inject(self, x, i, model_output, z, gt, keep, inj_noise, stem, next_buf, *, ddim, eta, clip,
                       cumulative, injection_schedule, want_out):
        """One K4 launch of a fused loop: the update at i, the injection at i - 1 unless it is gated, and the next
        evaluation's stem input.  `z` is drawn by the caller, before the injection noise.  Returns (K4's outputs, the
        state the next evaluation sees)."""
        nxt = i - 1
        do_inj = gt is not None and nxt >= 0 and not self._injection_gated(nxt, injection_schedule)
        fused = stem is not None
        r = self._step(L.STEP_UPDATE_INJECT if do_inj else L.STEP_UPDATE_ONLY, x, t=i, t_inject=nxt,
                       model_out=model_output, z=z if (not ddim or eta != 0.0) else None,
                       gt=gt if do_inj else None, keep=keep if do_inj else None,
                       inject_noise=inj_noise(nxt) if do_inj else None,
                       ddim=ddim, eta=eta, clip=clip, cumulative=cumulative,
                       want_sample=want_out or (not do_inj and not fused), want_x0=want_out,
                       want_next=do_inj or fused,
                       stem=stem if nxt >= 0 else None, t_next=self._t_value(nxt) if nxt >= 0 else None,
                       next_buf=next_buf)
        return r, (r["x_next"] if (do_inj or fused) else r["sample"])

    def _last_sample(self, loop):
        """Runs a loop generator to its end on a fresh injection-noise cache and returns its last "sample"."""
        self.clear_gt_noise_cache()
        final = None
        for final in loop:
            pass
        return final["sample"]

    def _loop(self, ddim, model, shape, noise, clip_denoised, denoised_fn, cond_fn, model_kwargs, device,
              progress, eta, use_inpainting_injection, injection_schedule, use_cumulative_noise,
              progressive, seeds):
        """Shared fused loop: per step one model call and ONE K4 launch ([update t] -> [inject t-1])."""
        indices = list(range(self.num_timesteps))[::-1]
        if progress and tqdm is not None:
            indices = tqdm(indices)
        mk = model_kwargs

        if denoised_fn is not None or cond_fn is not None:       # unfused compatibility path
            if seeds is not None:
                raise NotImplementedError("seeds are not supported with denoised_fn / cond_fn: that unfused path "
                                          "draws from torch's generator")
            device, img, _ = self._x_T(model, shape, noise, device)
            step = self.ddim_sample if ddim else self.p_sample
            extra = {"eta": eta} if ddim else {}
            for i in indices:
                t = torch.tensor([i] * shape[0], device=device)
                with torch.no_grad():
                    out = step(model, img, t, clip_denoised=clip_denoised, denoised_fn=denoised_fn,
                               cond_fn=cond_fn, model_kwargs=mk, use_inpainting_injection=use_inpainting_injection,
                               injection_schedule=injection_schedule, use_cumulative_noise=use_cumulative_noise,
                               **extra)
                    yield out
                    img = out["sample"]
            return

        gt, keep = _known_region(mk, use_inpainting_injection)
        x, rng, evaluate, stem, bufs = self._loop_start(model, shape, noise, device, mk, gt, keep,
                                                       self.num_timesteps - 1, injection_schedule,
                                                       use_cumulative_noise, seeds)
        with torch.no_grad():
            for k, i in enumerate(indices):
                model_output = evaluate(x, i)
                z = rng.step(x, k)                                   # RNG order: z_t, then n_{t-1}
                want_out = progressive or i == 0
                r, x = self._update_inject(x, i, model_output, z, gt, keep, rng.inject, stem,
                                           bufs[(k + 1) & 1] if bufs else None, ddim=ddim, eta=eta, clip=clip_denoised,
                                           cumulative=use_cumulative_noise, injection_schedule=injection_schedule,
                                           want_out=want_out)
                if want_out:
                    yield {"sample": r["sample"], "pred_xstart": r["pred_xstart"]}

    def p_sample_loop_progressive(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None,
                                  cond_fn=None, model_kwargs=None, device=None, progress=False,
                                  use_inpainting_injection=False, injection_schedule="all",
                                  use_cumulative_noise=True, seeds=None):
        """Generator over the per-step dicts {"sample", "pred_xstart"} (`:415-445`)."""
        yield from self._loop(False, model, shape, noise, clip_denoised, denoised_fn, cond_fn, model_kwargs,
                              device, progress, 0.0, use_inpainting_injection, injection_schedule,
                              use_cumulative_noise, True, seeds)

    def ddim_sample_loop_progressive(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None,
                                     cond_fn=None, model_kwargs=None, device=None, progress=False, eta=0.0,
                                     use_inpainting_injection=False, injection_schedule="all",
                                     use_cumulative_noise=True, seeds=None):
        """Generator over the per-step dicts {"sample", "pred_xstart"} (`:508-538`)."""
        yield from self._loop(True, model, shape, noise, clip_denoised, denoised_fn, cond_fn, model_kwargs,
                              device, progress, eta, use_inpainting_injection, injection_schedule,
                              use_cumulative_noise, True, seeds)

    def p_sample_loop(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None, cond_fn=None,
                      model_kwargs=None, device=None, progress=False, use_inpainting_injection=False,
                      injection_schedule="all", use_cumulative_noise=True, seeds=None):
        """DDPM sampling with optional known-region injection (`:390-413`).  seeds: one uint64 per image (a sequence
        of ints or an int64 / uint64 tensor) -- every noise value is then generated from the image's own seed inside
        the sampler kernels (seeded.py), so an image's result does not depend on its batch; torch's generator is not
        used.  The same holds for every loop of this class."""
        return self._last_sample(self._loop(False, model, shape, noise, clip_denoised, denoised_fn, cond_fn,
                                            model_kwargs, device, progress, 0.0, use_inpainting_injection,
                                            injection_schedule, use_cumulative_noise, False, seeds))

    def ddim_sample_loop(self, model, shape, noise=None, clip_denoised=True, denoised_fn=None, cond_fn=None,
                         model_kwargs=None, device=None, progress=False, eta=0.0,
                         use_inpainting_injection=False, injection_schedule="all", use_cumulative_noise=True,
                         seeds=None):
        """DDIM sampling with optional known-region injection (`:487-506`); seeds as in p_sample_loop."""
        return self._last_sample(self._loop(True, model, shape, noise, clip_denoised, denoised_fn, cond_fn,
                                            model_kwargs, device, progress, eta, use_inpainting_injection,
                                            injection_schedule, use_cumulative_noise, False, seeds))

    # ------------------------------------------------------------------ DPM-Solver++ multistep (K6)
    def _dpm_table(self, device, steps, order, cumulative):
        key = ("dpm", str(device), int(steps), int(order), bool(cumulative))
        if key not in self._coef_cache:
            self._coef_cache[key] = dpm_solver.coefficient_table(self, steps, order, cumulative).to(device)
        return self._coef_cache[key]

    def _multistep(self, tab, step, x, model_out, *, m_prev=None, want_next=True, clip=True, gt=None, keep=None,
                   inject_noise=None, stem=None, t_next=None):
        """One K6 launch with row `step` of the table `tab`: returns (m_k, state at t_{k+1} or None).  m_prev selects
        the second-order update; gt / keep / inject_noise the injection; stem = (NHWC network input, timestep tensor)
        of an engine plan receives the new state and `t_next` (step-boundary fusion, as in _step).  inject_noise may be a
        seeded.Draw (a seeded launch)."""
        sn = seeded.launch_args(None, inject_noise)
        if sn is not None:
            inject_noise = None
        L.require_cuda(x, model_out, m_prev, gt, keep, inject_noise)
        B, Cn = x.shape[0], x.shape[1]
        model_out = _f32(model_out)
        assert model_out.shape[0] == B and model_out.shape[2:] == x.shape[2:], tuple(model_out.shape)
        a = L.MultistepArgs()
        a.batch, a.channels, a.hw = B, Cn, x.numel() // (B * Cn)
        a.mean_type, a.out_channels, a.clip_denoised = _MEAN_CODE[self.model_mean_type], model_out.shape[1], int(bool(clip))
        a.steps, a.step = tab.shape[0], int(step)
        m = torch.empty_like(x)
        nxt = torch.empty_like(x) if want_next else None
        a.coef, a.x, a.model_out, a.m_prev, a.m_out, a.x_next = (L.ptr(v) for v in (tab, x, model_out, m_prev, m, nxt))
        a.mask_channels = 1
        if gt is not None:
            a.inject = 1
            gt, keep, inject_noise = _set_injection(a, x, gt, keep, inject_noise)
        _set_stem(a, stem, t_next)
        if sn is None:
            L.check(L.lib().fidm_multistep_step(C.byref(a), L.stream()), "multistep_step")
        else:
            L.check(L.lib().fidm_multistep_step_seeded(C.byref(a), C.byref(sn), L.stream()), "multistep_step_seeded")
        return m, nxt

    def _dpm_solver_loop(self, model, shape, steps, order, noise, clip_denoised, model_kwargs, device, progress,
                         use_inpainting_injection, injection_schedule, use_cumulative_noise, seeds):
        """Per evaluation one model call and ONE K6 launch (x0 prediction, update, injection, next stem input)."""
        if self.model_mean_type == ModelMeanType.PREVIOUS_X:
            raise NotImplementedError("DPM-Solver++ needs an eps or x0 prediction; PREVIOUS_X models are not supported")
        grid = dpm_solver.timestep_grid(self.num_timesteps, steps)
        orders = dpm_solver.step_orders(steps, order)
        mk = model_kwargs
        gt, keep = _known_region(mk, use_inpainting_injection)
        if gt is not None:           # once per loop; the injection noise is drawn like the fp32 copy
            gt, keep = _f32(gt), _f32(keep)
        x, rng, evaluate, stem, _ = self._loop_start(model, shape, noise, device, mk, gt, keep, int(grid[0]),
                                                      injection_schedule, use_cumulative_noise, seeds)
        tab = self._dpm_table(x.device, steps, order, use_cumulative_noise)
        ks = range(steps)
        if progress and tqdm is not None:
            ks = tqdm(ks)
        with torch.no_grad():
            m_prev = None
            for k in ks:
                model_output = evaluate(x, int(grid[k]))
                if k == steps - 1:                               # t = 0: the sample is the x0 prediction
                    m, _ = self._multistep(tab, k, x, model_output, want_next=False, clip=clip_denoised)
                    yield {"sample": m, "pred_xstart": m}
                    break
                nxt = int(grid[k + 1])
                do_inj = gt is not None and not self._injection_gated(nxt, injection_schedule)
                m, x = self._multistep(tab, k, x, model_output, m_prev=m_prev if orders[k] == 2 else None,
                                       clip=clip_denoised, gt=gt if do_inj else None, keep=keep if do_inj else None,
                                       inject_noise=rng.inject(nxt) if do_inj else None, stem=stem,
                                       t_next=self._t_value(nxt))
                m_prev = m
                yield {"sample": x, "pred_xstart": m}

    def dpm_solver_sample_loop_progressive(self, model, shape, steps=20, order=2, noise=None, clip_denoised=True,
                                           model_kwargs=None, device=None, progress=False,
                                           use_inpainting_injection=False, injection_schedule="all",
                                           use_cumulative_noise=True, seeds=None):
        """Generator over one dict {"sample", "pred_xstart"} per model evaluation of dpm_solver_sample_loop:
        "sample" is the state the next evaluation sees (after the injection), and the x0 prediction at t = 0 for the
        last one; "pred_xstart" is the x0 prediction of that evaluation.  Every yielded tensor is a fresh buffer."""
        yield from self._dpm_solver_loop(model, shape, steps, order, noise, clip_denoised, model_kwargs, device,
                                         progress, use_inpainting_injection, injection_schedule, use_cumulative_noise,
                                         seeds)

    def dpm_solver_sample_loop(self, model, shape, steps=20, order=2, noise=None, clip_denoised=True,
                               model_kwargs=None, device=None, progress=False, use_inpainting_injection=False,
                               injection_schedule="all", use_cumulative_noise=True, seeds=None):
        """DPM-Solver++ (multistep, `order` 1 or 2) in `steps` model evaluations on the timesteps
        round(linspace(T - 1, 0, steps)) of this diffusion's own table, with the class path's known-region injection
        (on x_T, then after every update) and RNG draw order (randn(shape), then one injection noise per injection;
        the solver itself draws nothing; seeds as in p_sample_loop).  Returns the x0 prediction at t = 0."""
        return self._last_sample(self._dpm_solver_loop(model, shape, steps, order, noise, clip_denoised, model_kwargs,
                                                       device, progress, use_inpainting_injection, injection_schedule,
                                                       use_cumulative_noise, seeds))

    # ------------------------------------------------------------------ RePaint resampling (K4 + K7)
    def _resample(self, x, u, undo_a, undo_s, *, t_inject=None, gt=None, keep=None, inject_noise=None, cumulative=True,
                  stem=None, t_next=None, next_buf=None):
        """One K7 launch: x' = undo_a*x + undo_s*u, then (t_inject not None) the injection at t_inject with the class
        table's coefficients; stem = (NHWC network input, timestep tensor) of an engine plan receives the new state and
        `t_next` (step-boundary fusion, as in _step).  u / inject_noise may be seeded.Draw values (a seeded launch).
        Returns the new state (next_buf when given)."""
        sn = seeded.launch_args(u, inject_noise)
        if sn is not None:
            u = inject_noise = None
        L.require_cuda(x, u, gt, keep, inject_noise)
        x, u = _f32(x), _f32(u)
        assert u is None or u.shape == x.shape, (tuple(u.shape), tuple(x.shape))
        B, Cn = x.shape[0], x.shape[1]
        a = L.ResampleArgs()
        a.batch, a.channels, a.hw = B, Cn, x.numel() // (B * Cn)
        a.undo_a, a.undo_s = float(undo_a), float(undo_s)
        out = next_buf if next_buf is not None else torch.empty_like(x)
        a.x, a.noise, a.x_next = L.ptr(x), L.ptr(u), L.ptr(out)
        a.mask_channels = 1
        if t_inject is not None:
            gt, keep, inject_noise = _set_injection(a, x, gt, keep, inject_noise)
            if "host" not in self._coef_cache:
                self._coef_cache["host"] = self.coefficient_table(0.0)
            cls = self._coef_cache["host"]
            ia, is_ = (L.C_SQRT_AB, L.C_SQRT_1MAB) if cumulative else (L.C_SQRT_AB_F32, L.C_SQRT_1MAB_F32)
            a.inject = 1
            a.inject_a, a.inject_s = float(cls[t_inject, ia]), float(cls[t_inject, is_])
        _set_stem(a, stem, t_next)
        if sn is None:
            L.check(L.lib().fidm_resample_undo(C.byref(a), L.stream()), "resample_undo")
        else:
            L.check(L.lib().fidm_resample_undo_seeded(C.byref(a), C.byref(sn), L.stream()), "resample_undo_seeded")
        return out

    def _repaint_plan(self, jump_length, jump_n_sample, model_kwargs, use_inpainting_injection, shape, seeds):
        """The evaluation plan, after every argument check (raises ValueError before any RNG draw or GPU work)."""
        plan = repaint.evaluation_plan(self.alphas_cumprod, jump_length, jump_n_sample)
        if seeds is not None:
            seeded.check_seeds(seeds, shape[0])
        if not use_inpainting_injection:
            raise ValueError("RePaint resampling needs the known-region injection (use_inpainting_injection=True)")
        if not model_kwargs or model_kwargs.get("gt") is None or model_kwargs.get("gt_keep_mask") is None:
            raise ValueError("RePaint resampling needs model_kwargs with 'gt' and 'gt_keep_mask'")
        return plan

    def _repaint_loop(self, evals, model, shape, noise, clip_denoised, model_kwargs, device, progress,
                      injection_schedule, use_cumulative_noise, progressive, seeds):
        """Per evaluation one model call and one K4 launch; when a jump follows the evaluation, K4 only updates and
        one K7 launch re-noises to t_up, injects at t_up and writes the next stem input."""
        mk = model_kwargs
        gt, keep = mk["gt"], mk["gt_keep_mask"]
        x, rng, evaluate, stem, bufs = self._loop_start(model, shape, noise, device, mk, gt, keep, evals[0].t,
                                                       injection_schedule, use_cumulative_noise, seeds)
        if progress and tqdm is not None:
            evals = tqdm(evals)
        with torch.no_grad():
            for k, (i, t_up, undo_a, undo_s) in enumerate(evals):
                model_output = evaluate(x, i)
                z = rng.step(x, k)                                   # RNG order: z_t, [u], then n of the next t
                want_out = progressive or i == 0
                nbuf = bufs[(k + 1) & 1] if bufs else None
                if t_up is None:                                     # as _loop's DDPM step
                    r, x = self._update_inject(x, i, model_output, z, gt, keep, rng.inject, stem, nbuf, ddim=False,
                                               eta=0.0, clip=clip_denoised, cumulative=use_cumulative_noise,
                                               injection_schedule=injection_schedule, want_out=want_out)
                else:
                    r = self._step(L.STEP_UPDATE_ONLY, x, t=i, model_out=model_output, z=z, ddim=False,
                                   clip=clip_denoised, want_sample=True, want_x0=want_out)
                    u = rng.undo(x, k)
                    do_inj = not self._injection_gated(t_up, injection_schedule)
                    x = self._resample(r["sample"], u, undo_a, undo_s, t_inject=t_up if do_inj else None,
                                       gt=gt, keep=keep, inject_noise=rng.inject(t_up) if do_inj else None,
                                       cumulative=use_cumulative_noise, stem=stem, t_next=self._t_value(t_up),
                                       next_buf=nbuf)
                if want_out:
                    yield {"sample": r["sample"], "pred_xstart": r["pred_xstart"], "t": i}

    def repaint_sample_loop_progressive(self, model, shape, jump_length=10, jump_n_sample=10, noise=None,
                                        clip_denoised=True, model_kwargs=None, device=None, progress=False,
                                        use_inpainting_injection=True, injection_schedule="all",
                                        use_cumulative_noise=True, seeds=None):
        """Generator over one dict {"sample", "pred_xstart", "t"} per model evaluation of repaint_sample_loop:
        "sample" is the DDPM output of the evaluation at timestep "t", before any undo or injection.  The arguments
        are checked when this is called, before the first draw."""
        evals = self._repaint_plan(jump_length, jump_n_sample, model_kwargs, use_inpainting_injection, shape, seeds)
        return self._repaint_loop(evals, model, shape, noise, clip_denoised, model_kwargs, device, progress,
                                  injection_schedule, use_cumulative_noise, True, seeds)

    def repaint_sample_loop(self, model, shape, jump_length=10, jump_n_sample=10, noise=None, clip_denoised=True,
                            model_kwargs=None, device=None, progress=False, use_inpainting_injection=True,
                            injection_schedule="all", use_cumulative_noise=True, seeds=None):
        """DDPM sampling with RePaint resampling (Lugmayr et al. 2022): the class path's DDPM step and known-region
        injection, on RePaint's jump schedule (repaint.py) -- every `jump_length` timesteps the state is re-noised
        back up `jump_length` levels and denoised again, `jump_n_sample - 1` times, so that the hole can agree with
        the known region.  T + (jump_n_sample - 1) * jump_length * len(range(0, T - jump_length, jump_length)) model
        evaluations.  RNG draw order: randn(shape), the injection noise at T - 1, then per evaluation the step noise,
        the undo noise if a jump follows, and the injection noise of the next evaluation (with use_cumulative_noise
        a revisited timestep reuses its cached noise; seeds as in p_sample_loop).  Returns the sample at t = 0, not
        re-blended."""
        evals = self._repaint_plan(jump_length, jump_n_sample, model_kwargs, use_inpainting_injection, shape, seeds)
        return self._last_sample(self._repaint_loop(evals, model, shape, noise, clip_denoised, model_kwargs, device,
                                                    progress, injection_schedule, use_cumulative_noise, False, seeds))

    # ------------------------------------------------------------------ continuous batching (K8, K9, K10)
    def continuous_sampler(self, model, slots=8, image_size=(256, 256), sampler="ddim", eta=0.0, clip_denoised=True,
                           use_inpainting_injection=True, injection_schedule="all", use_cumulative_noise=True,
                           channels=3, device=None, denoised_fn=None, cond_fn=None):
        """A continuous-batching sampler (continuous.py) over `slots` images of `image_size`: requests of one image
        each, submitted with their own seed at any time, each run through ddim_sample_loop ("ddim", any eta) or
        p_sample_loop ("ddpm") on this diffusion's T timesteps, its result bit-identical to that loop run alone with
        seeds=[seed].  Arguments are checked here and at submit, before any launch."""
        from .continuous import ContinuousSampler
        return ContinuousSampler(self, model, slots=slots, image_size=image_size, sampler=sampler, eta=eta,
                                 clip_denoised=clip_denoised, use_inpainting_injection=use_inpainting_injection,
                                 injection_schedule=injection_schedule, use_cumulative_noise=use_cumulative_noise,
                                 channels=channels, device=device, denoised_fn=denoised_fn, cond_fn=cond_fn)

    def continuous_dpm_solver_sampler(self, model, slots=8, image_size=(256, 256), steps=20, order=2, clip_denoised=True,
                                      use_inpainting_injection=True, injection_schedule="all",
                                      use_cumulative_noise=True, channels=3, device=None):
        """continuous_sampler for DPM-Solver++: every request takes `steps` model evaluations (multistep `order` 1 or
        2), its result bit-identical to dpm_solver_sample_loop(model, (1, C, H, W), steps=steps, order=order, ...,
        seeds=[seed]) run alone.  Same submit / step / pending / drain surface; arguments are checked here and at
        submit, before any launch."""
        from .continuous import ContinuousDPMSolverSampler
        return ContinuousDPMSolverSampler(self, model, slots=slots, image_size=image_size, steps=steps, order=order,
                                          clip_denoised=clip_denoised, use_inpainting_injection=use_inpainting_injection,
                                          injection_schedule=injection_schedule,
                                          use_cumulative_noise=use_cumulative_noise, channels=channels, device=device)

    def continuous_repaint_sampler(self, model, slots=8, image_size=(256, 256), jump_length=10, jump_n_sample=10,
                                   clip_denoised=True, use_inpainting_injection=True, injection_schedule="all",
                                   use_cumulative_noise=True, channels=3, device=None):
        """continuous_sampler for RePaint resampling: every request takes the same
        len(repaint.evaluation_plan(self.alphas_cumprod, jump_length, jump_n_sample)) model evaluations, its result
        bit-identical to repaint_sample_loop(model, (1, C, H, W), jump_length, jump_n_sample, ..., seeds=[seed]) run
        alone.  Same submit / step / pending / drain surface; arguments are checked here and at submit, before any
        launch."""
        from .continuous import ContinuousRePaintSampler
        return ContinuousRePaintSampler(self, model, slots=slots, image_size=image_size, jump_length=jump_length,
                                        jump_n_sample=jump_n_sample, clip_denoised=clip_denoised,
                                        use_inpainting_injection=use_inpainting_injection,
                                        injection_schedule=injection_schedule,
                                        use_cumulative_noise=use_cumulative_noise, channels=channels, device=device)

    def sample_with_advanced_inpainting(self, model, shape, gt=None, gt_keep_mask=None, use_ddim=True, eta=0.0,
                                        progress=True, device=None, injection_schedule="all",
                                        use_cumulative_noise=True):
        """Convenience entry (`:640-700`): builds model_kwargs {gt, gt_keep_mask, masked_image, mask}.

        As in the reference the kwargs are forwarded verbatim to `model`, so `model` must accept
        (and may ignore) `gt` / `gt_keep_mask` -- e.g. `train_inpainting.InpaintingModelFn`."""
        if device is None:
            device = next(model.parameters()).device
        mk, inject = {}, False
        if gt is not None and gt_keep_mask is not None:
            mk = {"gt": gt, "gt_keep_mask": gt_keep_mask,
                  "masked_image": gt * gt_keep_mask, "mask": 1 - gt_keep_mask}
            inject = True
        common = dict(model=model, shape=shape, device=device, progress=progress, model_kwargs=mk,
                      use_inpainting_injection=inject, injection_schedule=injection_schedule,
                      use_cumulative_noise=use_cumulative_noise)
        if use_ddim:
            return self.ddim_sample_loop(eta=eta, **common)
        return self.p_sample_loop(**common)

    # ------------------------------------------------------------------ out of scope
    def training_losses(self, *a, **k):
        raise NotImplementedError("training is outside the sampling path this package implements")

    _vb_terms_bpd = training_losses
