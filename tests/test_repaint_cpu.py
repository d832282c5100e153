"""CPU: RePaint resampling host logic -- the jump schedule and the evaluation plan against oracle/repaint_oracle.py, the
collapsed undo coefficients, argument checks before any draw, the C struct mirror, and the harmonization RePaint buys on
the correlated-Gaussian analytic model (float64 oracle)."""
import math
import os
import re

import numpy as np
import pytest
import torch

import fidm_b200 as F
from fidm_b200 import _lib, repaint
from oracle import repaint_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CASES = [(100, 10, 10), (1000, 10, 10), (7, 3, 2), (100, 10, 1), (1000, 10, 1), (10, 9, 3), (5, 1, 3), (250, 7, 4)]


@pytest.mark.parametrize("T,jl,jn", CASES)
def test_schedule_equals_the_paper_restatement(T, jl, jn):
    assert repaint.jump_schedule(T, jl, jn) == O.schedule(T, jl, jn)


@pytest.mark.parametrize("T,jl,jn", CASES)
def test_plan_follows_the_schedule(T, jl, jn):
    ab = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine").alphas_cumprod
    plan = repaint.evaluation_plan(ab, jl, jn)
    assert len(plan) == T + (jn - 1) * jl * len(range(0, T - jl, jl))
    # replaying the plan (one step down per evaluation, one collapsed undo per jump) visits the schedule's levels
    walk = []
    for e in plan:
        walk.append(e.t)
        if e.t_up is not None:
            assert e.t_up == e.t - 1 + jl
            walk += list(range(e.t - 1, e.t_up))
    walk.append(-1)
    assert walk == O.schedule(T, jl, jn)
    assert plan[-1].t == 0 and plan[-1].t_up is None
    if jn == 1:
        assert [e.t for e in plan] == list(range(T - 1, -1, -1)) and all(e.t_up is None for e in plan)


def test_evaluation_count_of_the_default_setting():
    ab = F.create_gaussian_diffusion(steps=100, noise_schedule="cosine").alphas_cumprod
    assert len(repaint.evaluation_plan(ab, 10, 10)) == 910


@pytest.mark.parametrize("sched", ["linear", "cosine", "quadratic"])
def test_collapsed_undo_equals_the_product_of_per_step_factors(sched):
    d = F.create_gaussian_diffusion(steps=1000, noise_schedule=sched)
    b = d.betas
    n = 0
    for e in repaint.evaluation_plan(d.alphas_cumprod, 10, 3):
        if e.t_up is None:
            continue
        a, s = repaint.undo_coefficients(d.alphas_cumprod, e.t, e.t_up)
        prod = math.prod(1.0 - b[k] for k in range(e.t, e.t_up + 1))
        assert abs(a - math.sqrt(prod)) <= 1e-12 and abs(s - math.sqrt(1.0 - prod)) <= 1e-12, (e.t, e.t_up)
        assert (e.undo_a, e.undo_s) == (float(np.float32(a)), float(np.float32(s)))
        n += 1
    assert n == 2 * len(range(0, 1000 - 10, 10))


def test_collapsed_undo_noise_reproduces_the_step_by_step_undo():
    b = F.create_gaussian_diffusion(steps=100, noise_schedule="linear").betas
    g = torch.Generator().manual_seed(0)
    x = torch.randn(3, 64, generator=g, dtype=torch.float64)
    zs = [torch.randn(3, 64, generator=g, dtype=torch.float64) for _ in range(10)]
    want = x.clone()
    for s, z in zip(range(31, 41), zs):
        want = math.sqrt(1 - b[s]) * want + math.sqrt(b[s]) * z
    a, s = repaint.undo_coefficients(np.cumprod(1 - b), 31, 40)
    got = a * x + s * O.collapse_undo_noise(b, 31, 40, zs)
    assert (got - want).abs().max().item() < 1e-12


@pytest.mark.parametrize("kw", [dict(jump_length=0), dict(jump_length=100), dict(jump_length=2.0),
                                dict(jump_length="10"), dict(jump_length=True), dict(jump_n_sample=0),
                                dict(jump_n_sample=1.0), dict(jump_n_sample="3"), dict(jump_n_sample=True),
                                dict(jump_n_sample=None), dict(use_inpainting_injection=False),
                                dict(model_kwargs=None), dict(model_kwargs={"gt": torch.zeros(1, 3, 8, 8)}),
                                dict(model_kwargs={"gt_keep_mask": torch.ones(1, 1, 8, 8)})])
def test_invalid_arguments_raise_before_any_draw(kw):
    d = F.create_gaussian_diffusion(steps=100, noise_schedule="linear")
    fn = lambda x, t, **k: torch.zeros_like(x)  # noqa: E731
    args = dict(model_kwargs={"gt": torch.zeros(1, 3, 8, 8), "gt_keep_mask": torch.ones(1, 1, 8, 8)}, device="cpu")
    args.update(kw)
    state = torch.get_rng_state()
    with pytest.raises(ValueError):
        d.repaint_sample_loop(fn, (1, 3, 8, 8), **args)
    with pytest.raises(ValueError):
        d.repaint_sample_loop_progressive(fn, (1, 3, 8, 8), **args)
    assert torch.equal(torch.get_rng_state(), state)


def test_no_cpu_fallback():
    d = F.create_gaussian_diffusion(steps=100, noise_schedule="linear")
    mk = {"gt": torch.zeros(1, 3, 8, 8), "gt_keep_mask": torch.ones(1, 1, 8, 8)}
    with pytest.raises(_lib.FidmError):
        d.repaint_sample_loop(lambda x, t, **k: torch.zeros_like(x), (1, 3, 8, 8), model_kwargs=mk, device="cpu")


def test_resample_struct_matches_header_field_order():
    text = open(os.path.join(ROOT, "include", "fidm_b200.h")).read()
    body = re.search(r"typedef struct fidm_resample_args \{(.*?)\} fidm_resample_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        decl = re.sub(r"^(const\s+)?(int32_t|int64_t|float|double|void)\s*\**", "", decl)
        for part in decl.split(","):
            names.append(re.sub(r"\[.*\]", "", part.replace("*", "").strip()))
    assert names == [f[0] for f in _lib.ResampleArgs._fields_]
    assert "fidm_resample_undo" in _lib.SYMBOLS


# ------------------------------------------------------------------------------------------ harmonization
def harmonization(jl, jn, seed, B=4000):
    """Hole-mean RMS error and hole-covariance relative error of RePaint(jl, jn) (jn = 1: plain injection) on the 8x8
    one-channel analytic model, 100-step linear table, FIXED_SMALL, left half known."""
    d = F.create_gaussian_diffusion(steps=100, noise_schedule="linear", sigma_small=True)
    am = O.CorrelatedGaussian(d.alphas_cumprod, 8, 8)
    g = torch.Generator().manual_seed(seed)
    gt = am.sample_prior(1, g)
    keep = torch.zeros(1, 1, 8, 8, dtype=torch.float64)
    keep[..., :4] = 1
    cache = {}

    def noise(kind, t, visit):
        if (kind, t, visit) not in cache or kind != "inject":
            cache[(kind, t, visit)] = torch.randn(B, 1, 8, 8, generator=g, dtype=torch.float64)
        return cache[(kind, t, visit)]

    x_T = torch.randn(B, 1, 8, 8, generator=g, dtype=torch.float64)
    out = O.sample_loop(d.betas, am.eps, x_T, jl, jn, gt=gt, keep=keep, noise=noise)
    mean, cov = am.hole_conditional(gt[0], keep[0])
    return O.harmonization_errors(out, keep, mean, cov)


@pytest.mark.parametrize("seed", [1, 2])
def test_repaint_harmonizes_the_hole_on_the_analytic_model(seed):
    plain = harmonization(10, 1, seed)
    rp = harmonization(10, 10, seed)
    print("seed %d: plain injection mean RMS %.4f cov %.4f | RePaint(10, 10) mean RMS %.4f cov %.4f"
          % (seed, *plain, *rp))
    assert plain[1] >= 0.25, plain
    assert rp[1] <= 0.12 and rp[1] <= 0.35 * plain[1], (rp, plain)
    assert rp[0] <= 0.8 * plain[0], (rp, plain)


def test_sample_sharded_rejects_an_unknown_sampler():
    from fidm_b200.parallel import sample_sharded
    d = F.create_gaussian_diffusion(steps=100, noise_schedule="linear")
    with pytest.raises(ValueError):
        sample_sharded(d, lambda x, t, **k: x, torch.zeros(1, 3, 8, 8), torch.ones(1, 1, 8, 8), sampler="ddim50")
