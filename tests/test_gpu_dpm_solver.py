"""GPU: the DPM-Solver++ multistep sampler -- K6 (fidm_multistep_step) bit-exact against its fp32 op-order mirror, the
known region, equality with the class path's DDIM on the full grid, convergence through the public loop on the
analytic model, and the UNet end to end (fused and unfused loops, float64 CPU oracle, the 1000-step checkpoint setup)."""
import ctypes
import itertools

import pytest
import torch

from helpers import SeqRandn, class_draw_order, psnr, rel_l2, seeded_noise

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def lib():
    import fidm_b200  # noqa: F401
    from fidm_b200 import _lib as L
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    L.check(L.lib().fidm_device_supported(0), "device")
    return L


@pytest.fixture(scope="module")
def t64_weights():
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_state_dict
    cfg = F.CONFIGS["T64"]
    return cfg, synth_state_dict(cfg, seed=2)


def _diffusion(steps=1000, schedule="quadratic", **kw):
    import fidm_b200 as F
    return F.create_gaussian_diffusion(steps=steps, noise_schedule=schedule, **kw)


def _dpm_draw_order(grid, inject=True):
    """RNG draws of dpm_solver_sample_loop: x_T, then one injection noise per injection (t_0 .. t_{N-1})."""
    return [("xT", 0)] + ([("inject", int(t)) for t in grid] if inject else [])


def _model(cfg, sd, precision):
    import fidm_b200 as F
    m = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
    m.load_state_dict(sd, strict=True)
    m.to(DEV)
    m.base_model.set_precision(precision)
    return m


# ------------------------------------------------------------------------------------------ 1, 2: single launches
def test_kernel_bit_exact_against_fp32_mirror(lib):
    """Every switch of one K6 launch against oracle/dpm_solver_oracle.mirror_step, bit for bit; known pixels after an
    injection are exactly fl(fl(ia*gt) + fl(is*n)); the stem input is x_next rounded as the pack kernel rounds."""
    from fidm_b200 import dpm_solver
    from oracle import dpm_solver_oracle as O
    N, k = 10, 3
    n_cases = 0
    for order, mean, och, clip, inj, mch, (H, W), sdt in itertools.product(
            (1, 2), ("epsilon", "start_x"), (3, 6), (True, False), ("off", "cumulative", "fresh"), (1, 3),
            ((8, 8), (7, 9)), (torch.float32, torch.bfloat16, torch.float16)):
        if inj == "off" and mch == 3:
            continue
        d = _diffusion(learn_sigma=och == 6, predict_xstart=mean == "start_x")
        tab = dpm_solver.coefficient_table(d, N, order, inj != "fresh")
        g = torch.Generator().manual_seed(n_cases)
        B, C = 2, 3
        x = torch.randn(B, C, H, W, generator=g) * 3
        mo = torch.randn(B, och, H, W, generator=g) * (1.5 if mean == "start_x" else 1.0)
        mp = torch.rand(B, C, H, W, generator=g) * 2 - 1
        gt = torch.rand(B, C, H, W, generator=g) * 2 - 1
        keep = (torch.rand(B, mch, H, W, generator=g) > 0.4).float()
        n = torch.randn(B, C, H, W, generator=g)
        second = order == 2
        want_m, want_x = O.mirror_step(tab[k].tolist(), x, mo, m_prev=mp if second else None, clip=clip,
                                       mean_type=mean, gt=gt if inj != "off" else None, keep=keep, noise=n)
        x_in = torch.zeros(B, H, W, 16, device=DEV, dtype=sdt)
        t_in = torch.zeros(B, device=DEV)
        dv = [v.to(DEV) for v in (x, mo, mp, gt, keep, n)]
        m, xn = d._multistep(tab.to(DEV), k, dv[0], dv[1], m_prev=dv[2] if second else None, clip=clip,
                             gt=dv[3] if inj != "off" else None, keep=dv[4], inject_noise=dv[5],
                             stem=(x_in, t_in), t_next=37.0)
        tag = (order, mean, och, clip, inj, mch, H, W, sdt)
        assert torch.equal(m.cpu(), want_m), tag
        assert torch.equal(xn.cpu(), want_x), tag
        if inj != "off":
            known = keep.expand_as(x) == 1
            ia, is_ = (torch.tensor(v, dtype=torch.float32) for v in tab[k, lib.MS_INJ_A:].tolist())
            assert torch.equal(xn.cpu()[known], (ia * gt + is_ * n)[known]), tag
        assert torch.equal(x_in[..., :C], want_x.permute(0, 2, 3, 1).to(sdt).to(DEV)), tag
        assert not x_in[..., C:].any() and torch.equal(t_in, torch.full((B,), 37.0, device=DEV)), tag
        n_cases += 1
    # the last evaluation computes m only
    d = _diffusion(learn_sigma=True)
    tab = dpm_solver.coefficient_table(d, N, 2).to(DEV)
    x, mo = torch.randn(2, 3, 8, 8, device=DEV), torch.randn(2, 6, 8, 8, device=DEV)
    m, xn = d._multistep(tab, N - 1, x, mo, want_next=False)
    want_m, _ = O.mirror_step(tab[N - 1].tolist(), x.cpu(), mo.cpu(), update=False)
    assert xn is None and torch.equal(m.cpu(), want_m)
    assert n_cases == 2 * 2 * 2 * 2 * 5 * 2 * 3


# ------------------------------------------------------------------------------------------ 3: order 1 = DDIM
def test_order1_full_grid_equals_class_ddim(lib):
    """On the full grid (N = T) the first-order solver is DDIM (eta = 0): the two loops differ only by rounding."""
    from fidm_b200.utils.synth import synth_batch
    from oracle import dpm_solver_oracle as O
    T = 100
    d = _diffusion(T, "cosine")
    shape = (2, 3, 32, 32)
    am = O.AnalyticGaussian(d.alphas_cumprod, shape, seed=3)
    am.mu, am.s = am.mu.to(DEV), am.s.to(DEV)
    model = lambda x, t, **k: am.eps(x, int(t[0])).float()  # noqa: E731
    data = synth_batch(2, 32, seed=5, device=DEV)
    kw = dict(model_kwargs={"gt": data["gt"], "gt_keep_mask": data["gt_keep_mask"]}, device=DEV,
              use_inpainting_injection=True)
    with SeqRandn(class_draw_order(T), 11, device=DEV):
        ddim = d.ddim_sample_loop(model, shape, **kw)
    with SeqRandn(_dpm_draw_order(range(T - 1, -1, -1)), 11, device=DEV) as rng:
        dpm = d.dpm_solver_sample_loop(model, shape, steps=T, order=1, **kw)
    assert rng.i == len(rng.seq)
    err = rel_l2(dpm.cpu(), ddim.cpu())
    print("order 1 vs DDIM-100 rel-L2 %.2e" % err)
    assert err <= 1e-5, err


# ------------------------------------------------------------------------------------------ 4: convergence on the GPU
def test_convergence_through_public_loop_matches_float64_oracle(lib):
    from oracle import dpm_solver_oracle as O
    d = _diffusion(1000, "linear")
    shape = (2, 3, 32, 32)
    am = O.AnalyticGaussian(d.alphas_cumprod, shape, seed=1)
    x_T = torch.randn(*shape, generator=torch.Generator().manual_seed(2))
    ref = am.reference(x_T.double())
    am_gpu = O.AnalyticGaussian(d.alphas_cumprod, shape, seed=1)
    am_gpu.mu, am_gpu.s = am.mu.to(DEV), am.s.to(DEV)
    model = lambda x, t, **k: am_gpu.eps(x, int(t[0])).float()  # noqa: E731
    for N in (20, 40, 80):
        got = d.dpm_solver_sample_loop(model, shape, steps=N, order=2, noise=x_T.to(DEV), clip_denoised=False,
                                       device=DEV)
        cpu = O.sample_loop(d.alphas_cumprod, am.eps, x_T.double(), N, 2)
        e_gpu = ((got.cpu().double() - ref) ** 2).mean().sqrt().item()
        e_cpu = ((cpu - ref) ** 2).mean().sqrt().item()
        print("2M N=%d: RMS error GPU %.6e, float64 oracle %.6e" % (N, e_gpu, e_cpu))
        assert abs(e_gpu - e_cpu) <= 1e-5, (N, e_gpu, e_cpu)


# ------------------------------------------------------------------------------------------ 5: UNet end to end, T64
@pytest.mark.parametrize("precision,min_psnr", [("fp32", 60.0), ("bf16", 38.0)])
def test_t64_unet_2m20_fused_unfused_and_oracle(lib, t64_weights, precision, min_psnr):
    import fidm_b200 as F
    from fidm_b200 import dpm_solver
    from fidm_b200.utils.synth import synth_batch
    from oracle import dpm_solver_oracle as O
    from oracle import unet_oracle as uor
    cfg, sd = t64_weights
    d = _diffusion(1000, "quadratic", learn_sigma=True)
    N, seed = 20, 29
    shape = (2, 3, 64, 64)
    grid = dpm_solver.timestep_grid(1000, N)
    data = synth_batch(2, 64, seed=8, device=DEV)
    gt, keep = data["gt"], data["gt_keep_mask"]
    fn = F.InpaintingModelFn(_model(cfg, sd, precision))
    runs = {}
    for name, model in (("fused", fn), ("unfused", lambda x, t, **k: fn(x, t, **k))):
        d.clear_gt_noise_cache()
        with SeqRandn(_dpm_draw_order(grid), seed, device=DEV) as rng:
            runs[name] = [(o["sample"].clone(), o["pred_xstart"].clone()) for o in d.dpm_solver_sample_loop_progressive(
                model, shape, steps=N, model_kwargs={"gt": gt, "gt_keep_mask": keep}, device=DEV,
                use_inpainting_injection=True)]
        assert rng.i == len(rng.seq)
    assert len(runs["fused"]) == N
    for (s1, p1), (s0, p0) in zip(runs["fused"], runs["unfused"]):
        assert torch.equal(s1, s0) and torch.equal(p1, p0), precision
    gtc, keepc = gt.cpu(), keep.cpu()
    with torch.no_grad():
        want = O.sample_loop(
            d.alphas_cumprod,
            lambda x, t: uor.inpaint_forward(sd, cfg, x.float(), torch.full((2,), t), gtc * keepc, 1 - keepc),
            seeded_noise("xT", 0, shape, seed), N, 2, clip=True, gt=gtc, keep=keepc,
            noise_fn=lambda t: seeded_noise("inject", t, shape, seed))
    p = psnr(runs["fused"][-1][0].cpu(), want.float())
    print("T64 2M-20 %s: PSNR vs float64 oracle %.1f dB" % (precision, p))
    assert p >= min_psnr, (precision, p)


# ------------------------------------------------------------------------------------------ 6: the checkpoint's setup
def test_ref_ffhq256_quadratic_1000_fused_known_region_exact(lib):
    import fidm_b200 as F
    from fidm_b200 import dpm_solver
    from fidm_b200.utils.synth import synth_batch
    model, d, _ = F.create_model_and_diffusion(None, DEV)
    assert d.num_timesteps == 1000
    fn = F.InpaintingModelFn(model)
    plans = []
    inner = fn.fused_plan
    fn.fused_plan = lambda *a: plans.append(inner(*a)) or plans[-1]
    data = synth_batch(2, 256, seed=4, device=DEV)
    gt, keep = data["gt"], data["gt_keep_mask"]
    N = 20
    torch.manual_seed(0)
    d.clear_gt_noise_cache()
    outs = list(d.dpm_solver_sample_loop_progressive(fn, (2, 3, 256, 256), steps=N, device=DEV,
                                                     model_kwargs={"gt": gt, "gt_keep_mask": keep},
                                                     use_inpainting_injection=True))
    assert len(plans) == 1 and plans[0] is not None          # the loop ran on the engine plan (step-boundary fusion)
    assert len(outs) == N and torch.isfinite(outs[-1]["sample"]).all()
    cls = d.coefficient_table(0.0)
    known = keep.expand(2, 3, 256, 256) == 1
    for t, o in zip(dpm_solver.timestep_grid(1000, N)[1:], outs[:-1]):
        n = d._gt_noises_cache[(gt.shape, int(t), gt.device)]
        wg = cls[t, 0].item() * gt + cls[t, 1].item() * n
        assert torch.equal(o["sample"][known], wg[known]), int(t)


# ------------------------------------------------------------------------------------------ 7: errors
def test_invalid_arguments_raise(lib):
    from fidm_b200 import dpm_solver
    d = _diffusion(1000, "quadratic", learn_sigma=True)
    tab = dpm_solver.coefficient_table(d, 20, 2).to(DEV)
    x, mo = torch.zeros(1, 3, 8, 8, device=DEV), torch.zeros(1, 6, 8, 8, device=DEV)
    gt, n = torch.zeros_like(x), torch.zeros_like(x)
    with pytest.raises(lib.FidmError):                                       # step out of range
        d._multistep(tab, 20, x, mo)
    with pytest.raises(lib.FidmError):                                       # no history at step 0
        d._multistep(tab, 0, x, mo, m_prev=x)
    with pytest.raises(lib.FidmError):                                       # mask channels
        d._multistep(tab, 3, x, mo, gt=gt, keep=torch.zeros(1, 2, 8, 8, device=DEV), inject_noise=n)
    with pytest.raises(lib.FidmError):                                       # stem dtype
        d._multistep(tab, 3, x, mo, stem=(torch.zeros(1, 8, 8, 16, device=DEV, dtype=torch.uint8),
                                          torch.zeros(1, device=DEV)))
    with pytest.raises(lib.FidmError):                                       # model output channels
        d._multistep(tab, 3, x, torch.zeros(1, 4, 8, 8, device=DEV))
    a = lib.MultistepArgs()                                                  # null pointers through the C ABI
    assert lib.lib().fidm_multistep_step(ctypes.byref(a), lib.stream()) == -1
    with pytest.raises(ValueError):
        d.dpm_solver_sample_loop(lambda x, t, **k: mo, (1, 3, 8, 8), steps=1001, device=DEV)
