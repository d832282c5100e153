"""GPU: K4 (fused sampler step), layout converters and the K5 timestep path, through the C ABI."""
import math
import os

import pytest
import torch

pytestmark = pytest.mark.gpu


def _case_inputs(c, dev):
    g = torch.Generator().manual_seed(c["seed"])
    B, C, H, W = c["sample"].shape
    t, T = c["t"], c["T"]
    x = torch.randn(B, C, H, W, generator=g) * (1.0 + t / T)
    gt = torch.rand(B, C, H, W, generator=g) * 2 - 1
    keep = (torch.rand(B, 1, H, W, generator=g) > 0.4).float()
    mo = torch.randn(B, 2 * C if c["var_type"] == "learned_range" else C, H, W, generator=g)
    n_inj = torch.randn(B, C, H, W, generator=g)
    z = torch.randn(B, C, H, W, generator=g)
    return [v.to(dev) for v in (x, gt, keep, mo, n_inj, z)]


def test_sampler_step_matches_reference_golden(cuda_lib, golden_dir):
    """Every mode of the step kernel against outputs of the UNMODIFIED reference:
    injection and DDIM bit-exact, DDPM to 1e-6 (device expf)."""
    import fidm_b200 as F
    from fidm_b200 import _lib as L
    dev = torch.device("cuda:0")
    cases = torch.load(os.path.join(golden_dir, "sampler_steps.pt"))
    n_exact = 0
    for c in cases:
        d = F.create_gaussian_diffusion(steps=c["T"], learn_sigma=c["var_type"] == "learned_range",
                                        sigma_small=c["var_type"] == "fixed_small", noise_schedule=c["sched"])
        x, gt, keep, mo, n_inj, z = _case_inputs(c, dev)
        t = c["t"]
        tt = torch.full((x.shape[0],), t, dtype=torch.int64, device=dev)
        # (1) public single-step API with per-sample t tensor, injection noise through the cache / randn_like
        d.clear_gt_noise_cache()
        draws = iter([n_inj, z])
        rl = torch.randn_like
        torch.randn_like = lambda a, **k: next(draws)
        try:
            fn = d.ddim_sample if c["mode"] == "ddim" else d.p_sample
            kw = {"eta": c["eta"]} if c["mode"] == "ddim" else {}
            got = fn(lambda xx, ts, **k: mo, x, tt, clip_denoised=True, model_kwargs={"gt": gt, "gt_keep_mask": keep},
                     use_inpainting_injection=True, use_cumulative_noise=c["cumulative"], **kw)
        finally:
            torch.randn_like = rl
        # (2) fused kernel: inject-only, then update-only with scalar t
        xi = d._step(L.STEP_INJECT_ONLY, x, t_inject=t, gt=gt, keep=keep, inject_noise=n_inj,
                     cumulative=c["cumulative"], want_next=True)["x_next"]
        assert torch.equal(xi.cpu(), c["x_inj"]), (c["sched"], t, "inject")
        r = d._step(L.STEP_UPDATE_ONLY, xi, t=t, model_out=mo, z=z, ddim=c["mode"] == "ddim", eta=c["eta"],
                    want_sample=True, want_x0=True)
        for out in (got, r):
            assert torch.equal(out["pred_xstart"].cpu(), c["pred_xstart"]), (c["sched"], t, c["mode"])
            if c["mode"] == "ddim":
                assert torch.equal(out["sample"].cpu(), c["sample"]), (c["sched"], t, c["eta"])
                n_exact += 1
            else:
                assert torch.allclose(out["sample"].cpu(), c["sample"], rtol=2e-6, atol=2e-6)
    assert n_exact == 2 * 72


def test_fused_update_inject_equals_two_launches(cuda_lib):
    import fidm_b200 as F
    from fidm_b200 import _lib as L
    dev = torch.device("cuda:0")
    d = F.create_gaussian_diffusion(steps=100, learn_sigma=True, noise_schedule="cosine")
    g = torch.Generator(device=dev).manual_seed(3)
    B, H = 3, 32
    x = torch.randn(B, 3, H, H, device=dev, generator=g)
    mo = torch.randn(B, 6, H, H, device=dev, generator=g)
    gt = torch.rand(B, 3, H, H, device=dev, generator=g) * 2 - 1
    keep = (torch.rand(B, 1, H, H, device=dev, generator=g) > 0.5).float()
    z = torch.randn(B, 3, H, H, device=dev, generator=g)
    n = torch.randn(B, 3, H, H, device=dev, generator=g)
    for ddim, eta in ((True, 0.0), (True, 0.5), (False, 0.0)):
        a = d._step(L.STEP_UPDATE_ONLY, x, t=40, model_out=mo, z=z, ddim=ddim, eta=eta, want_sample=True)["sample"]
        b = d._step(L.STEP_INJECT_ONLY, a, t_inject=39, gt=gt, keep=keep, inject_noise=n, want_next=True)["x_next"]
        f = d._step(L.STEP_UPDATE_INJECT, x, t=40, t_inject=39, model_out=mo, z=z, gt=gt, keep=keep, inject_noise=n,
                    ddim=ddim, eta=eta, want_sample=True, want_next=True)
        assert torch.equal(f["sample"], a) and torch.equal(f["x_next"], b)
        # known-region pixels are exactly q_sample(gt, 39) with the supplied noise; holes keep the update
        m = keep.expand_as(b) == 1
        c = d.coefficient_table(0.0)[39]
        wg = c[0].item() * gt + c[1].item() * n      # fp32 scalar * tensor, one rounding per op
        assert torch.equal(b[m], wg[m]) and torch.equal(b[~m], a[~m])


def test_step_argument_errors(cuda_lib):
    import fidm_b200 as F
    from fidm_b200 import _lib as L
    d = F.create_gaussian_diffusion(steps=50, learn_sigma=True, noise_schedule="cosine")
    x = torch.zeros(1, 3, 8, 8, device="cuda")
    with pytest.raises(ValueError):
        d._step(L.STEP_UPDATE_ONLY, x, t=50, model_out=torch.zeros(1, 6, 8, 8, device="cuda"), want_sample=True)
    with pytest.raises(AssertionError):
        d._step(L.STEP_UPDATE_ONLY, x, t=3, model_out=torch.zeros(1, 3, 8, 8, device="cuda"), want_sample=True)


@pytest.mark.parametrize("schedule", ["all", "low"])
@pytest.mark.parametrize("loop", ["ddim", "ddpm", "repaint", "dpm_solver"])
def test_fused_loops_equal_for_channels_last_noise(cuda_lib, loop, schedule, monkeypatch):
    """T64 (synthetic weights) on the engine plan: a channels_last x_T gives every loop bit for bit what the same x_T
    in NCHW order gives.  The kernels write NCHW state, so the loops must not allocate their state like x_T."""
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_batch, synth_state_dict
    monkeypatch.setenv("FIDM_FUSED_STEP", "1")
    dev = torch.device("cuda:0")
    cfg = F.CONFIGS["T64"]
    model = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
    model.load_state_dict(synth_state_dict(cfg, seed=2), strict=True)
    fn = F.InpaintingModelFn(model.to(dev))
    plans = []
    inner = fn.fused_plan
    fn.fused_plan = lambda *a: plans.append(inner(*a)) or plans[-1]
    d = F.create_gaussian_diffusion(steps=20, learn_sigma=True, noise_schedule="cosine")
    data = synth_batch(2, 64, seed=6, device=dev)
    shape = (2, 3, 64, 64)
    noise = torch.randn(shape, device=dev, generator=torch.Generator(device=dev).manual_seed(1))
    kw = dict(model_kwargs={"gt": data["gt"], "gt_keep_mask": data["gt_keep_mask"]}, device=dev,
              use_inpainting_injection=True, injection_schedule=schedule)
    run = {"ddim": lambda x_T: d.ddim_sample_loop(fn, shape, noise=x_T, **kw),
           "ddpm": lambda x_T: d.p_sample_loop(fn, shape, noise=x_T, **kw),
           "repaint": lambda x_T: d.repaint_sample_loop(fn, shape, jump_length=4, jump_n_sample=2, noise=x_T, **kw),
           "dpm_solver": lambda x_T: d.dpm_solver_sample_loop(fn, shape, steps=8, noise=x_T, **kw)}[loop]
    outs = []
    for x_T in (noise, noise.contiguous(memory_format=torch.channels_last)):
        torch.manual_seed(4)
        outs.append(run(x_T))
    assert len(plans) == 2 and all(p is not None for p in plans)      # both runs were fused
    assert torch.isfinite(outs[0]).all() and torch.equal(outs[1], outs[0]), (loop, schedule)


def test_pack_unpack_roundtrip(cuda_lib):
    from fidm_b200 import ops
    dev = "cuda"
    x = torch.randn(2, 3, 16, 24, device=dev)
    mi = torch.randn(2, 3, 16, 24, device=dev)
    m = (torch.rand(2, 1, 16, 24, device=dev) > 0.5).float()
    for dt in (torch.float32, torch.bfloat16):
        p = ops.pack_nchw_to_nhwc([(x, 1), (mi, 1), (m, 3)], dtype=dt, c_pad=64)
        want = torch.cat([x, mi, m.repeat(1, 3, 1, 1)], 1).permute(0, 2, 3, 1)
        assert torch.equal(p[..., :9].float(), want.to(dt).float())
        assert not p[..., 9:].any()
        back = ops.unpack_nhwc_to_nchw(p, 9)
        assert torch.equal(back, want.to(dt).float().permute(0, 3, 1, 2))


def test_timestep_path(cuda_lib):
    from fidm_b200 import ops
    dev = "cuda"
    dim = 256
    half = dim // 2
    freqs = torch.exp(-math.log(10000) * torch.arange(half, dtype=torch.float32) / half)
    t = torch.tensor([0.0, 1.0, 37.0, 999.0], device=dev)
    emb = ops.timestep_embedding(t, freqs.to(dev), dim)
    ang = t[:, None] * freqs.to(dev)[None]
    want = torch.cat([ang.cos(), ang.sin()], -1)
    assert torch.allclose(emb, want, atol=2e-6, rtol=0)
    for B, K, O in ((4, 256, 1024), (9, 1024, 3072), (1, 64, 128)):
        x = torch.randn(B, K, device=dev)
        w = torch.randn(O, K, device=dev) / math.sqrt(K)
        b = torch.randn(O, device=dev)
        y = ops.linear_small(x, w, b, silu_input=True)
        want = torch.nn.functional.linear(torch.nn.functional.silu(x.double()), w.double(), b.double()).float()
        assert torch.allclose(y, want, atol=2e-5, rtol=1e-5)
        y16 = ops.linear_small(x, w.bfloat16(), b)
        want16 = torch.nn.functional.linear(x.double(), w.bfloat16().double(), b.double()).float()
        assert torch.allclose(y16, want16, atol=2e-5, rtol=1e-5)


def test_io_adapters_match_reference_conventions(cuda_lib):
    """data/dataset.py:38-42,130-142 (ToTensor + Normalize, mask < 0.5) and toU8 / final blend
    (test_inp_ddim_100.py:33-41, 693-696), bit-exact against the same torch ops."""
    from fidm_b200 import ops
    g = torch.Generator().manual_seed(0)
    img = torch.randint(0, 256, (3, 32, 24, 3), dtype=torch.uint8, generator=g).cuda()
    msk = torch.randint(0, 256, (3, 32, 24), dtype=torch.uint8, generator=g).cuda()
    d = ops.prepare_inputs_u8(img, msk)
    # the reference's DataLoader runs these ops on the CPU (true IEEE division; CUDA torch multiplies by 1/255)
    t = img.cpu().permute(0, 3, 1, 2).float().div(255)
    want_img = ((t - 0.5) / 0.5).cuda()
    want_mask = (msk.cpu().float().div(255)[:, None] < 0.5).float().cuda()
    assert torch.equal(d["image"], want_img) and torch.equal(d["mask"], want_mask)
    assert torch.equal(d["masked_image"], want_img * (1 - want_mask))
    assert torch.equal(d["gt_keep_mask"], 1 - want_mask)
    sample = torch.randn(3, 3, 32, 24, device="cuda") * 1.5
    out = ops.blend_to_u8(sample, d["image"], d["mask"])
    res = sample * d["mask"] + d["image"] * (1 - d["mask"])
    want = ((res + 1) * 127.5).clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1).contiguous()
    assert torch.equal(out, want)
    # (the reference's toU8 truncates, so known pixels come back within one code of the original bytes)
    keep = (1 - d["mask"]).bool().expand(-1, 3, -1, -1).permute(0, 2, 3, 1)
    assert (out[keep].int() - img[keep].int()).abs().max().item() <= 1
    assert torch.equal(ops.blend_to_u8(sample), ((sample + 1) * 127.5).clamp(0, 255).to(torch.uint8).permute(0, 2, 3, 1))
