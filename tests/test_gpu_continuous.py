"""GPU: continuous batching -- K8 (fidm_sampler_step_slots) bit for bit against the seeded K4 per slot, the continuous
sampler against each request run alone through the seeded loops, the T64 UNet fused against unfused and against
lockstep batches, REF-FFHQ256 at 256x256, and no synchronisation per iteration on the fused path."""
import ctypes
import itertools

import pytest
import torch

from helpers import psnr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SENT = 4096.0                   # exact in fp32, bf16 and fp16


@pytest.fixture(scope="module")
def lib():
    import fidm_b200  # noqa: F401
    from fidm_b200 import _lib as L
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    L.check(L.lib().fidm_device_supported(0), "device")
    return L


def _seeds(vals):
    from fidm_b200 import seeded
    return seeded.check_seeds(vals, len(vals)).to(DEV)


# ------------------------------------------------------------------------------------------ 1: K8 against seeded K4
def _k8(L, d, x, mo, gt, keep, actions, seeds, *, ddim, eta, cumulative, schedule, stem, out, x_next):
    """One K8 launch on explicit buffers (as continuous.ContinuousSampler fills its arguments)."""
    from fidm_b200 import continuous
    from fidm_b200.gaussian_diffusion import _MEAN_CODE, _VAR_CODE
    B, Cn = x.shape[:2]
    T = d.num_timesteps
    a = L.StepArgs()
    a.batch, a.channels, a.hw = B, Cn, x.numel() // (B * Cn)
    a.sampler = L.SAMPLER_DDIM if ddim else L.SAMPLER_DDPM
    a.mean_type, a.var_type = _MEAN_CODE[d.model_mean_type], _VAR_CODE[d.model_var_type]
    a.clip_denoised, a.cumulative, a.mask_channels, a.num_timesteps = 1, int(cumulative), keep.shape[1], T
    coef = d._coef(x.device, eta if ddim else 0.0)
    tv = torch.tensor([d._t_value(t) for t in range(T)], dtype=torch.float32, device=DEV)
    inj = torch.tensor(continuous.injection_draws(d, schedule, cumulative), dtype=torch.int32, device=DEV)
    a.coef, a.x, a.model_out, a.gt, a.keep_mask, a.x_next = (L.ptr(v) for v in (coef, x, mo, gt, keep, x_next))
    x_in, t_in = stem
    a.stem_out, a.stem_dtype, a.stem_ld, a.t_out = L.ptr(x_in), L.dtype_code(x_in.dtype), x_in.shape[-1], L.ptr(t_in)
    s = L.SlotArgs()
    s.t_value, s.inject_draw, s.out = L.ptr(tv), L.ptr(inj), L.ptr(out)
    s.step_noise = int(not ddim or eta != 0.0)
    for b in range(B):
        s.action[b] = actions[b]
        s.seeds[b] = int(seeds[b]) & ((1 << 64) - 1)
    L.check(L.lib().fidm_sampler_step_slots(ctypes.byref(a), ctypes.byref(s), L.stream()), "sampler_step_slots")
    torch.cuda.synchronize()
    return inj.tolist()


def _k4_alone(L, d, x, mo, gt, keep, act, seeds, draws, *, ddim, eta, cumulative, schedule, sdt):
    """What the seeded loop computes for one image for K8's action `act`: (state, stem channels, t_out) or the
    sample at t = 0."""
    from fidm_b200 import seeded
    T = d.num_timesteps
    H, W = x.shape[2:]
    x_in = torch.full((1, H, W, 16), SENT, device=DEV, dtype=sdt)
    t_in = torch.full((1,), SENT, device=DEV)
    tag = L.NOISE_INJECT if cumulative else L.NOISE_INJECT_FRESH
    if act == L.SLOT_ADMIT:
        xt = seeded.randn(seeds, tuple(x.shape), L.NOISE_XT, 0)
        if draws[T - 1] < 0:          # gated: the loop's state is x_T, packed as is (round to nearest even)
            x_in[..., :x.shape[1]] = xt.permute(0, 2, 3, 1).to(sdt)
            t_in.fill_(d._t_value(T - 1))
            return xt, x_in, t_in
        r = d._step(L.STEP_INJECT_ONLY, xt, t_inject=T - 1, gt=gt, keep=keep,
                    inject_noise=seeded.Draw(seeds, tag, draws[T - 1]), cumulative=cumulative, want_next=True,
                    stem=(x_in, t_in), t_next=d._t_value(T - 1))
        return r["x_next"], x_in, t_in
    t = act
    do_inj = t >= 1 and draws[t - 1] >= 0
    z = seeded.Draw(seeds, L.NOISE_STEP, T - 1 - t) if (not ddim or eta != 0.0) else None
    r = d._step(L.STEP_UPDATE_INJECT if do_inj else L.STEP_UPDATE_ONLY, x, t=t, t_inject=t - 1, model_out=mo, z=z,
                gt=gt if do_inj else None, keep=keep if do_inj else None,
                inject_noise=seeded.Draw(seeds, tag, draws[t - 1]) if do_inj else None, ddim=ddim, eta=eta,
                cumulative=cumulative, want_sample=t == 0, want_next=t > 0,
                stem=(x_in, t_in) if t > 0 else None, t_next=d._t_value(t - 1) if t > 0 else None)
    if t == 0:
        return r["sample"], None, None
    return r["x_next"], x_in, t_in


K8_CASES = list(itertools.product(
    [(True, 0.0), (True, 0.6), (False, 0.0)],                        # DDIM eta 0, eta > 0, DDPM
    [dict(learn_sigma=True), dict(), dict(sigma_small=True), dict(predict_xstart=True, learn_sigma=True)],
    [True, False]))                                                  # cumulative / fresh


@pytest.mark.parametrize("sampler,dkw,cumulative", K8_CASES)
def test_k8_slots_equal_seeded_k4_alone(lib, sampler, dkw, cumulative):
    import fidm_b200 as F
    L = lib
    ddim, eta = sampler
    T = 20
    i = K8_CASES.index((sampler, dkw, cumulative))
    d = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine", rescale_timesteps=bool(i % 2), **dkw)
    learn = dkw.get("learn_sigma", False)
    # layouts x mask channels x stem dtypes x injection schedules, varied over the cases
    odd = (i // 2) % 2 == 1
    mc = 1 if i % 2 == 0 else 3
    sdt = (torch.bfloat16, torch.float16, torch.float32)[i % 3]
    schedule = ("all", "high", "low")[(i // 3) % 3]
    H, W = (7, 9) if odd else (8, 8)
    # slot actions: admit, idle, T-1, a middle t, both sides of the high/low gate, 1, 0, idle
    actions = [L.SLOT_ADMIT, L.SLOT_IDLE, T - 1, 13, T // 2, T // 2 - 1, 1, 0, L.SLOT_IDLE]
    B, Cn = len(actions), 3
    seed_vals = [3 + 7 * b for b in range(B)]
    seed_vals[2] = 2 ** 64 - 1
    seeds = _seeds(seed_vals)
    g = torch.Generator().manual_seed(i)
    x = (torch.randn(B, Cn, H, W, generator=g) * 1.5).to(DEV)
    mo = torch.randn(B, 2 * Cn if learn else Cn, H, W, generator=g).to(DEV)
    gt = (torch.rand(B, Cn, H, W, generator=g) * 2 - 1).to(DEV)
    keep = (torch.rand(B, mc, H, W, generator=g) > 0.5).float().to(DEV)
    x_in = torch.full((B, H, W, 16), SENT, device=DEV, dtype=sdt)
    t_in = torch.full((B,), SENT, device=DEV)
    out = torch.full_like(x, SENT)
    x_next = torch.full_like(x, SENT)
    kw = dict(ddim=ddim, eta=eta, cumulative=cumulative, schedule=schedule)
    draws = _k8(L, d, x, mo, gt, keep, actions, seed_vals, stem=(x_in, t_in), out=out, x_next=x_next, **kw)
    for b, act in enumerate(actions):
        tag = (b, act)
        if act == L.SLOT_IDLE:
            assert (x_next[b] == SENT).all() and (out[b] == SENT).all(), tag
            assert (x_in[b].float() == SENT).all() and t_in[b].item() == SENT, tag
            continue
        want, w_stem, w_t = _k4_alone(L, d, x[b:b + 1], mo[b:b + 1], gt[b:b + 1], keep[b:b + 1], act, seeds[b:b + 1],
                                      draws, sdt=sdt, **kw)
        if act == 0:
            assert torch.equal(out[b:b + 1], want), tag
            assert (x_next[b] == SENT).all() and (x_in[b].float() == SENT).all() and t_in[b].item() == SENT, tag
            continue
        assert (out[b] == SENT).all(), tag
        assert torch.equal(x_next[b:b + 1], want), tag
        assert torch.equal(x_in[b:b + 1, :, :, :Cn], w_stem[:, :, :, :Cn]), tag
        assert (x_in[b, :, :, Cn:].float() == SENT).all(), tag                # conditioning channels untouched
        assert torch.equal(t_in[b:b + 1], w_t), tag


@pytest.mark.parametrize("odd", [False, True])
@pytest.mark.parametrize("sampler", [(True, 0.0), (True, 0.6), (False, 0.0)])
def test_k8_all_slots_at_one_t_equal_seeded_k4_on_the_batch(lib, sampler, odd):
    """Every slot updating at the same t, in place (x_next = x), against one seeded K4 launch on the whole batch."""
    import fidm_b200 as F
    from fidm_b200 import continuous, seeded
    L = lib
    ddim, eta = sampler
    T, t = 30, 17
    d = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine", learn_sigma=True)
    H, W = (5, 11) if odd else (16, 16)
    B, Cn = 8, 3
    vals = list(range(100, 100 + B))
    seeds = _seeds(vals)
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, Cn, H, W, generator=g).to(DEV)
    mo = torch.randn(B, 2 * Cn, H, W, generator=g).to(DEV)
    gt = (torch.rand(B, Cn, H, W, generator=g) * 2 - 1).to(DEV)
    keep = (torch.rand(B, 1, H, W, generator=g) > 0.5).float().to(DEV)
    for cumulative in (True, False):
        draws = continuous.injection_draws(d, "all", cumulative)
        x_in = torch.zeros(B, H, W, 16, device=DEV, dtype=torch.bfloat16)
        t_in = torch.zeros(B, device=DEV)
        tag = L.NOISE_INJECT if cumulative else L.NOISE_INJECT_FRESH
        r = d._step(L.STEP_UPDATE_INJECT, x, t=t, t_inject=t - 1, model_out=mo,
                    z=seeded.Draw(seeds, L.NOISE_STEP, T - 1 - t) if (not ddim or eta) else None, gt=gt, keep=keep,
                    inject_noise=seeded.Draw(seeds, tag, draws[t - 1]), ddim=ddim, eta=eta, cumulative=cumulative,
                    want_next=True, stem=(x_in, t_in), t_next=d._t_value(t - 1))
        xs = x.clone()
        k_in = torch.zeros_like(x_in)
        k_t = torch.zeros_like(t_in)
        _k8(L, d, xs, mo, gt, keep, [t] * B, vals, ddim=ddim, eta=eta, cumulative=cumulative, schedule="all",
            stem=(k_in, k_t), out=torch.empty_like(x), x_next=xs)
        assert torch.equal(xs, r["x_next"]) and torch.equal(k_in, x_in) and torch.equal(k_t, t_in), cumulative


def test_k8_refuses_bad_arguments(lib):
    L = lib
    x = torch.zeros(2, 3, 8, 8, device=DEV)
    tv = torch.zeros(10, device=DEV)
    inj = torch.zeros(10, dtype=torch.int32, device=DEV)
    a = L.StepArgs()
    a.batch, a.channels, a.hw, a.mask_channels, a.num_timesteps, a.sampler = 2, 3, 64, 1, 10, L.SAMPLER_DDIM
    a.var_type = L.VAR_FIXED
    a.coef, a.x, a.model_out, a.gt, a.keep_mask, a.x_next = (L.ptr(x),) * 6
    s = L.SlotArgs()
    s.t_value, s.inject_draw, s.out = L.ptr(tv), L.ptr(inj), L.ptr(x)
    s.action[0], s.action[1] = 3, L.SLOT_IDLE

    def rc():
        return L.lib().fidm_sampler_step_slots(ctypes.byref(a), ctypes.byref(s), L.stream())

    assert rc() == 0
    for field, bad in (("action", 10), ("action", -3)):
        s.action[0] = bad
        assert rc() == -1 and b"sampler_step_slots" in L.lib().fidm_last_error_string()
    s.action[0] = 3
    for name, val in (("batch", 0), ("batch", L.MAX_SLOTS + 1), ("sampler", L.SAMPLER_DDIM_SCRIPT),
                      ("t_dev", L.ptr(x)), ("z", L.ptr(x)), ("inject_noise", L.ptr(x)), ("sample", L.ptr(x)),
                      ("model_out", None), ("mask_channels", 2)):
        old = getattr(a, name)
        setattr(a, name, val)
        assert rc() == -1, name
        setattr(a, name, old)
    s.out = None
    assert rc() == -1
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ 2: the contract
def _standin(x, t, **k):
    """Per-sample elementwise eps model (test_gpu_seeded_noise.py): its value per image is batch independent."""
    return torch.tanh(0.7 * x) * torch.cos(t.float().view(-1, 1, 1, 1) * 0.01) + 0.05 * k["gt"]


def _alone(d, model, sampler, eta, gt, keep, seed, schedule, cumulative):
    kw = dict(model_kwargs={"gt": gt, "gt_keep_mask": keep}, device=DEV, use_inpainting_injection=True,
              injection_schedule=schedule, use_cumulative_noise=cumulative, seeds=[seed])
    if sampler == "ddim":
        return d.ddim_sample_loop(model, tuple(gt.shape), eta=eta, **kw)
    return d.p_sample_loop(model, tuple(gt.shape), **kw)


def _staggered(cs, gts, keeps, seeds, plan):
    """Submit requests per `plan` ([number to submit before step i]) and step until done: {ticket: image}."""
    results, k, i = {}, 0, 0
    tickets = []
    while k < len(gts) or cs.pending():
        for _ in range(plan[i] if i < len(plan) else len(gts) - k):
            if k < len(gts):
                tickets.append(cs.submit(gts[k], keeps[k], seeds[k]))
                k += 1
        results.update(cs.step())
        i += 1
    return [results[tk] for tk in tickets]


CONTRACT = [("ddim", 0.0, "all", True, False), ("ddim", 0.6, "high", False, True), ("ddpm", 0.0, "low", True, True),
            ("ddpm", 0.0, "all", False, False), ("ddim", 0.0, "low", False, True), ("ddim", 0.6, "all", True, False)]


@pytest.mark.parametrize("sampler,eta,schedule,cumulative,rescale", CONTRACT)
def test_continuous_equals_each_request_alone(lib, sampler, eta, schedule, cumulative, rescale):
    import fidm_b200 as F
    d = F.create_gaussian_diffusion(steps=12, noise_schedule="cosine", rescale_timesteps=rescale)
    g = torch.Generator().manual_seed(11)
    S, n = 8, 7
    gts = [(torch.rand(3, S, S, generator=g) * 2 - 1).to(DEV) for _ in range(n)]
    keeps = [(torch.rand(1 if k % 2 else 3, S, S, generator=g) > 0.5).float().to(DEV) for k in range(n)]
    seeds = [5, 2 ** 64 - 1, 17, 17, 2 ** 40 + 3, 0, 99]
    cpu_state, cuda_state = torch.get_rng_state(), torch.cuda.get_rng_state()
    cs = d.continuous_sampler(_standin, slots=3, image_size=(S, S), sampler=sampler, eta=eta,
                              injection_schedule=schedule, use_cumulative_noise=cumulative, device=DEV)
    got = _staggered(cs, gts, keeps, seeds, [2, 0, 1, 0, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 1])
    assert not cs.pending()
    for k in range(n):
        want = _alone(d, _standin, sampler, eta, gts[k][None], keeps[k][None], seeds[k], schedule, cumulative)
        assert torch.equal(got[k], want), k
    assert torch.isfinite(torch.cat(got)).all() and not torch.equal(got[0], got[1])
    assert torch.equal(torch.get_rng_state(), cpu_state) and torch.equal(torch.cuda.get_rng_state(), cuda_state)
    assert not d._gt_noises_cache


def test_submit_argument_errors(lib):
    import fidm_b200 as F
    d = F.create_gaussian_diffusion(steps=5, noise_schedule="cosine")
    cs = d.continuous_sampler(_standin, slots=2, image_size=(8, 8), device=DEV)
    gt, keep = torch.zeros(3, 8, 8, device=DEV), torch.ones(1, 8, 8, device=DEV)
    bad = [(torch.zeros(3, 8, 9, device=DEV), keep, 1), (torch.zeros(2, 3, 8, 8, device=DEV), keep, 1),
           (torch.zeros(4, 8, 8, device=DEV), keep, 1), (gt.cpu(), keep, 1), (gt.double(), keep, 1),
           (gt, torch.ones(2, 8, 8, device=DEV), 1), (gt, keep.half(), 1), (gt, keep, -1), (gt, keep, 2 ** 64),
           (gt, keep, 1.5), ([0.0], keep, 1)]
    for k, (a, b, s) in enumerate(bad):
        with pytest.raises(ValueError):
            cs.submit(a, b, s)
    assert not cs.pending()
    assert cs.step() == []


# ------------------------------------------------------------------------------------------ 3-4: the UNet, bf16
def _unet(name, seed):
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_state_dict
    cfg = F.CONFIGS[name]
    m = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
    m.load_state_dict(synth_state_dict(cfg, seed=seed), strict=True)
    m.to(DEV)
    m.base_model.set_precision("bf16")
    return F.InpaintingModelFn(m)


def _against_lockstep(d, fn, S, steps_plan, label):
    from fidm_b200.utils.synth import synth_batch
    data = synth_batch(4, S, seed=8, device=DEV)
    gt, keep = data["gt"], data["gt_keep_mask"]
    seeds = [3, 2 ** 40, 77, 2 ** 63 + 1]
    lock = d.ddim_sample_loop(fn, (4, 3, S, S), model_kwargs={"gt": gt, "gt_keep_mask": keep}, device=DEV,
                              use_inpainting_injection=True, seeds=seeds)
    cs = d.continuous_sampler(fn, slots=4, image_size=(S, S), sampler="ddim")
    assert cs.plan is not None
    got = torch.cat(_staggered(cs, list(gt), list(keep), seeds, steps_plan))
    p = min(psnr(got[k][keep[k].expand(3, S, S) == 0], lock[k][keep[k].expand(3, S, S) == 0]) for k in range(4))
    print("%s: continuous (staggered admissions) vs lockstep batch 4, min hole PSNR %.1f dB, bit-identical: %s"
          % (label, p, torch.equal(got, lock)))
    assert torch.isfinite(got).all() and p >= 40.0, p
    return got


def test_t64_fused_equals_unfused_and_lockstep(lib, monkeypatch):
    import fidm_b200 as F
    fn = _unet("T64", 2)
    d = F.create_gaussian_diffusion(steps=20, learn_sigma=True, noise_schedule="cosine")
    fused = _against_lockstep(d, fn, 64, [1, 2, 0, 0, 0, 1], "T64 DDIM-20 bf16")
    monkeypatch.setenv("FIDM_FUSED_STEP", "0")
    cs = d.continuous_sampler(fn, slots=4, image_size=(64, 64), sampler="ddim")
    assert cs.plan is None
    from fidm_b200.utils.synth import synth_batch
    data = synth_batch(4, 64, seed=8, device=DEV)
    unfused = torch.cat(_staggered(cs, list(data["gt"]), list(data["gt_keep_mask"]), [3, 2 ** 40, 77, 2 ** 63 + 1],
                                   [1, 2, 0, 0, 0, 1]))
    assert torch.equal(fused, unfused)


def test_ref_ffhq256_against_lockstep(lib):
    import fidm_b200 as F
    fn = _unet("REF_FFHQ256", 3)
    d = F.create_gaussian_diffusion(steps=10, learn_sigma=True, noise_schedule="cosine")
    _against_lockstep(d, fn, 256, [2, 0, 1, 0, 1], "REF-FFHQ256 DDIM-10 bf16 256x256")


# ------------------------------------------------------------------------------------------ 5: no synchronisation
def test_fused_step_does_not_synchronise(lib):
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_batch
    fn = _unet("T64", 2)
    d = F.create_gaussian_diffusion(steps=8, learn_sigma=True, noise_schedule="cosine")
    data = synth_batch(3, 64, seed=1, device=DEV)
    cs = d.continuous_sampler(fn, slots=2, image_size=(64, 64), sampler="ddim")
    for k in range(3):
        cs.submit(data["gt"][k], data["gt_keep_mask"][k], k)
    cs.step()                                        # warm-up: graph capture, first admissions
    torch.cuda.synchronize()
    done = []
    try:
        torch.cuda.set_sync_debug_mode("error")
        while cs.pending():
            done += cs.step()                        # steady iterations, a finish, an admission
        cs.submit(data["gt"][0], data["gt_keep_mask"][0], 9)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert len(done) == 3
    assert cs.drain() and not cs.pending()
