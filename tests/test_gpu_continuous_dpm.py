"""GPU: continuous batching of the DPM-Solver++ loop -- K9 (fidm_multistep_step_slots) bit for bit against the seeded
K6 per slot and on a whole batch, its argument checks, the continuous DPM-Solver++ sampler against each request run
alone through the seeded dpm_solver_sample_loop, the T64 UNet fused against unfused, REF-FFHQ256 at 256x256 against a
lockstep batch, and no synchronisation per iteration on the fused path."""
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


def _history_sentinel(like):
    """NaN and -0 alternating: a history that is read, or multiplied by zero and added, changes the result."""
    v = torch.full_like(like, float("nan"))
    v.view(-1)[1::2] = -0.0
    return v


# ------------------------------------------------------------------------------------------ 1: K9 against seeded K6
def _k9(L, d, steps, order, x, mo, m_prev, gt, keep, actions, seeds, *, clip, cumulative, schedule, stem, out,
        x_next, m_out, inject=True):
    """One K9 launch on explicit buffers (as continuous.ContinuousDPMSolverSampler fills its arguments).  Returns the
    grid, the per-grid-point draws and orders."""
    from fidm_b200 import continuous, dpm_solver
    from fidm_b200.gaussian_diffusion import _MEAN_CODE
    B, Cn = x.shape[:2]
    grid = dpm_solver.timestep_grid(d.num_timesteps, steps)
    tv, draws, orders = continuous.dpm_slot_tables(d, grid, order, schedule, cumulative, inject)
    tv_d = torch.tensor(tv, dtype=torch.float32, device=DEV)
    dr_d = torch.tensor(draws, dtype=torch.int32, device=DEV)
    or_d = torch.tensor(orders, dtype=torch.int32, device=DEV)
    coef = d._dpm_table(x.device, steps, order, cumulative)
    a = L.MultistepArgs()
    a.batch, a.channels, a.hw = B, Cn, x.numel() // (B * Cn)
    a.mean_type, a.out_channels, a.clip_denoised = _MEAN_CODE[d.model_mean_type], mo.shape[1], int(clip)
    a.mask_channels, a.steps = keep.shape[1], steps
    a.coef, a.x, a.model_out, a.m_prev, a.m_out, a.x_next, a.gt, a.keep_mask = (
        L.ptr(v) for v in (coef, x, mo, m_prev, m_out, x_next, gt, keep))
    if stem is not None:
        x_in, t_in = stem
        a.stem_out, a.stem_dtype, a.stem_ld, a.t_out = (L.ptr(x_in), L.dtype_code(x_in.dtype), x_in.shape[-1],
                                                        L.ptr(t_in))
    s = L.MsSlotArgs()
    s.t_value, s.inject_draw, s.order, s.out = L.ptr(tv_d), L.ptr(dr_d), L.ptr(or_d), L.ptr(out)
    s.inject_tag = L.NOISE_INJECT if cumulative else L.NOISE_INJECT_FRESH
    cls = d.coefficient_table(0.0)
    ia, is_ = (L.C_SQRT_AB, L.C_SQRT_1MAB) if cumulative else (L.C_SQRT_AB_F32, L.C_SQRT_1MAB_F32)
    s.admit_inject_a, s.admit_inject_s = float(cls[int(grid[0]), ia]), float(cls[int(grid[0]), is_])
    for b in range(B):
        s.action[b] = actions[b]
        s.seeds[b] = int(seeds[b]) & ((1 << 64) - 1)
    L.check(L.lib().fidm_multistep_step_slots(ctypes.byref(a), ctypes.byref(s), L.stream()), "multistep_step_slots")
    torch.cuda.synchronize()
    return grid, draws, orders


def _k6_alone(L, d, steps, order, grid, draws, orders, x, mo, mp, gt, keep, act, seeds, *, clip, cumulative, sdt):
    """What the seeded loop computes for one image for K9's action `act`: (state, history, stem channels, t_out), or
    (None, x0 prediction, None, None) at the last grid point."""
    from fidm_b200 import seeded
    T = d.num_timesteps
    H, W = x.shape[2:]
    x_in = torch.full((1, H, W, 16), SENT, device=DEV, dtype=sdt)
    t_in = torch.full((1,), SENT, device=DEV)
    tag = L.NOISE_INJECT if cumulative else L.NOISE_INJECT_FRESH
    if act == L.SLOT_ADMIT:
        xt = seeded.randn(seeds, tuple(x.shape), L.NOISE_XT, 0)
        if draws[0] < 0:              # gated: the loop's state is x_T, packed as is (round to nearest even)
            x_in[..., :x.shape[1]] = xt.permute(0, 2, 3, 1).to(sdt)
            t_in.fill_(d._t_value(T - 1))
            return xt, None, x_in, t_in
        r = d._step(L.STEP_INJECT_ONLY, xt, t_inject=T - 1, gt=gt, keep=keep,
                    inject_noise=seeded.Draw(seeds, tag, draws[0]), cumulative=cumulative, want_next=True,
                    stem=(x_in, t_in), t_next=d._t_value(T - 1))
        return r["x_next"], None, x_in, t_in
    k = act
    tab = d._dpm_table(x.device, steps, order, cumulative)
    if k == steps - 1:
        m, _ = d._multistep(tab, k, x, mo, want_next=False, clip=clip)
        return None, m, None, None
    inj = draws[k + 1] >= 0
    m, nxt = d._multistep(tab, k, x, mo, m_prev=mp if orders[k] == 2 else None, clip=clip,
                          gt=gt if inj else None, keep=keep if inj else None,
                          inject_noise=seeded.Draw(seeds, tag, draws[k + 1]) if inj else None,
                          stem=(x_in, t_in), t_next=d._t_value(int(grid[k + 1])))
    return nxt, m, x_in, t_in


K9_CASES = list(itertools.product(
    [dict(learn_sigma=True), dict(), dict(predict_xstart=True), dict(predict_xstart=True, learn_sigma=True)],
    [True, False],                                                   # clip
    [True, False]))                                                  # cumulative / fresh


@pytest.mark.parametrize("dkw,clip,cumulative", K9_CASES)
def test_k9_slots_equal_seeded_k6_alone(lib, dkw, clip, cumulative):
    import fidm_b200 as F
    from fidm_b200 import continuous, dpm_solver
    L = lib
    i = K9_CASES.index((dkw, clip, cumulative))
    T, steps, order = 20, 8, 2
    d = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine", rescale_timesteps=bool(i % 2), **dkw)
    learn = dkw.get("learn_sigma", False)
    # layouts x mask channels x stem dtypes x injection schedules, varied over the cases
    odd = (i // 2) % 2 == 1
    mc = 1 if i % 2 == 0 else 3
    sdt = (torch.bfloat16, torch.float32)[(i // 4) % 2]
    schedule = ("all", "high", "low")[i % 3]
    H, W = (7, 9) if odd else (8, 8)
    # slot actions: admit, idle, k = 0, second-order k = 1 and 3, k = steps-2 (first order into t = 0), steps-1, idle
    actions = [L.SLOT_ADMIT, L.SLOT_IDLE, 0, 1, 3, steps - 2, steps - 1, L.SLOT_IDLE]
    B, Cn = len(actions), 3
    seed_vals = [3 + 7 * b for b in range(B)]
    seed_vals[2], seed_vals[3] = 2 ** 64 - 1, 0
    seeds = _seeds(seed_vals)
    g = torch.Generator().manual_seed(i)
    x = (torch.randn(B, Cn, H, W, generator=g) * 1.5).to(DEV)
    mo = (torch.randn(B, 2 * Cn if learn else Cn, H, W, generator=g) * 1.3).to(DEV)
    mp = torch.randn(B, Cn, H, W, generator=g).to(DEV)
    gt = (torch.rand(B, Cn, H, W, generator=g) * 2 - 1).to(DEV)
    keep = (torch.rand(B, mc, H, W, generator=g) > 0.5).float().to(DEV)
    _, _, orders = continuous.dpm_slot_tables(d, dpm_solver.timestep_grid(T, steps), order, schedule, cumulative)
    for b, act in enumerate(actions):            # a history K9 must not read: the admitted and first-order slots
        if act == L.SLOT_ADMIT or (act >= 0 and orders[act] != 2):
            mp[b] = _history_sentinel(mp[b])
    x_in = torch.full((B, H, W, 16), SENT, device=DEV, dtype=sdt)
    t_in = torch.full((B,), SENT, device=DEV)
    out, x_next, m_out = (torch.full_like(x, SENT) for _ in range(3))
    kw = dict(clip=clip, cumulative=cumulative)
    grid, draws, orders = _k9(L, d, steps, order, x, mo, mp, gt, keep, actions, seed_vals, schedule=schedule,
                              stem=(x_in, t_in), out=out, x_next=x_next, m_out=m_out, **kw)
    assert orders[1] == orders[3] == 2 and orders[0] == orders[steps - 2] == 1
    for b, act in enumerate(actions):
        tag = (b, act)
        if act == L.SLOT_IDLE:
            assert (x_next[b] == SENT).all() and (out[b] == SENT).all() and (m_out[b] == SENT).all(), tag
            assert (x_in[b].float() == SENT).all() and t_in[b].item() == SENT, tag
            continue
        want, w_m, w_stem, w_t = _k6_alone(L, d, steps, order, grid, draws, orders, x[b:b + 1], mo[b:b + 1],
                                           mp[b:b + 1], gt[b:b + 1], keep[b:b + 1], act, seeds[b:b + 1], sdt=sdt, **kw)
        if act == steps - 1:
            assert torch.equal(out[b:b + 1], w_m), tag
            assert (x_next[b] == SENT).all() and (m_out[b] == SENT).all(), tag
            assert (x_in[b].float() == SENT).all() and t_in[b].item() == SENT, tag
            continue
        assert (out[b] == SENT).all(), tag
        assert torch.equal(x_next[b:b + 1], want), tag
        if act == L.SLOT_ADMIT:
            assert (m_out[b] == SENT).all(), tag
        else:
            assert torch.equal(m_out[b:b + 1], w_m), tag
        assert torch.isfinite(x_next[b]).all(), tag
        assert torch.equal(x_in[b:b + 1, :, :, :Cn], w_stem[:, :, :, :Cn]), tag
        assert (x_in[b, :, :, Cn:].float() == SENT).all(), tag                # conditioning channels untouched
        assert torch.equal(t_in[b:b + 1], w_t), tag


@pytest.mark.parametrize("odd", [False, True])
@pytest.mark.parametrize("k", [0, 3])
def test_k9_all_slots_at_one_k_equal_seeded_k6_on_the_batch(lib, k, odd):
    """Every slot at grid point k, in place (x_next = x, m_out = m_prev), against one seeded K6 launch on the batch."""
    import fidm_b200 as F
    from fidm_b200 import seeded
    L = lib
    T, steps, order = 30, 8, 2
    d = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine", learn_sigma=True)
    H, W = (5, 11) if odd else (16, 16)
    B, Cn = 8, 3
    vals = list(range(100, 100 + B))
    seeds = _seeds(vals)
    g = torch.Generator().manual_seed(7)
    x = torch.randn(B, Cn, H, W, generator=g).to(DEV)
    mo = torch.randn(B, 2 * Cn, H, W, generator=g).to(DEV)
    mp = torch.randn(B, Cn, H, W, generator=g).to(DEV)
    gt = (torch.rand(B, Cn, H, W, generator=g) * 2 - 1).to(DEV)
    keep = (torch.rand(B, 1, H, W, generator=g) > 0.5).float().to(DEV)
    for cumulative in (True, False):
        xs, ms = x.clone(), mp.clone()
        k_in = torch.zeros(B, H, W, 16, device=DEV, dtype=torch.bfloat16)
        k_t = torch.zeros(B, device=DEV)
        grid, draws, orders = _k9(L, d, steps, order, xs, mo, ms, gt, keep, [k] * B, vals, clip=True,
                                  cumulative=cumulative, schedule="all", stem=(k_in, k_t), out=torch.empty_like(x),
                                  x_next=xs, m_out=ms)
        assert orders[k] == (2 if k else 1)
        x_in = torch.zeros_like(k_in)
        t_in = torch.zeros_like(k_t)
        tag = L.NOISE_INJECT if cumulative else L.NOISE_INJECT_FRESH
        m, nxt = d._multistep(d._dpm_table(x.device, steps, order, cumulative), k, x, mo,
                              m_prev=mp if orders[k] == 2 else None, gt=gt, keep=keep,
                              inject_noise=seeded.Draw(seeds, tag, draws[k + 1]), stem=(x_in, t_in),
                              t_next=d._t_value(int(grid[k + 1])))
        assert torch.equal(xs, nxt) and torch.equal(ms, m), cumulative
        assert torch.equal(k_in, x_in) and torch.equal(k_t, t_in), cumulative


def test_k9_refuses_bad_arguments(lib):
    L = lib
    x = torch.zeros(2, 3, 8, 8, device=DEV)
    tab = torch.zeros(10, 7, device=DEV)
    tv = torch.zeros(10, device=DEV)
    ints = torch.zeros(10, dtype=torch.int32, device=DEV)
    x_in = torch.zeros(2, 8, 8, 16, device=DEV)
    a = L.MultistepArgs()
    a.batch, a.channels, a.hw, a.mask_channels, a.steps = 2, 3, 64, 1, 10
    a.mean_type, a.out_channels = L.MEAN_EPSILON, 3
    a.coef, a.x, a.model_out, a.m_prev, a.m_out, a.x_next, a.gt, a.keep_mask = (L.ptr(tab),) + (L.ptr(x),) * 7
    a.stem_out, a.stem_dtype, a.stem_ld = L.ptr(x_in), L.F32, 16
    s = L.MsSlotArgs()
    s.t_value, s.inject_draw, s.order, s.out = L.ptr(tv), L.ptr(ints), L.ptr(ints), L.ptr(x)
    s.inject_tag = L.NOISE_INJECT
    s.action[0], s.action[1] = L.SLOT_IDLE, L.SLOT_IDLE

    def rc():
        return L.lib().fidm_multistep_step_slots(ctypes.byref(a), ctypes.byref(s), L.stream())

    assert rc() == 0                                # every slot idle: the launch writes nothing
    torch.cuda.synchronize()
    for bad in (10, -3, 11):
        s.action[0] = bad
        assert rc() == -1 and b"multistep_step_slots" in L.lib().fidm_last_error_string(), bad
    s.action[0] = 3
    for name, val in (("batch", 0), ("batch", L.MAX_SLOTS + 1), ("mean_type", L.MEAN_PREVIOUS_X),
                      ("out_channels", 4), ("mask_channels", 2), ("inject_noise", L.ptr(x)), ("model_out", None),
                      ("coef", None), ("x", None), ("m_prev", None), ("m_out", None), ("x_next", None), ("gt", None),
                      ("keep_mask", None), ("stem_ld", 2), ("stem_dtype", 7), ("steps", 0)):
        old = getattr(a, name)
        setattr(a, name, val)
        assert rc() == -1 and b"multistep_step_slots" in L.lib().fidm_last_error_string(), name
        setattr(a, name, old)
    for name in ("out", "t_value", "inject_draw", "order"):
        old = getattr(s, name)
        setattr(s, name, None)
        assert rc() == -1, name
        setattr(s, name, old)
    for tag in (L.NOISE_XT, L.NOISE_STEP, L.NOISE_UNDO):
        s.inject_tag = tag
        assert rc() == -1, tag
    s.inject_tag = L.NOISE_INJECT
    assert L.lib().fidm_multistep_step_slots(None, ctypes.byref(s), L.stream()) == -1
    assert L.lib().fidm_multistep_step_slots(ctypes.byref(a), None, L.stream()) == -1
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ 2: the contract
def _standin(x, t, **k):
    """Per-sample elementwise eps model (test_gpu_continuous.py): its value per image is batch independent."""
    return torch.tanh(0.7 * x) * torch.cos(t.float().view(-1, 1, 1, 1) * 0.01) + 0.05 * k["gt"]


def _alone(d, model, steps, order, gt, keep, seed, schedule, cumulative):
    return d.dpm_solver_sample_loop(model, tuple(gt.shape), steps=steps, order=order,
                                    model_kwargs={"gt": gt, "gt_keep_mask": keep}, device=DEV,
                                    use_inpainting_injection=True, injection_schedule=schedule,
                                    use_cumulative_noise=cumulative, seeds=[seed])


def _staggered(cs, gts, keeps, seeds, plan):
    """Submit requests per `plan` ([number to submit before step i]) and step until done: [image per request]."""
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


CONTRACT = [(2, 8, "all", True, False), (2, 8, "high", False, True), (1, 8, "low", True, True),
            (2, 3, "all", False, False), (2, 2, "low", False, True), (1, 3, "high", True, False),
            (2, 12, "all", False, True)]


@pytest.mark.parametrize("order,steps,schedule,cumulative,rescale", CONTRACT)
def test_continuous_dpm_equals_each_request_alone(lib, order, steps, schedule, cumulative, rescale):
    import fidm_b200 as F
    d = F.create_gaussian_diffusion(steps=12, noise_schedule="cosine", rescale_timesteps=rescale)
    g = torch.Generator().manual_seed(11)
    S, n = 8, 7
    gts = [(torch.rand(3, S, S, generator=g) * 2 - 1).to(DEV) for _ in range(n)]
    keeps = [(torch.rand(1 if k % 2 else 3, S, S, generator=g) > 0.5).float().to(DEV) for k in range(n)]
    seeds = [5, 2 ** 64 - 1, 17, 17, 2 ** 40 + 3, 0, 99]
    cpu_state, cuda_state = torch.get_rng_state(), torch.cuda.get_rng_state()
    cs = d.continuous_dpm_solver_sampler(_standin, slots=3, image_size=(S, S), steps=steps, order=order,
                                         injection_schedule=schedule, use_cumulative_noise=cumulative, device=DEV)
    assert cs.plan is None
    got = _staggered(cs, gts, keeps, seeds, [2, 0, 1, 0, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 1])
    assert not cs.pending()
    assert torch.equal(torch.get_rng_state(), cpu_state) and torch.equal(torch.cuda.get_rng_state(), cuda_state)
    for k in range(n):
        want = _alone(d, _standin, steps, order, gts[k][None], keeps[k][None], seeds[k], schedule, cumulative)
        assert torch.equal(got[k], want), k
    assert torch.isfinite(torch.cat(got)).all() and not torch.equal(got[0], got[1])
    assert torch.equal(torch.get_rng_state(), cpu_state) and torch.equal(torch.cuda.get_rng_state(), cuda_state)
    assert not d._gt_noises_cache


# ------------------------------------------------------------------------------------------ 3: the UNet, bf16
def _unet(name, seed):
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_state_dict
    cfg = F.CONFIGS[name]
    m = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
    m.load_state_dict(synth_state_dict(cfg, seed=seed), strict=True)
    m.to(DEV)
    m.base_model.set_precision("bf16")
    return F.InpaintingModelFn(m)


def _run(d, fn, S, steps, plan):
    from fidm_b200.utils.synth import synth_batch
    data = synth_batch(4, S, seed=8, device=DEV)
    cs = d.continuous_dpm_solver_sampler(fn, slots=4, image_size=(S, S), steps=steps)
    got = torch.cat(_staggered(cs, list(data["gt"]), list(data["gt_keep_mask"]), [3, 2 ** 40, 77, 2 ** 63 + 1], plan))
    return cs, got, data


def test_t64_fused_equals_unfused(lib, monkeypatch):
    import fidm_b200 as F
    fn = _unet("T64", 2)
    d = F.create_gaussian_diffusion(steps=20, learn_sigma=True, noise_schedule="cosine")
    cs, fused, _ = _run(d, fn, 64, 8, [1, 2, 0, 0, 0, 1])
    assert cs.plan is not None
    monkeypatch.setenv("FIDM_FUSED_STEP", "0")
    cs, unfused, _ = _run(d, fn, 64, 8, [1, 2, 0, 0, 0, 1])
    assert cs.plan is None
    assert torch.isfinite(fused).all() and torch.equal(fused, unfused)


def test_ref_ffhq256_against_lockstep(lib):
    import fidm_b200 as F
    fn = _unet("REF_FFHQ256", 3)
    d = F.create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="quadratic")
    S = 256
    cs, got, data = _run(d, fn, S, 10, [2, 0, 1, 0, 1])
    assert cs.plan is not None
    gt, keep = data["gt"], data["gt_keep_mask"]
    lock = d.dpm_solver_sample_loop(fn, (4, 3, S, S), steps=10, model_kwargs={"gt": gt, "gt_keep_mask": keep},
                                    device=DEV, use_inpainting_injection=True, seeds=[3, 2 ** 40, 77, 2 ** 63 + 1])
    p = min(psnr(got[k][keep[k].expand(3, S, S) == 0], lock[k][keep[k].expand(3, S, S) == 0]) for k in range(4))
    print("REF-FFHQ256 DPM-Solver++ 2M-10 bf16 256x256: continuous (staggered admissions) vs lockstep batch 4, "
          "min hole PSNR %.1f dB, bit-identical: %s" % (p, torch.equal(got, lock)))
    assert torch.isfinite(got).all() and p >= 40.0, p


# ------------------------------------------------------------------------------------------ 4: no synchronisation
def test_fused_dpm_step_does_not_synchronise(lib):
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_batch
    fn = _unet("T64", 2)
    d = F.create_gaussian_diffusion(steps=20, learn_sigma=True, noise_schedule="cosine")
    data = synth_batch(3, 64, seed=1, device=DEV)
    cs = d.continuous_dpm_solver_sampler(fn, slots=2, image_size=(64, 64), steps=5)
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
