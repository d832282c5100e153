"""GPU: continuous batching of the RePaint loop -- K10 (fidm_repaint_step_slots) bit for bit against the seeded
lockstep launches per slot (K4 for an admission and a plain evaluation, K4 STEP_UPDATE_ONLY then K7 for a jump
evaluation), its argument checks, the continuous RePaint sampler against each request run alone through the seeded
repaint_sample_loop and, without jumps, against the continuous DDPM sampler, the T64 UNet fused against unfused and
against a lockstep batch, REF-FFHQ256 at 256x256 against a lockstep batch, and no synchronisation per iteration."""
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


def _diffusion(T, var, mean, rescale=False):
    import fidm_b200 as F
    from fidm_b200.utils.schedules import get_named_beta_schedule
    return F.GaussianDiffusion(betas=get_named_beta_schedule("cosine", T), model_mean_type=mean, model_var_type=var,
                               loss_type=F.LossType.MSE, rescale_timesteps=rescale)


# ------------------------------------------------------------------------------------------ 1: K10 against K4 (+ K7)
def _k10(L, d, jl, jn, x, mo, gt, keep, actions, seeds, *, clip, cumulative, schedule, stem, out, x_next):
    """One K10 launch on explicit buffers (as continuous.ContinuousRePaintSampler fills its arguments).  Returns the
    tables (eval_t, next_t, undo, inject_draw, admit_draw)."""
    from fidm_b200 import continuous
    from fidm_b200.gaussian_diffusion import _MEAN_CODE, _VAR_CODE
    B, Cn = x.shape[:2]
    T = d.num_timesteps
    tables = continuous.repaint_slot_tables(d, jl, jn, schedule, cumulative)
    eval_t, next_t, undo, draws, admit_draw = tables
    a = L.StepArgs()
    a.batch, a.channels, a.hw = B, Cn, x.numel() // (B * Cn)
    a.sampler = L.SAMPLER_DDPM
    a.mean_type, a.var_type = _MEAN_CODE[d.model_mean_type], _VAR_CODE[d.model_var_type]
    a.clip_denoised, a.cumulative, a.mask_channels, a.num_timesteps = int(clip), int(cumulative), keep.shape[1], T
    coef = d._coef(x.device, 0.0)
    tv = torch.tensor([d._t_value(t) for t in range(T)], dtype=torch.float32, device=DEV)
    et, nt, dr = (torch.tensor(v, dtype=torch.int32, device=DEV) for v in (eval_t, next_t, draws))
    ud = torch.tensor(undo, dtype=torch.float32, device=DEV)
    a.coef, a.x, a.model_out, a.gt, a.keep_mask, a.x_next = (L.ptr(v) for v in (coef, x, mo, gt, keep, x_next))
    x_in, t_in = stem
    a.stem_out, a.stem_dtype, a.stem_ld, a.t_out = L.ptr(x_in), L.dtype_code(x_in.dtype), x_in.shape[-1], L.ptr(t_in)
    s = L.RpSlotArgs()
    s.t_value, s.eval_t, s.next_t, s.undo, s.inject_draw, s.out = (L.ptr(v) for v in (tv, et, nt, ud, dr, out))
    s.n_evals, s.admit_draw = len(eval_t), admit_draw
    for b in range(B):
        s.action[b] = actions[b]
        s.seeds[b] = int(seeds[b]) & ((1 << 64) - 1)
    L.check(L.lib().fidm_repaint_step_slots(ctypes.byref(a), ctypes.byref(s), L.stream()), "repaint_step_slots")
    torch.cuda.synchronize()
    return tables


def _lockstep_alone(L, d, tables, x, mo, gt, keep, act, seeds, *, clip, cumulative, sdt):
    """What the seeded repaint_sample_loop computes for one image for K10's action `act`, with its own launches:
    (state, stem channels, t_out), or (sample, None, None) at the last evaluation."""
    from fidm_b200 import seeded
    eval_t, next_t, undo, draws, admit_draw = tables
    T = d.num_timesteps
    H, W = x.shape[2:]
    x_in = torch.full((1, H, W, 16), SENT, device=DEV, dtype=sdt)
    t_in = torch.full((1,), SENT, device=DEV)
    tag = L.NOISE_INJECT if cumulative else L.NOISE_INJECT_FRESH
    if act == L.SLOT_ADMIT:                          # K4 STEP_INJECT_ONLY on x_T
        xt = seeded.randn(seeds, tuple(x.shape), L.NOISE_XT, 0)
        if admit_draw < 0:
            x_in[..., :x.shape[1]] = xt.permute(0, 2, 3, 1).to(sdt)
            t_in.fill_(d._t_value(T - 1))
            return xt, x_in, t_in
        r = d._step(L.STEP_INJECT_ONLY, xt, t_inject=T - 1, gt=gt, keep=keep,
                    inject_noise=seeded.Draw(seeds, tag, admit_draw), cumulative=cumulative, want_next=True,
                    stem=(x_in, t_in), t_next=d._t_value(T - 1))
        return r["x_next"], x_in, t_in
    k = act
    t, nt, (ua, us), draw = eval_t[k], next_t[k], undo[k], draws[k]
    z = seeded.Draw(seeds, L.NOISE_STEP, k)
    inj = seeded.Draw(seeds, tag, draw) if draw >= 0 else None
    if nt == t - 1:                                  # K4 STEP_UPDATE_INJECT / STEP_UPDATE_ONLY
        r = d._step(L.STEP_UPDATE_INJECT if inj else L.STEP_UPDATE_ONLY, x, t=t, t_inject=t - 1, model_out=mo, z=z,
                    gt=gt if inj else None, keep=keep if inj else None, inject_noise=inj, ddim=False, clip=clip,
                    cumulative=cumulative, want_sample=t == 0, want_next=t > 0,
                    stem=(x_in, t_in) if t > 0 else None, t_next=d._t_value(t - 1) if t > 0 else None)
        if t == 0:
            return r["sample"], None, None
        return r["x_next"], x_in, t_in
    # a jump: K4 STEP_UPDATE_ONLY, then K7 (undo to t_up, injection at t_up)
    r = d._step(L.STEP_UPDATE_ONLY, x, t=t, model_out=mo, z=z, ddim=False, clip=clip, want_sample=True)
    nxt = d._resample(r["sample"], seeded.Draw(seeds, L.NOISE_UNDO, k), ua, us, t_inject=nt if inj else None,
                      gt=gt, keep=keep, inject_noise=inj, cumulative=cumulative, stem=(x_in, t_in),
                      t_next=d._t_value(nt))
    return nxt, x_in, t_in


def _model_kinds():
    from fidm_b200.losses import ModelMeanType as M, ModelVarType as V
    return [(V.LEARNED_RANGE, M.EPSILON), (V.FIXED_LARGE, M.EPSILON), (V.FIXED_SMALL, M.EPSILON),
            (V.LEARNED, M.EPSILON), (V.LEARNED_RANGE, M.START_X), (V.FIXED_LARGE, M.PREVIOUS_X)]


K10_CASES = list(itertools.product(range(6), [True, False]))        # model kind x cumulative / fresh


@pytest.mark.parametrize("kind,cumulative", K10_CASES)
def test_k10_slots_equal_seeded_lockstep_alone(lib, kind, cumulative):
    from fidm_b200 import continuous
    L = lib
    var, mean = _model_kinds()[kind]
    i = K10_CASES.index((kind, cumulative))
    T, jl, jn = 20, 4, 3
    d = _diffusion(T, var, mean, rescale=bool(i % 2))
    learn = var.name.startswith("LEARNED")
    # layouts x mask channels x stem dtypes x injection schedules x clipping, varied over the cases
    odd = (i // 2) % 2 == 1
    mc = 1 if i % 2 == 0 else 3
    sdt = (torch.bfloat16, torch.float16, torch.float32)[i % 3]
    schedule = ("all", "high", "low")[(i // 3) % 3]
    clip = i % 5 != 4
    H, W = (7, 9) if odd else (8, 8)
    eval_t, next_t, _, _, _ = continuous.repaint_slot_tables(d, jl, jn, schedule, cumulative)
    n = len(eval_t)
    assert n == 52
    jumps = [k for k in range(n) if next_t[k] != eval_t[k] - 1]
    plain = [k for k in range(n) if next_t[k] == eval_t[k] - 1]
    # a jump from above the high/low gate, one from below it, one whose t_up crosses it, and plain evaluations on
    # both sides of the gate
    gate = T // 2
    cross = [k for k in jumps if eval_t[k] - 1 < gate <= next_t[k]]
    pick = [jumps[0], jumps[-1], cross[0] if cross else jumps[1],
            next(k for k in plain if eval_t[k] == gate), next(k for k in plain if eval_t[k] == gate + 1)]
    actions = [L.SLOT_ADMIT, L.SLOT_IDLE, 0] + pick + [n - 2, n - 1, L.SLOT_IDLE]
    B, Cn = len(actions), 3
    seed_vals = [3 + 7 * b for b in range(B)]
    seed_vals[2], seed_vals[3] = 2 ** 64 - 1, 0
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
    kw = dict(clip=clip, cumulative=cumulative)
    tables = _k10(L, d, jl, jn, x, mo, gt, keep, actions, seed_vals, schedule=schedule, stem=(x_in, t_in), out=out,
                  x_next=x_next, **kw)
    for b, act in enumerate(actions):
        tag = (b, act)
        if act == L.SLOT_IDLE:
            assert (x_next[b] == SENT).all() and (out[b] == SENT).all(), tag
            assert (x_in[b].float() == SENT).all() and t_in[b].item() == SENT, tag
            continue
        want, w_stem, w_t = _lockstep_alone(L, d, tables, x[b:b + 1], mo[b:b + 1], gt[b:b + 1], keep[b:b + 1], act,
                                            seeds[b:b + 1], sdt=sdt, **kw)
        if act == n - 1:
            assert torch.equal(out[b:b + 1], want), tag
            assert (x_next[b] == SENT).all() and (x_in[b].float() == SENT).all() and t_in[b].item() == SENT, tag
            continue
        assert (out[b] == SENT).all(), tag
        assert torch.isfinite(x_next[b]).all(), tag
        assert torch.equal(x_next[b:b + 1], want), tag
        assert torch.equal(x_in[b:b + 1, :, :, :Cn], w_stem[:, :, :, :Cn]), tag
        assert (x_in[b, :, :, Cn:].float() == SENT).all(), tag                # conditioning channels untouched
        assert torch.equal(t_in[b:b + 1], w_t), tag


def test_k10_refuses_bad_arguments(lib):
    L = lib
    x = torch.zeros(2, 3, 8, 8, device=DEV)
    tab = torch.zeros(10, L.COEF_COLS, device=DEV)
    tv = torch.zeros(10, device=DEV)
    ints = torch.zeros(30, dtype=torch.int32, device=DEV)
    undo = torch.zeros(30, 2, device=DEV)
    x_in = torch.zeros(2, 8, 8, 16, device=DEV)
    a = L.StepArgs()
    a.batch, a.channels, a.hw, a.mask_channels, a.num_timesteps = 2, 3, 64, 1, 10
    a.sampler, a.mean_type, a.var_type = L.SAMPLER_DDPM, L.MEAN_EPSILON, L.VAR_FIXED
    a.coef, a.x, a.model_out, a.gt, a.keep_mask, a.x_next = (L.ptr(tab),) + (L.ptr(x),) * 5
    a.stem_out, a.stem_dtype, a.stem_ld = L.ptr(x_in), L.F32, 16
    s = L.RpSlotArgs()
    s.t_value, s.eval_t, s.next_t, s.undo, s.inject_draw, s.out = (L.ptr(v) for v in (tv, ints, ints, undo, ints, x))
    s.n_evals, s.admit_draw = 30, -1
    s.action[0], s.action[1] = L.SLOT_IDLE, L.SLOT_IDLE

    def rc():
        return L.lib().fidm_repaint_step_slots(ctypes.byref(a), ctypes.byref(s), L.stream())

    def refused(what):
        assert rc() == -1 and b"repaint_step_slots" in L.lib().fidm_last_error_string(), what

    assert rc() == 0                                # every slot idle: the launch writes nothing
    torch.cuda.synchronize()
    for bad in (30, -3, 31):
        s.action[0] = bad
        refused(bad)
    s.action[0] = 3
    for name, val in (("batch", 0), ("batch", L.MAX_SLOTS + 1), ("sampler", L.SAMPLER_DDIM),
                      ("sampler", L.SAMPLER_DDIM_SCRIPT), ("mask_channels", 2), ("model_out", None), ("coef", None),
                      ("x", None), ("x_next", None), ("gt", None), ("keep_mask", None), ("z", L.ptr(x)),
                      ("inject_noise", L.ptr(x)), ("t_dev", L.ptr(x)), ("sample", L.ptr(x)),
                      ("pred_xstart", L.ptr(x)), ("mean_out", L.ptr(x)), ("logvar_out", L.ptr(x)), ("stem_ld", 2),
                      ("stem_dtype", 7), ("num_timesteps", 0)):
        old = getattr(a, name)
        setattr(a, name, val)
        refused(name)
        setattr(a, name, old)
    for name in ("out", "t_value", "eval_t", "next_t", "undo", "inject_draw"):
        old = getattr(s, name)
        setattr(s, name, None)
        refused(name)
        setattr(s, name, old)
    s.n_evals = 0
    refused("n_evals")
    s.n_evals = 30
    s.action[0] = L.SLOT_ADMIT                      # an admission reads no model output
    a.model_out = None
    assert rc() == 0
    assert L.lib().fidm_repaint_step_slots(None, ctypes.byref(s), L.stream()) == -1
    assert L.lib().fidm_repaint_step_slots(ctypes.byref(a), None, L.stream()) == -1
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ 2: the contract
def _standin(x, t, **k):
    """Per-sample elementwise eps model (test_gpu_continuous.py): its value per image is batch independent."""
    return torch.tanh(0.7 * x) * torch.cos(t.float().view(-1, 1, 1, 1) * 0.01) + 0.05 * k["gt"]


def _alone(d, model, jl, jn, gt, keep, seed, schedule, cumulative):
    return d.repaint_sample_loop(model, tuple(gt.shape), jump_length=jl, jump_n_sample=jn,
                                 model_kwargs={"gt": gt, "gt_keep_mask": keep}, device=DEV,
                                 injection_schedule=schedule, use_cumulative_noise=cumulative, seeds=[seed])


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


def _requests(n, S, seed):
    g = torch.Generator().manual_seed(seed)
    gts = [(torch.rand(3, S, S, generator=g) * 2 - 1).to(DEV) for _ in range(n)]
    keeps = [(torch.rand(1 if k % 2 else 3, S, S, generator=g) > 0.5).float().to(DEV) for k in range(n)]
    return gts, keeps


# a request takes 30 evaluations at (3, 3) on T = 12: submissions while slots are busy, idle slots, a late request
PLAN = [2, 0, 1] + [0] * 30 + [3] + [0] * 40 + [1]
CONTRACT = [(3, 3, "all", True, False), (3, 3, "high", False, True), (3, 3, "low", True, True),
            (3, 3, "all", False, False), (2, 4, "low", False, False), (5, 2, "high", True, True)]


@pytest.mark.parametrize("jl,jn,schedule,cumulative,rescale", CONTRACT)
def test_continuous_repaint_equals_each_request_alone(lib, jl, jn, schedule, cumulative, rescale):
    import fidm_b200 as F
    d = F.create_gaussian_diffusion(steps=12, noise_schedule="cosine", rescale_timesteps=rescale)
    S, n = 8, 7
    gts, keeps = _requests(n, S, 11)
    seeds = [5, 2 ** 64 - 1, 17, 17, 2 ** 40 + 3, 0, 99]
    cpu_state, cuda_state = torch.get_rng_state(), torch.cuda.get_rng_state()
    cs = d.continuous_repaint_sampler(_standin, slots=3, image_size=(S, S), jump_length=jl, jump_n_sample=jn,
                                      injection_schedule=schedule, use_cumulative_noise=cumulative, device=DEV)
    assert cs.plan is None
    got = _staggered(cs, gts, keeps, seeds, PLAN)
    assert not cs.pending()
    assert torch.equal(torch.get_rng_state(), cpu_state) and torch.equal(torch.cuda.get_rng_state(), cuda_state)
    assert not d._gt_noises_cache
    for k in range(n):
        want = _alone(d, _standin, jl, jn, gts[k][None], keeps[k][None], seeds[k], schedule, cumulative)
        assert torch.equal(got[k], want), k
    assert torch.isfinite(torch.cat(got)).all() and not torch.equal(got[0], got[1])
    assert torch.equal(got[2], got[3]) == torch.equal(gts[2] * keeps[2], gts[3] * keeps[3])
    assert torch.equal(torch.get_rng_state(), cpu_state) and torch.equal(torch.cuda.get_rng_state(), cuda_state)
    assert not d._gt_noises_cache


@pytest.mark.parametrize("schedule,cumulative", [("all", True), ("high", False), ("low", True)])
def test_without_jumps_equals_continuous_ddpm(lib, schedule, cumulative):
    import fidm_b200 as F
    d = F.create_gaussian_diffusion(steps=12, noise_schedule="cosine", learn_sigma=False)
    S, n = 8, 5
    gts, keeps = _requests(n, S, 4)
    seeds = [1, 2, 2 ** 63, 4, 5]
    kw = dict(slots=2, image_size=(S, S), injection_schedule=schedule, use_cumulative_noise=cumulative, device=DEV)
    rp = _staggered(d.continuous_repaint_sampler(_standin, jump_length=3, jump_n_sample=1, **kw), gts, keeps, seeds,
                    [1, 0, 2, 0, 0, 1])
    dd = _staggered(d.continuous_sampler(_standin, sampler="ddpm", **kw), gts, keeps, seeds, [1, 0, 2, 0, 0, 1])
    for k in range(n):
        assert torch.equal(rp[k], dd[k]), k


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


SEEDS4 = [3, 2 ** 40, 77, 2 ** 63 + 1]


def _run(d, fn, S, jl, jn, plan):
    from fidm_b200.utils.synth import synth_batch
    data = synth_batch(4, S, seed=8, device=DEV)
    cs = d.continuous_repaint_sampler(fn, slots=4, image_size=(S, S), jump_length=jl, jump_n_sample=jn)
    got = torch.cat(_staggered(cs, list(data["gt"]), list(data["gt_keep_mask"]), SEEDS4, plan))
    return cs, got, data


def _lockstep(d, fn, S, jl, jn, data):
    gt, keep = data["gt"], data["gt_keep_mask"]
    return d.repaint_sample_loop(fn, (4, 3, S, S), jump_length=jl, jump_n_sample=jn,
                                 model_kwargs={"gt": gt, "gt_keep_mask": keep}, device=DEV, seeds=SEEDS4)


def _hole_psnr(got, lock, keep, S):
    return min(psnr(got[k][keep[k].expand(3, S, S) == 0], lock[k][keep[k].expand(3, S, S) == 0])
               for k in range(got.shape[0]))


def test_t64_fused_equals_unfused_and_lockstep(lib, monkeypatch):
    import fidm_b200 as F
    fn = _unet("T64", 2)
    d = F.create_gaussian_diffusion(steps=20, learn_sigma=True, noise_schedule="cosine")
    S, jl, jn = 64, 4, 3
    stagger = [1, 2, 0, 0, 0, 1]
    cs, fused, data = _run(d, fn, S, jl, jn, stagger)
    assert cs.plan is not None and cs.schedule.T == 52
    lock = _lockstep(d, fn, S, jl, jn, data)
    p = _hole_psnr(fused, lock, data["gt_keep_mask"], S)
    print("T64 RePaint(4, 3) T=20 bf16: continuous (staggered admissions) vs lockstep batch 4, min hole PSNR %.1f dB, "
          "bit-identical: %s" % (p, torch.equal(fused, lock)))
    assert torch.isfinite(fused).all() and p >= 40.0, p
    _, together, _ = _run(d, fn, S, jl, jn, [4])           # all admitted in the first iteration: the lockstep batch
    assert torch.equal(together, lock)
    monkeypatch.setenv("FIDM_FUSED_STEP", "0")
    cs, unfused, _ = _run(d, fn, S, jl, jn, stagger)
    assert cs.plan is None
    assert torch.equal(fused, unfused)


def test_ref_ffhq256_against_lockstep(lib):
    import fidm_b200 as F
    fn = _unet("REF_FFHQ256", 3)
    d = F.create_gaussian_diffusion(steps=10, learn_sigma=True, noise_schedule="cosine")
    S, jl, jn = 256, 2, 2
    cs, got, data = _run(d, fn, S, jl, jn, [2, 0, 1, 0, 1])
    assert cs.plan is not None and cs.schedule.T == 18
    lock = _lockstep(d, fn, S, jl, jn, data)
    p = _hole_psnr(got, lock, data["gt_keep_mask"], S)
    print("REF-FFHQ256 RePaint(2, 2) T=10 bf16 256x256: continuous (staggered admissions) vs lockstep batch 4, "
          "min hole PSNR %.1f dB, bit-identical: %s" % (p, torch.equal(got, lock)))
    assert torch.isfinite(got).all() and p >= 40.0, p


# ------------------------------------------------------------------------------------------ 4: no synchronisation
def test_fused_repaint_step_does_not_synchronise(lib):
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_batch
    fn = _unet("T64", 2)
    d = F.create_gaussian_diffusion(steps=6, learn_sigma=True, noise_schedule="cosine")
    data = synth_batch(3, 64, seed=1, device=DEV)
    cs = d.continuous_repaint_sampler(fn, slots=2, image_size=(64, 64), jump_length=2, jump_n_sample=2)
    assert cs.schedule.T == 10 and any(a != b - 1 for a, b in zip(cs._next_t.tolist(), cs._eval_t.tolist()))
    for k in range(3):
        cs.submit(data["gt"][k], data["gt_keep_mask"][k], k)
    cs.step()                                        # warm-up: graph capture, first admissions
    torch.cuda.synchronize()
    done = []
    try:
        torch.cuda.set_sync_debug_mode("error")
        while cs.pending():
            done += cs.step()                        # steady iterations with jumps, a finish, an admission
        cs.submit(data["gt"][0], data["gt_keep_mask"][0], 9)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert len(done) == 3
    assert cs.drain() and not cs.pending()
