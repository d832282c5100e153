"""GPU: per-image seeded noise -- fidm_randn_seeded against the Philox oracle and N(0, 1), every seeded sampler entry bit
for bit against its unseeded launch fed fidm_randn_seeded tensors, batch invariance of every loop, the T64 UNet fused
against unfused, the real bf16 engine alone against a batch of 4, and the RePaint harmonization bars in seeded mode."""
import ctypes
import itertools
import math

import numpy as np
import pytest
import torch

from helpers import psnr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SEEDS = [0, 1, 2 ** 32 + 7, 2 ** 63 + 5, 2 ** 64 - 1]


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


def _diffusion(steps, schedule="cosine", **kw):
    import fidm_b200 as F
    return F.create_gaussian_diffusion(steps=steps, noise_schedule=schedule, **kw)


# ------------------------------------------------------------------------------------------ 1: the generator
def _fill(L, seeds, B, n, tag, draw, misaligned=False):
    buf = torch.full((B * n + 1,), float("nan"), device=DEV)
    out = buf[1:] if misaligned else buf[:-1]
    L.check(L.lib().fidm_randn_seeded(L.ptr(out), L.ptr(seeds), B, n, tag, draw, L.stream()), "randn_seeded")
    return out.view(B, n)


@pytest.mark.parametrize("hw,misaligned", [((8, 8), False), ((7, 9), False), ((8, 8), True)])
def test_randn_seeded_matches_oracle(lib, hw, misaligned):
    from oracle import philox_oracle as P
    B, C = len(SEEDS), 3
    n = C * hw[0] * hw[1]
    seeds = _seeds(SEEDS)
    for tag, draw in ((0, 0), (1, 17), (2, 999), (3, 4), (4, 2 ** 31 - 1)):
        got = _fill(lib, seeds, B, n, tag, draw, misaligned).cpu().double().numpy()
        want = P.randn(SEEDS, (B, n), tag, draw)
        assert np.all(np.abs(got - want) <= 1e-5 * np.maximum(1.0, np.abs(want))), (hw, misaligned, tag, draw)


def test_randn_seeded_distribution(lib):
    from scipy import stats
    from fidm_b200 import seeded
    seeds = _seeds(list(range(100, 116)))
    shape = (16, 3, 256, 256)
    x = seeded.randn(seeds, shape, 1, 3).double().flatten()
    N = x.numel()
    assert N >= 3_000_000
    mean, var = x.mean().item(), x.var().item()
    assert abs(mean) < 5 / math.sqrt(N) and abs(var - 1) < 5 * math.sqrt(2 / N), (mean, var)
    xs = x.cpu().numpy()
    p = stats.kstest(xs[::4], "norm").pvalue              # 1M points: the KS statistic resolves ~1e-3 in the CDF
    assert p > 1e-3, p
    for k in (3, 4):
        pk = 2 * stats.norm.sf(k)
        cnt = int((np.abs(xs) > k).sum())
        assert abs(cnt - N * pk) < 5 * math.sqrt(N * pk * (1 - pk)) + 1, (k, cnt, N * pk)
    assert np.abs(xs).max() < 6.8

    def corr(a, b):
        a, b = a.flatten() - a.mean(), b.flatten() - b.mean()
        return abs((a * b).sum().item() / math.sqrt((a * a).sum().item() * (b * b).sum().item()))

    bar = 5 / math.sqrt(N)
    assert corr(x[:-1], x[1:]) < 5 / math.sqrt(N - 1)                                  # adjacent elements
    for other in (seeded.randn(seeds, shape, 1, 4),                                      # next draw
                  seeded.randn(seeds, shape, 2, 3),                                      # other tag
                  seeded.randn(_seeds(list(range(101, 117))), shape, 1, 3)):            # seeds s + 1
        assert corr(x, other.double()) < bar


# ------------------------------------------------------------------------------------------ 2: seeded = unseeded + fill
def _layout(t, layout):
    if layout != "misaligned":
        return t
    v = torch.cat([torch.zeros(1, device=DEV), t.reshape(-1)])[1:].view(t.shape)
    assert v.data_ptr() % 16 != 0
    return v


def _same(a, b, tag):
    for k in a:
        assert torch.equal(a[k], b[k]), (k, tag)


def test_sampler_step_seeded_bit_identical(lib):
    from fidm_b200 import seeded
    L = lib
    n_cases = 0
    for learn, layout, sdt in itertools.product((True, False), ("vec4", "odd", "misaligned"),
                                                (torch.float32, torch.bfloat16, torch.float16)):
        d = _diffusion(50, learn_sigma=learn)
        H, W = (7, 9) if layout == "odd" else (8, 8)
        B, C = 3, 3
        seeds = _seeds(SEEDS[:B])
        g = torch.Generator().manual_seed(n_cases)
        x = _layout((torch.randn(B, C, H, W, generator=g) * 1.5).to(DEV), layout)
        mo = torch.randn(B, 2 * C if learn else C, H, W, generator=g).to(DEV)
        gt = (torch.rand(B, C, H, W, generator=g) * 2 - 1).to(DEV)
        keep = (torch.rand(B, 1, H, W, generator=g) > 0.5).float().to(DEV)
        for mode, (ddim, eta), cumulative in itertools.product(
                (L.STEP_INJECT_ONLY, L.STEP_UPDATE_ONLY, L.STEP_UPDATE_INJECT),
                ((True, 0.0), (True, 0.7), (False, 0.0)), (True, False)):
            z_draw = seeded.Draw(seeds, L.NOISE_STEP, 11) if (not ddim or eta != 0.0) else None
            itag = L.NOISE_INJECT if cumulative else L.NOISE_INJECT_FRESH
            n_draw = seeded.Draw(seeds, itag, 23)
            z = seeded.randn(seeds, x.shape, L.NOISE_STEP, 11) if z_draw else None
            n = seeded.randn(seeds, x.shape, itag, 23)
            upd, inj = mode != L.STEP_INJECT_ONLY, mode != L.STEP_UPDATE_ONLY
            outs = []
            for zz, nn in ((z_draw, n_draw), (z, n)):
                x_in = torch.zeros(B, H, W, 16, device=DEV, dtype=sdt)
                t_in = torch.zeros(B, device=DEV)
                r = d._step(mode, x, t=30 if upd else None, t_inject=29 if inj else None,
                            model_out=mo if upd else None, z=zz if upd else None, gt=gt if inj else None,
                            keep=keep if inj else None, inject_noise=nn if inj else None, ddim=ddim, eta=eta,
                            cumulative=cumulative, want_sample=upd, want_x0=upd, want_next=True,
                            want_mean=upd, want_logvar=upd, stem=(x_in, t_in), t_next=29.0)
                r["stem"], r["t"] = x_in, t_in
                outs.append(r)
            _same(outs[0], outs[1], (learn, layout, sdt, mode, ddim, eta, cumulative))
            n_cases += 1
    assert n_cases == 2 * 3 * 3 * 18


def test_multistep_seeded_bit_identical(lib):
    from fidm_b200 import seeded
    L = lib
    d = _diffusion(100, learn_sigma=True)
    for order, layout, sdt, cumulative in itertools.product((1, 2), ("vec4", "odd", "misaligned"),
                                                            (torch.float32, torch.bfloat16, torch.float16),
                                                            (True, False)):
        tab = d._dpm_table(torch.device(DEV), 10, order, cumulative)
        H, W = (7, 9) if layout == "odd" else (8, 8)
        B, C = 3, 3
        seeds = _seeds(SEEDS[-B:])
        g = torch.Generator().manual_seed(order)
        x = _layout(torch.randn(B, C, H, W, generator=g).to(DEV), layout)
        mo = torch.randn(B, 2 * C, H, W, generator=g).to(DEV)
        mp = torch.randn(B, C, H, W, generator=g).to(DEV)
        gt = (torch.rand(B, C, H, W, generator=g) * 2 - 1).to(DEV)
        keep = (torch.rand(B, 3, H, W, generator=g) > 0.5).float().to(DEV)
        itag = L.NOISE_INJECT if cumulative else L.NOISE_INJECT_FRESH
        outs = []
        for nn in (seeded.Draw(seeds, itag, 7), seeded.randn(seeds, x.shape, itag, 7)):
            x_in = torch.zeros(B, H, W, 16, device=DEV, dtype=sdt)
            t_in = torch.zeros(B, device=DEV)
            m, nxt = d._multistep(tab, 4, x, mo, m_prev=mp if order == 2 else None, gt=gt, keep=keep,
                                  inject_noise=nn, stem=(x_in, t_in), t_next=12.0)
            outs.append({"m": m, "x": nxt, "stem": x_in, "t": t_in})
        _same(outs[0], outs[1], (order, layout, sdt, cumulative))


def test_resample_seeded_bit_identical(lib):
    from fidm_b200 import seeded
    L = lib
    d = _diffusion(100)
    for inj, layout, sdt in itertools.product(("off", "cumulative", "fresh"), ("vec4", "odd", "misaligned"),
                                              (torch.float32, torch.bfloat16, torch.float16)):
        H, W = (7, 9) if layout == "odd" else (8, 8)
        B, C = 2, 3
        seeds = _seeds([SEEDS[1], SEEDS[3]])
        g = torch.Generator().manual_seed(5)
        x = _layout(torch.randn(B, C, H, W, generator=g).to(DEV), layout)
        gt = (torch.rand(B, C, H, W, generator=g) * 2 - 1).to(DEV)
        keep = (torch.rand(B, 1, H, W, generator=g) > 0.5).float().to(DEV)
        itag = L.NOISE_INJECT if inj == "cumulative" else L.NOISE_INJECT_FRESH
        outs = []
        for u, nn in ((seeded.Draw(seeds, L.NOISE_UNDO, 9), seeded.Draw(seeds, itag, 57)),
                      (seeded.randn(seeds, x.shape, L.NOISE_UNDO, 9), seeded.randn(seeds, x.shape, itag, 57))):
            x_in = torch.zeros(B, H, W, 16, device=DEV, dtype=sdt)
            t_in = torch.zeros(B, device=DEV)
            out = d._resample(x, u, 0.93, 0.37, t_inject=57 if inj != "off" else None, gt=gt, keep=keep,
                              inject_noise=nn if inj != "off" else None, cumulative=inj != "fresh",
                              stem=(x_in, t_in), t_next=57.0)
            outs.append({"x": out, "stem": x_in, "t": t_in})
        _same(outs[0], outs[1], (inj, layout, sdt))


def test_seeded_entries_refuse_noise_pointers(lib):
    L = lib
    x = torch.zeros(1, 3, 8, 8, device=DEV)
    seeds = _seeds([1])
    s = L.SeededNoise()
    s.seeds, s.draw = L.ptr(seeds), 0
    a = L.ResampleArgs()
    a.batch, a.channels, a.hw, a.mask_channels = 1, 3, 64, 1
    a.x, a.x_next, a.noise = L.ptr(x), L.ptr(x), L.ptr(x)
    assert L.lib().fidm_resample_undo_seeded(ctypes.byref(a), ctypes.byref(s), L.stream()) == -1
    assert b"resample_undo_seeded" in L.lib().fidm_last_error_string()
    a.noise = None
    assert L.lib().fidm_resample_undo_seeded(ctypes.byref(a), None, L.stream()) == -1
    assert L.lib().fidm_resample_undo_seeded(ctypes.byref(a), ctypes.byref(s), L.stream()) == 0
    st = L.StepArgs()                                                       # K4 seeded: loops only, no t_dev
    t_dev = torch.zeros(1, dtype=torch.int64, device=DEV)
    st.batch, st.channels, st.hw, st.mode, st.mask_channels, st.num_timesteps = 1, 3, 64, L.STEP_UPDATE_ONLY, 1, 10
    st.coef, st.x, st.model_out, st.t_dev = L.ptr(x), L.ptr(x), L.ptr(x), L.ptr(t_dev)
    assert L.lib().fidm_sampler_step_seeded(ctypes.byref(st), ctypes.byref(s), L.stream()) == -1
    assert b"sampler_step_seeded" in L.lib().fidm_last_error_string()
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------ 3: batch invariance
def _standin(x, t, **k):
    """Per-sample elementwise eps model: no reduction over the batch, so its value per image is batch independent."""
    return torch.tanh(0.7 * x) * torch.cos(t.float().view(-1, 1, 1, 1) * 0.01) + 0.05 * k["gt"]


LOOP_CASES = [("ddim", {}), ("ddim", {"eta": 0.6}), ("ddpm", {}), ("dpm_solver", {"steps": 8, "order": 2}),
              ("repaint", {"jump_length": 3, "jump_n_sample": 3})]


def _run_loop(d, loop, extra, gt, keep, seeds, cumulative, model=_standin, **kw):
    fns = {"ddim": d.ddim_sample_loop, "ddpm": d.p_sample_loop, "dpm_solver": d.dpm_solver_sample_loop,
           "repaint": d.repaint_sample_loop}
    return fns[loop](model, tuple(gt.shape), model_kwargs={"gt": gt, "gt_keep_mask": keep}, device=DEV,
                     use_inpainting_injection=True, use_cumulative_noise=cumulative, seeds=seeds, **extra, **kw)


@pytest.mark.parametrize("loop,extra", LOOP_CASES)
@pytest.mark.parametrize("cumulative", [True, False])
def test_loops_are_batch_invariant(lib, loop, extra, cumulative, monkeypatch):
    import fidm_b200.parallel as par
    d = _diffusion(20)
    g = torch.Generator().manual_seed(3)
    S = 8
    gts = (torch.rand(7, 3, S, S, generator=g) * 2 - 1).to(DEV)
    keeps = (torch.rand(7, 1, S, S, generator=g) > 0.5).float().to(DEV)
    sd = [11, 2 ** 64 - 3, 5, 6, 7, 8, 9]
    cpu_state, cuda_state = torch.get_rng_state(), torch.cuda.get_rng_state()
    alone = _run_loop(d, loop, extra, gts[:1], keeps[:1], sd[:1], cumulative)
    a = [0, 1, 2, 3]
    b = [4, 5, 0, 6]
    out_a = _run_loop(d, loop, extra, gts[a], keeps[a], [sd[i] for i in a], cumulative)
    out_b = _run_loop(d, loop, extra, gts[b], keeps[b], torch.tensor([sd[i] for i in b], dtype=torch.uint64),
                      cumulative)
    assert torch.equal(out_a[0], alone[0]) and torch.equal(out_b[2], alone[0])
    assert torch.isfinite(out_a).all() and not torch.equal(out_a[0], out_a[1])
    # sample_sharded over 2 ranks: each rank's shard equals its slice of the one-GPU batch
    monkeypatch.setattr(par.dist, "is_initialized", lambda: True)
    monkeypatch.setattr(par.dist, "get_world_size", lambda: 2)
    monkeypatch.setattr(par, "gather_batch", lambda local, batch: local)
    sampler = loop if loop != "ddim" else "ddim"
    for rank in (0, 1):
        monkeypatch.setattr(par.dist, "get_rank", lambda rank=rank: rank)
        kw = {k: v for k, v in extra.items() if k != "eta"}
        got = par.sample_sharded(d, _standin, gts[a], keeps[a], sampler=sampler, eta=extra.get("eta", 0.0),
                                 seeds=[sd[i] for i in a], use_cumulative_noise=cumulative, **kw)
        assert torch.equal(got, out_a[2 * rank: 2 * rank + 2]), rank
    # duplicate seeds on the same inputs give duplicate images
    dup = _run_loop(d, loop, extra, gts[[0, 0, 0]], keeps[[0, 0, 0]], [sd[0], sd[0], sd[1]], cumulative)
    assert torch.equal(dup[0], dup[1]) and torch.equal(dup[0], alone[0]) and not torch.equal(dup[0], dup[2])
    assert torch.equal(torch.get_rng_state(), cpu_state) and torch.equal(torch.cuda.get_rng_state(), cuda_state)
    assert not d._gt_noises_cache


# ------------------------------------------------------------------------------------------ 4: T64 fused = unfused
@pytest.mark.parametrize("loop,extra", LOOP_CASES)
def test_t64_seeded_fused_equals_unfused(lib, loop, extra, monkeypatch):
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_batch, synth_state_dict
    cfg = F.CONFIGS["T64"]
    m = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
    m.load_state_dict(synth_state_dict(cfg, seed=2), strict=True)
    m.to(DEV)
    m.base_model.set_precision("bf16")
    fn = F.InpaintingModelFn(m)
    d = _diffusion(20, learn_sigma=True)
    data = synth_batch(2, 64, seed=8, device=DEV)
    outs = {}
    for fused in ("1", "0"):
        monkeypatch.setenv("FIDM_FUSED_STEP", fused)
        outs[fused] = _run_loop(d, loop, extra, data["gt"], data["gt_keep_mask"], [3, 2 ** 40], True, model=fn)
    assert torch.isfinite(outs["1"]).all() and torch.equal(outs["1"], outs["0"]), loop


# ------------------------------------------------------------------------------------------ 5: the real bf16 engine
def test_ref_ffhq256_alone_vs_batch_of_4(lib):
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_batch, synth_state_dict
    cfg = F.CONFIGS["REF_FFHQ256"]
    m = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
    m.load_state_dict(synth_state_dict(cfg, seed=3), strict=True)
    m.to(DEV)
    m.base_model.set_precision("bf16")
    fn = F.InpaintingModelFn(m)
    d = _diffusion(100, learn_sigma=True)
    data = synth_batch(4, 256, seed=5, device=DEV)
    gt, keep = data["gt"], data["gt_keep_mask"]
    seeds = [21, 22, 23, 24]
    four = _run_loop(d, "ddim", {}, gt, keep, seeds, True, model=fn)
    alone = _run_loop(d, "ddim", {}, gt[2:3], keep[2:3], seeds[2:3], True, model=fn)
    hole = (keep[2:3] == 0).expand_as(alone)
    p = psnr(alone[hole], four[2:3][hole])
    print("REF-FFHQ256 DDIM-100 bf16, image alone vs in a batch of 4: hole PSNR %.1f dB, bit-identical: %s"
          % (p, torch.equal(alone, four[2:3])))
    assert p >= 40.0, p


# ------------------------------------------------------------------------------------------ 6: harmonization, seeded
@pytest.mark.parametrize("seed", [1, 2])
def test_harmonization_seeded(lib, seed):
    from oracle import repaint_oracle as O
    torch.backends.cuda.matmul.allow_tf32 = False
    d = _diffusion(100, "linear", sigma_small=True)
    am = O.CorrelatedGaussian(d.alphas_cumprod, 8, 8)
    gt = am.sample_prior(1, torch.Generator().manual_seed(seed))
    keep = torch.zeros(1, 1, 8, 8)
    keep[..., :4] = 1
    B = 4000
    mk = {"gt": gt.float().expand(B, 1, 8, 8).contiguous().to(DEV), "gt_keep_mask": keep.expand(B, 1, 8, 8).to(DEV)}
    model = lambda x, t, **k: am.eps(x, int(t[0])).float()  # noqa: E731
    mean, cov = am.hole_conditional(gt[0], keep[0])
    seeds = [seed * 1_000_003 + i for i in range(B)]
    errs = {}
    for jn in (1, 10):
        out = d.repaint_sample_loop(model, (B, 1, 8, 8), jump_length=10, jump_n_sample=jn, clip_denoised=False,
                                    model_kwargs=mk, device=DEV, seeds=seeds)
        errs[jn] = O.harmonization_errors(out.cpu(), keep, mean, cov)
    plain, rp = errs[1], errs[10]
    print("seeded, seed %d: plain injection mean RMS %.4f cov %.4f | RePaint(10, 10) mean RMS %.4f cov %.4f"
          % (seed, *plain, *rp))
    assert plain[1] >= 0.25, plain
    assert rp[1] <= 0.12 and rp[1] <= 0.35 * plain[1], (rp, plain)
