"""GPU: RePaint resampling -- K7 (fidm_resample_undo) bit-exact against its fp32 op-order mirror, the loop without jumps
against p_sample_loop, the T64 UNet fused against unfused with jumps, the public loop against the float64 oracle fed the
same noise, the harmonization bars on the analytic model, a 256x256 UNet loop's known region, sharding and errors."""
import ctypes
import hashlib
import itertools

import numpy as np
import pytest
import torch

from helpers import _REAL_RANDN, rel_l2

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


def _diffusion(steps, schedule="cosine", **kw):
    import fidm_b200 as F
    return F.create_gaussian_diffusion(steps=steps, noise_schedule=schedule, **kw)


def _model(cfg, sd, precision):
    import fidm_b200 as F
    m = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
    m.load_state_dict(sd, strict=True)
    m.to(DEV)
    m.base_model.set_precision(precision)
    return m


def _inpaint_data(B, S, seed):
    from fidm_b200.utils.synth import synth_batch
    data = synth_batch(B, S, seed=seed, device=DEV)
    return {"gt": data["gt"], "gt_keep_mask": data["gt_keep_mask"]}


# ------------------------------------------------------------------------------------------ 1: one K7 launch
def test_kernel_bit_exact_against_fp32_mirror(lib):
    """Every switch of one K7 launch against oracle/repaint_oracle.mirror_undo, bit for bit, on the vec4 path (8x8) and
    the scalar path (7x9, and 8x8 at a misaligned address); known pixels after an injection are exactly
    fl(fl(ia*gt) + fl(is*n)); the stem input is x_next rounded as the pack kernel rounds; t_out is written."""
    from oracle import repaint_oracle as O
    d = _diffusion(100)
    cls = d.coefficient_table(0.0)
    t_up, n_cases = 57, 0
    for inj, mch, layout, sdt in itertools.product(("off", "cumulative", "fresh"), (1, 3),
                                                    ("vec4", "odd", "misaligned"),
                                                    (torch.float32, torch.bfloat16, torch.float16)):
        if inj == "off" and mch == 3:
            continue
        H, W = (7, 9) if layout == "odd" else (8, 8)
        g = torch.Generator().manual_seed(n_cases)
        B, C = 2, 3
        x, u, n = (torch.randn(B, C, H, W, generator=g) * s for s in (2.0, 1.0, 1.0))
        gt = torch.rand(B, C, H, W, generator=g) * 2 - 1
        keep = (torch.rand(B, mch, H, W, generator=g) > 0.4).float()
        a_u, s_u = (float(np.float32(v)) for v in (0.93, 0.37))
        ia, is_ = (0, 1) if inj == "cumulative" else (2, 3)
        want = O.mirror_undo(x, u, a_u, s_u, gt=gt if inj != "off" else None, keep=keep, noise=n,
                             inject_a=cls[t_up, ia].item(), inject_s=cls[t_up, is_].item())
        dv = [v.to(DEV) for v in (x, u, gt, keep, n)]
        if layout == "misaligned":        # a view one element into a larger buffer: the scalar path
            dv[0] = torch.cat([torch.zeros(1, device=DEV), dv[0].reshape(-1)])[1:].view(B, C, H, W)
            assert dv[0].data_ptr() % 16 != 0
        x_in = torch.zeros(B, H, W, 16, device=DEV, dtype=sdt)
        t_in = torch.zeros(B, device=DEV)
        out = d._resample(dv[0], dv[1], a_u, s_u, t_inject=t_up if inj != "off" else None, gt=dv[2], keep=dv[3],
                          inject_noise=dv[4], cumulative=inj != "fresh", stem=(x_in, t_in), t_next=41.0)
        tag = (inj, mch, layout, sdt)
        assert torch.equal(out.cpu(), want), tag
        if inj != "off":
            known = keep.expand_as(x) == 1
            fa, fs = (torch.tensor(cls[t_up, c].item(), dtype=torch.float32) for c in (ia, is_))
            assert torch.equal(out.cpu()[known], (fa * gt + fs * n)[known]), tag
        assert torch.equal(x_in[..., :C], want.permute(0, 2, 3, 1).to(sdt).to(DEV)), tag
        assert not x_in[..., C:].any() and torch.equal(t_in, torch.full((B,), 41.0, device=DEV)), tag
        n_cases += 1
    assert n_cases == 5 * 3 * 3


# ------------------------------------------------------------------------------------------ 2: no jumps = p_sample_loop
@pytest.mark.parametrize("schedule", ["all", "high", "low"])
@pytest.mark.parametrize("cumulative", [True, False])
def test_without_jumps_equals_p_sample_loop(lib, t64_weights, schedule, cumulative):
    import fidm_b200 as F
    cfg, sd = t64_weights
    d = _diffusion(20, learn_sigma=True)
    mk = _inpaint_data(2, 64, seed=6)
    fn = F.InpaintingModelFn(_model(cfg, sd, "bf16"))
    shape = (2, 3, 64, 64)
    kw = dict(model_kwargs=mk, device=DEV, injection_schedule=schedule, use_cumulative_noise=cumulative)
    for name, model in (("fused", fn), ("plain", lambda x, t, **k: fn(x, t, **k))):
        torch.manual_seed(3)
        want = d.p_sample_loop(model, shape, use_inpainting_injection=True, **kw)
        torch.manual_seed(3)
        got = d.repaint_sample_loop(model, shape, jump_length=5, jump_n_sample=1, **kw)
        assert torch.equal(got, want), (name, schedule, cumulative)


# ------------------------------------------------------------------------------------------ 3: jumps, fused = unfused
@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_t64_with_jumps_fused_equals_unfused(lib, t64_weights, precision, monkeypatch):
    import fidm_b200 as F
    cfg, sd = t64_weights
    d = _diffusion(20, learn_sigma=True)
    mk = _inpaint_data(2, 64, seed=7)
    fn = F.InpaintingModelFn(_model(cfg, sd, precision))
    runs = {}
    for fused in ("1", "0"):
        monkeypatch.setenv("FIDM_FUSED_STEP", fused)
        torch.manual_seed(5)
        d.clear_gt_noise_cache()
        runs[fused] = [{k: (v.clone() if torch.is_tensor(v) else v) for k, v in o.items()}
                       for o in d.repaint_sample_loop_progressive(fn, (2, 3, 64, 64), jump_length=4, jump_n_sample=3,
                                                                  model_kwargs=mk, device=DEV)]
    assert len(runs["1"]) == 20 + 2 * 4 * len(range(0, 16, 4))
    for a, b in zip(runs["1"], runs["0"]):
        assert a["t"] == b["t"] and torch.equal(a["sample"], b["sample"]), (precision, a["t"])
        assert torch.equal(a["pred_xstart"], b["pred_xstart"]), (precision, a["t"])
    assert torch.isfinite(runs["1"][-1]["sample"]).all()


# ------------------------------------------------------------------------------------------ 4: against the float64 oracle
def _keyed_noise(kind, t, visit, shape, seed):
    h = int.from_bytes(hashlib.sha256(f"{seed}/{kind}/{t}/{visit}".encode()).digest()[:6], "little")
    # the unpatched randn: PlanRandn replaces torch.randn while the loop runs and calls this from inside
    return _REAL_RANDN(*shape, generator=torch.Generator().manual_seed(h))        # fp32, as the GPU loop consumes it


class PlanRandn:
    """torch.randn / randn_like patched to the loop's documented draw order, each draw keyed (kind, t, visit) as the
    oracle keys them: x_T, the injection at T-1, then per evaluation the step noise, the undo noise (the collapsed
    draw equivalent to the oracle's per-level draws) if a jump follows, and the next evaluation's injection noise
    (with cumulative noise only on a timestep's first visit)."""

    def __init__(self, plan, betas, noise, schedule="all", cumulative=True):
        T = len(betas)
        gated = lambda t: (schedule == "high" and t < T // 2) or (schedule == "low" and t >= T // 2)  # noqa: E731
        visits = {}

        def key(kind, t):
            v = visits.get((kind, t), 0)
            visits[(kind, t)] = v + 1
            return lambda: noise(kind, t, 0 if (kind == "inject" and cumulative) else v)

        def inject(t):
            if t >= 0 and not gated(t):
                first = (("inject", t) not in visits)
                k = key("inject", t)
                if first or not cumulative:
                    self.seq.append(k)

        self.seq = [lambda: noise("xT", 0, 0)]
        inject(T - 1)
        for e in plan:
            self.seq.append(key("step", e.t))
            if e.t_up is not None:
                ks = [key("undo", s) for s in range(e.t, e.t_up + 1)]
                self.seq.append(lambda e=e, ks=ks: _collapse(betas, e, ks))
            inject(e.t_up if e.t_up is not None else e.t - 1)
        self.i = 0

    def _next(self, shape):
        v = self.seq[self.i]()
        self.i += 1
        assert tuple(v.shape) == tuple(shape)
        return v.float().to(DEV)

    def __enter__(self):
        self._r, self._rl = torch.randn, torch.randn_like
        torch.randn = lambda *s, **k: self._next(s[0] if len(s) == 1 and not isinstance(s[0], int) else s)
        torch.randn_like = lambda x, **k: self._next(x.shape)
        return self

    def __exit__(self, *a):
        torch.randn, torch.randn_like = self._r, self._rl


def _collapse(betas, e, ks):
    from oracle import repaint_oracle as O
    return O.collapse_undo_noise(betas, e.t, e.t_up, [k() for k in ks])


@pytest.mark.parametrize("schedule,cumulative", [("all", True), ("low", False)])
def test_public_loop_matches_float64_oracle_with_the_same_noise(lib, schedule, cumulative):
    from fidm_b200 import repaint
    from oracle import repaint_oracle as O
    torch.backends.cuda.matmul.allow_tf32 = False
    d = _diffusion(100, "linear", sigma_small=True)
    B, C, S, jl, jn = 2, 3, 8, 10, 3
    shape = (B, C, S, S)
    am = O.CorrelatedGaussian(d.alphas_cumprod, S, S, channels=C)
    gt = am.sample_prior(B, torch.Generator().manual_seed(1)).float()
    keep = torch.zeros(B, 1, S, S)
    keep[..., : S // 2] = 1
    noise = lambda kind, t, visit: _keyed_noise(kind, t, visit, shape, 17)  # noqa: E731
    model = lambda x, t, **k: am.eps(x, int(t[0])).float()  # noqa: E731
    plan = repaint.evaluation_plan(d.alphas_cumprod, jl, jn)
    with PlanRandn(plan, d.betas, noise, schedule, cumulative) as rng:
        got = d.repaint_sample_loop(model, shape, jump_length=jl, jump_n_sample=jn, clip_denoised=False,
                                    model_kwargs={"gt": gt.to(DEV), "gt_keep_mask": keep.to(DEV)}, device=DEV,
                                    injection_schedule=schedule, use_cumulative_noise=cumulative)
    assert rng.i == len(rng.seq)
    want = O.sample_loop(d.betas, am.eps, noise("xT", 0, 0).double(), jl, jn, gt=gt.double(), keep=keep, noise=noise,
                         var="small", injection_schedule=schedule, cumulative=cumulative)
    err = rel_l2(got.cpu(), want)
    print("RePaint(%d, %d) %s cumulative=%s: rel-L2 vs float64 oracle %.3e" % (jl, jn, schedule, cumulative, err))
    assert err <= 1e-4, err


# ------------------------------------------------------------------------------------------ 5: harmonization on the GPU
@pytest.mark.parametrize("seed", [1, 2])
def test_harmonization_through_the_public_loop(lib, seed):
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
    errs = {}
    for jn in (1, 10):
        torch.manual_seed(seed)
        out = d.repaint_sample_loop(model, (B, 1, 8, 8), jump_length=10, jump_n_sample=jn, clip_denoised=False,
                                    model_kwargs=mk, device=DEV)
        errs[jn] = O.harmonization_errors(out.cpu(), keep, mean, cov)
    plain, rp = errs[1], errs[10]
    print("GPU seed %d: plain injection mean RMS %.4f cov %.4f | RePaint(10, 10) mean RMS %.4f cov %.4f"
          % (seed, *plain, *rp))
    assert plain[1] >= 0.25, plain
    assert rp[1] <= 0.12 and rp[1] <= 0.35 * plain[1], (rp, plain)
    assert rp[0] <= 0.8 * plain[0], (rp, plain)


# ------------------------------------------------------------------------------------------ 6: a 256x256 UNet
def test_ref_ffhq256_with_jumps_known_region_exact(lib):
    """REF-FFHQ256 (synthetic weights, bf16) at 256x256 with jumps: the state every evaluation sees carries exactly
    fl(fl(a*gt) + fl(s*n_t)) in the known region, after K4's and after K7's injections; the fused loop equals it."""
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_state_dict
    cfg = F.CONFIGS["REF_FFHQ256"]
    fn = F.InpaintingModelFn(_model(cfg, synth_state_dict(cfg, seed=3), "bf16"))
    d = _diffusion(20, learn_sigma=True)
    mk = _inpaint_data(2, 256, seed=4)
    gt, keep = mk["gt"], mk["gt_keep_mask"]
    seen = []

    def plain(x, t, **k):
        seen.append((int(t[0]), x.clone()))
        return fn(x, t, **k)

    shape = (2, 3, 256, 256)
    outs = {}
    for name, model in (("plain", plain), ("fused", fn)):
        torch.manual_seed(0)
        outs[name] = d.repaint_sample_loop(model, shape, jump_length=5, jump_n_sample=2, model_kwargs=mk, device=DEV)
        if name == "plain":
            cache = dict(d._gt_noises_cache)
    assert len(seen) == 20 + 5 * len(range(0, 15, 5))
    assert torch.isfinite(outs["plain"]).all() and torch.equal(outs["fused"], outs["plain"])
    cls = d.coefficient_table(0.0)
    known = keep.expand(shape) == 1
    for t, x in seen:
        n = cache[(gt.shape, t, gt.device)]
        wg = cls[t, 0].item() * gt + cls[t, 1].item() * n
        assert torch.equal(x[known], wg[known]), t


# ------------------------------------------------------------------------------------------ 7: sharding
def test_sample_sharded_repaint_equals_direct_call(lib, t64_weights):
    import fidm_b200 as F
    from fidm_b200.parallel import sample_sharded
    cfg, sd = t64_weights
    d = _diffusion(20, learn_sigma=True)
    mk = _inpaint_data(2, 64, seed=9)
    fn = F.InpaintingModelFn(_model(cfg, sd, "bf16"))
    got = sample_sharded(d, fn, mk["gt"], mk["gt_keep_mask"], sampler="repaint", seed=11, jump_length=4,
                         jump_n_sample=2)
    torch.manual_seed(11)
    torch.cuda.manual_seed(11)
    want = d.repaint_sample_loop(fn, (2, 3, 64, 64), jump_length=4, jump_n_sample=2, model_kwargs=mk, device=DEV)
    assert torch.equal(got, want)


# ------------------------------------------------------------------------------------------ 8: errors
def test_invalid_arguments_raise(lib):
    d = _diffusion(100)
    x = torch.zeros(1, 3, 8, 8, device=DEV)
    with pytest.raises(lib.FidmError):                                       # mask channels
        d._resample(x, x, 1.0, 0.0, t_inject=5, gt=x, keep=torch.zeros(1, 2, 8, 8, device=DEV), inject_noise=x)
    with pytest.raises(lib.FidmError):                                       # stem dtype
        d._resample(x, x, 1.0, 0.0, stem=(torch.zeros(1, 8, 8, 16, device=DEV, dtype=torch.uint8),
                                          torch.zeros(1, device=DEV)))
    with pytest.raises(lib.FidmError):                                       # stem narrower than the state
        d._resample(x, x, 1.0, 0.0, stem=(torch.zeros(1, 8, 8, 2, device=DEV), torch.zeros(1, device=DEV)))
    a = lib.ResampleArgs()                                                   # null pointers through the C ABI
    assert lib.lib().fidm_resample_undo(ctypes.byref(a), lib.stream()) == -1
    mk = {"gt": x, "gt_keep_mask": torch.ones(1, 1, 8, 8, device=DEV)}
    fn = lambda x, t, **k: torch.zeros_like(x)  # noqa: E731
    for kw in (dict(jump_length=100), dict(jump_n_sample=0), dict(use_inpainting_injection=False)):
        with pytest.raises(ValueError):
            d.repaint_sample_loop(fn, (1, 3, 8, 8), model_kwargs=mk, device=DEV, **kw)
