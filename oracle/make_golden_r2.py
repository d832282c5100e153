"""Round-2 golden fixtures, made by running the UNMODIFIED reference (imported read-only from
/root/reference/code) in the build container; the first-round fixtures stay as oracle/make_golden.py wrote them.

    python oracle/make_golden_r2.py [small|ref256|adm256|all]

What is pinned here (VERDICT r1 "next round" item 1):
  small   sampler_steps_modes.pt   single steps for the K4 branches the first fixtures do not cover: START_X and PREVIOUS_X
                                   mean types, LEARNED variance (gaussian_diffusion.py:213-298), p_mean_variance outputs
          t64_loop_variants.pt     T64 loops through the reference's class path with injection_schedule high / low,
                                   use_cumulative_noise=False, predict_xstart=True, rescale_timesteps=True, eta > 0,
                                   denoised_fn / cond_fn, and both sample_with_advanced_inpainting entry points
                                   (gaussian_diffusion.py:640-700, train_inpainting.py:265-310)
  ref256  ref_ffhq256_ddim100.pt   the reference's literal model (train_inpainting.py:208-224): DDIM-100 cosine, B=1,
                                   injection on: final image + pred_xstart / sample at loop index 50
          ref_ffhq256_ddpm25.pt    p_sample_loop over a 25-step linear schedule (full loop)
  adm256  adm256_eval_b8.pt        one evaluation at batch 8 with per-image timesteps (stride-2 pixel subsample of eps)
          adm256_lora_quad.pt      LoRA-merged attention weights, quadratic T=100: first 3 DDIM steps (progressive)
          adm256_ddpm25.pt         p_sample_loop over a 25-step linear schedule (full loop)
          adm256_ddim100.pt        DDIM-100 cosine, B=1, injection on: final + index 50

Large outputs are stored as a seeded element subset (oracle/golden_subset.py) so that every file stays under 1 MB.
While generating, the oracle restatement is checked against the reference wherever it has the mode
(the script aborts on disagreement).  Inputs are regenerated from integer seeds by the tests.
"""
import ast
import os
import sys
import textwrap
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, "/root/reference/code")

import numpy as np  # noqa: E402
import torch  # noqa: E402

import fidm_b200  # noqa: E402,F401
from fidm_b200.arch import CONFIGS  # noqa: E402
from fidm_b200.utils.synth import merge_lora, synth_batch, synth_state_dict  # noqa: E402
from oracle import diffusion_oracle as dor  # noqa: E402
from oracle.golden_subset import shrink  # noqa: E402
from oracle import unet_oracle as uor  # noqa: E402

import gaussian_diffusion as ref_gd  # noqa: E402  (reference)
from losses import LossType, ModelMeanType, ModelVarType  # noqa: E402  (reference)
from unet import DiffusionInpaintingModel, UNetModel  # noqa: E402  (reference)
from utils.schedules import create_gaussian_diffusion, get_named_beta_schedule  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden")
torch.set_num_threads(int(os.environ.get("GOLDEN_THREADS", os.cpu_count())))
_REAL_RANDN = torch.randn


def seeded_noise(kind, t, shape, seed):
    g = torch.Generator().manual_seed(seed * 100003 + {"xT": 0, "inject": 1, "step": 2}[kind] * 50021 + int(t))
    return _REAL_RANDN(*shape, generator=g)


def draw_order(T, inject=True, schedule="all", first=True):
    """The class path's RNG draw order (gaussian_diffusion.py:96-101,146,381,478,428,521) with the
    high / low gating of :132-135."""
    seq = [("xT", 0)] if first else []
    for t in range(T - 1, -1, -1):
        gated = (schedule == "high" and t < T // 2) or (schedule == "low" and t >= T // 2)
        if inject and not gated:
            seq.append(("inject", t))
        seq.append(("step", t))
    return seq


class SeqRandn:
    def __init__(self, seq, seed, strict=True):
        self.seq, self.i, self.seed, self.strict = list(seq), 0, seed, strict

    def _next(self, shape):
        kind, t = self.seq[self.i]
        self.i += 1
        return seeded_noise(kind, t, tuple(shape), self.seed)

    def __enter__(self):
        self._r, self._rl = torch.randn, torch.randn_like
        torch.randn = lambda *s, **k: self._next(s[0] if len(s) == 1 and not isinstance(s[0], int) else s)
        torch.randn_like = lambda x, **k: self._next(x.shape)
        return self

    def __exit__(self, et, *a):
        torch.randn, torch.randn_like = self._r, self._rl
        if et is None and self.strict:
            assert self.i == len(self.seq), (self.i, len(self.seq))


def build_ref_model(name, seed, lora=False):
    cfg = CONFIGS[name]
    model = DiffusionInpaintingModel(UNetModel(**dict(cfg, in_channels=3)), in_channels=9).eval()
    sd = synth_state_dict(cfg, seed=seed)
    if lora:
        sd = merge_lora(sd, rank=8, alpha=64.0, seed=seed)
    model.load_state_dict(sd, strict=True)
    return model, sd, cfg


def psnr(a, b):
    return 10 * np.log10(4.0 / max(((a.double() - b.double()) ** 2).mean().item(), 1e-30))


# ----------------------------------------------------------------------------- small: K4 branches
def golden_step_modes():
    B, C, H, W = 2, 3, 8, 8
    cases, seed = [], 501
    combos = [(ModelMeanType.START_X, ModelVarType.LEARNED_RANGE), (ModelMeanType.START_X, ModelVarType.FIXED_SMALL),
              (ModelMeanType.PREVIOUS_X, ModelVarType.LEARNED), (ModelMeanType.PREVIOUS_X, ModelVarType.FIXED_LARGE),
              (ModelMeanType.EPSILON, ModelVarType.LEARNED), (ModelMeanType.EPSILON, ModelVarType.LEARNED_RANGE)]
    for sched, T in (("cosine", 100), ("linear", 1000)):
        betas = get_named_beta_schedule(sched, T)
        for mean_type, var_type in combos:
            d = ref_gd.GaussianDiffusion(betas=betas, model_mean_type=mean_type, model_var_type=var_type,
                                         loss_type=LossType.MSE)
            two = var_type in (ModelVarType.LEARNED, ModelVarType.LEARNED_RANGE)
            for t in (0, 1, T // 2, T - 1):
                for mode, eta, clip in (("ddim", 0.0, True), ("ddim", 0.5, False), ("ddpm", 0.0, True)):
                    seed += 1
                    g = torch.Generator().manual_seed(seed)
                    x = torch.randn(B, C, H, W, generator=g) * (1.0 + t / T)
                    gt = torch.rand(B, C, H, W, generator=g) * 2 - 1
                    keep = (torch.rand(B, 1, H, W, generator=g) > 0.4).float()
                    mo = torch.randn(B, 2 * C if two else C, H, W, generator=g)
                    if var_type == ModelVarType.LEARNED:
                        mo[:, C:] = mo[:, C:] * 0.5 - 3.0           # a log-variance
                    n_inj = torch.randn(B, C, H, W, generator=g)
                    z = torch.randn(B, C, H, W, generator=g)
                    tt = torch.full((B,), t, dtype=torch.int64)
                    d.clear_gt_noise_cache()
                    draws = iter([n_inj, z])
                    rl = torch.randn_like
                    torch.randn_like = lambda a, **k: next(draws)
                    try:
                        fn = d.ddim_sample if mode == "ddim" else d.p_sample
                        kw = dict(eta=eta) if mode == "ddim" else {}
                        got = fn(lambda xx, ts, **k: mo, x, tt, clip_denoised=clip,
                                 model_kwargs={"gt": gt, "gt_keep_mask": keep},
                                 use_inpainting_injection=True, **kw)
                        d.clear_gt_noise_cache()
                        draws = iter([n_inj])
                        x_inj = d.apply_inpainting_injection(x, tt, gt, keep)
                    finally:
                        torch.randn_like = rl
                    pmv = d.p_mean_variance(lambda xx, ts, **k: mo, x_inj, tt, clip_denoised=clip)
                    cases.append(dict(sched=sched, T=T, mean_type=mean_type.name, var_type=var_type.name, t=t, mode=mode,
                                      eta=eta, clip=clip, seed=seed, sample=got["sample"].clone(),
                                      pred_xstart=got["pred_xstart"].clone(), mean=pmv["mean"].clone(),
                                      log_variance=pmv["log_variance"].clone(), variance=pmv["variance"].clone()))
    cases = [shrink(c, ["sample", "pred_xstart", "mean", "log_variance", "variance"], 192) for c in cases]
    torch.save(cases, os.path.join(OUT, "sampler_steps_modes.pt"))
    print("sampler step mode cases:", len(cases))


# ----------------------------------------------------------------------------- small: T64 loop variants
def _train_inpainting_helper():
    """train_inpainting.sample_with_advanced_inpainting, extracted from the source (the module imports torchvision
    at the top; only this function is needed)."""
    src = open("/root/reference/code/train_inpainting.py").read()
    tree = ast.parse(src)
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "sample_with_advanced_inpainting"][0]
    ns = {"torch": torch}
    exec(textwrap.dedent(ast.get_source_segment(src, fn)), ns)
    return ns["sample_with_advanced_inpainting"]


class _Swallow(torch.nn.Module):
    """The kwargs-swallowing wrapper every working call site of the reference uses (SURVEY fact 5)."""

    def __init__(self, model):
        super().__init__()
        self.model = model

    def forward(self, x, t, gt=None, gt_keep_mask=None, masked_image=None, mask=None, **kw):
        if masked_image is None:
            masked_image, mask = gt * gt_keep_mask, 1 - gt_keep_mask
        return self.model(x, t, masked_image=masked_image, mask=mask)


def golden_t64_loop_variants():
    model, sd, cfg = build_ref_model("T64", seed=1)
    data = synth_batch(2, 64, seed=14)
    gt, keep = data["gt"], data["gt_keep_mask"]
    shape = (2, 3, 64, 64)
    wrap = _Swallow(model).eval()
    out = {}
    T = 20

    def run(tag, seed, *, ddim=True, diff_kw=None, loop_kw=None, schedule="all", oracle_kw=None, fn=None):
        d = create_gaussian_diffusion(**dict(dict(steps=T, learn_sigma=True, noise_schedule="cosine"), **(diff_kw or {})))
        lk = dict(model_kwargs={"gt": gt, "gt_keep_mask": keep}, device="cpu", use_inpainting_injection=True,
                  injection_schedule=schedule)
        lk.update(loop_kw or {})
        trace = []
        with SeqRandn(draw_order(T, inject=lk["use_inpainting_injection"], schedule=schedule), seed), torch.no_grad():
            gen = (d.ddim_sample_loop_progressive if ddim else d.p_sample_loop_progressive)(fn or wrap, shape, **lk)
            for o in gen:
                trace.append(o)
        fin = trace[-1]["sample"]
        if oracle_kw is not None:
            tab = dor.Tables(d.betas)
            with torch.no_grad():
                mine = dor.sample_loop(tab, lambda xx, ts, **k: uor.inpaint_forward(sd, cfg, xx, ts, gt * keep, 1 - keep),
                                       shape, ddim=ddim, x_T=seeded_noise("xT", 0, shape, seed), gt=gt, keep=keep,
                                       noise_fn=lambda kind, t: seeded_noise(kind, t, shape, seed), schedule=schedule,
                                       **oracle_kw)
            p = psnr(mine, fin)
            print(f"  {tag}: oracle vs reference {p:.1f} dB")
            assert p > 80, (tag, p)
        out[tag] = {"T": T, "seed_noise": seed, "final": fin.clone(), "pred_xstart_mid": trace[T // 2]["pred_xstart"].clone()}
        print("t64 variant", tag, "done")

    run("ddim_high", 41, schedule="high", oracle_kw={})
    run("ddim_low", 42, schedule="low", oracle_kw={})
    run("ddpm_high", 43, ddim=False, schedule="high", oracle_kw={})
    run("ddim_fresh_noise", 44, loop_kw={"use_cumulative_noise": False}, oracle_kw={"cumulative": False})
    run("ddpm_fresh_noise", 45, ddim=False, loop_kw={"use_cumulative_noise": False}, oracle_kw={"cumulative": False})
    run("ddim_eta", 46, loop_kw={"eta": 0.8}, oracle_kw={"eta": 0.8})
    run("ddim_noclip", 47, loop_kw={"clip_denoised": False}, oracle_kw={"clip": False})
    run("ddim_predict_xstart", 48, diff_kw={"predict_xstart": True})
    run("ddpm_predict_xstart", 49, ddim=False, diff_kw={"predict_xstart": True})
    run("ddim_rescale_t", 50, diff_kw={"rescale_timesteps": True})
    run("ddim_fixed_small", 51, diff_kw={"learn_sigma": False, "sigma_small": True},
        fn=lambda x, t, **k: wrap(x, t, **k)[:, :3], oracle_kw=None)
    run("ddpm_fixed_large", 52, ddim=False, diff_kw={"learn_sigma": False},
        fn=lambda x, t, **k: wrap(x, t, **k)[:, :3], oracle_kw=None)
    run("ddim_denoised_fn", 53, loop_kw={"denoised_fn": lambda v: v * 0.9})
    run("ddpm_cond_fn", 54, ddim=False, loop_kw={"cond_fn": lambda x, t, **k: -0.5 * x})
    run("ddim_cond_fn", 55, loop_kw={"cond_fn": lambda x, t, **k: -0.5 * x})
    run("ddim_no_injection", 56, loop_kw={"use_inpainting_injection": False})

    # GaussianDiffusion.sample_with_advanced_inpainting (:640-700), both samplers
    for tag, use_ddim, seed in (("method_ddim", True, 61), ("method_ddpm", False, 62)):
        d = create_gaussian_diffusion(steps=T, learn_sigma=True, noise_schedule="cosine")
        with SeqRandn(draw_order(T), seed), torch.no_grad():
            fin = d.sample_with_advanced_inpainting(wrap, shape, gt=gt, gt_keep_mask=keep, use_ddim=use_ddim,
                                                    progress=False, device="cpu")
        out[tag] = {"T": T, "seed_noise": seed, "final": fin.clone()}
    # train_inpainting.sample_with_advanced_inpainting (:265-310): gt re-derived from the masked image
    helper = _train_inpainting_helper()
    d = create_gaussian_diffusion(steps=T, learn_sigma=True, noise_schedule="cosine")
    with SeqRandn(draw_order(T, schedule="low"), 63), torch.no_grad():
        fin = helper(wrap, d, data["masked_image"], data["mask"], "cpu", use_ddim=True, injection_schedule="low")
    out["helper_ddim_low"] = {"T": T, "seed_noise": 63, "final": fin.clone()}
    out = {k: shrink(v, [a for a in ("final", "pred_xstart_mid") if a in v], 4096) for k, v in out.items()}
    out["_meta"] = {"seed_weights": 1, "seed_data": 14, "batch": 2}
    torch.save(out, os.path.join(OUT, "t64_loop_variants.pt"))


# ----------------------------------------------------------------------------- 256x256
def loop_256(name, T, sched, *, ddim, seed_w, seed_d, seed_n, fname, check_oracle_steps=0):
    model, sd, cfg = build_ref_model(name, seed=seed_w)
    S = cfg["image_size"]
    data = synth_batch(1, S, seed=seed_d)
    gt, keep = data["gt"], data["gt_keep_mask"]
    shape = (1, 3, S, S)
    d = create_gaussian_diffusion(steps=T, learn_sigma=True, noise_schedule=sched)
    wrap = _Swallow(model).eval()
    trace = {}
    t0 = time.time()
    with SeqRandn(draw_order(T), seed_n), torch.no_grad():
        gen = (d.ddim_sample_loop_progressive if ddim else d.p_sample_loop_progressive)(
            wrap, shape, model_kwargs={"gt": gt, "gt_keep_mask": keep}, device="cpu", use_inpainting_injection=True)
        for i, o in enumerate(gen):
            if i in (T // 2, T - 1):
                trace[i] = {k: v.clone() for k, v in o.items()}
            if i % 10 == 0:
                print(f"  {name} {fname}: step {i}/{T}  {time.time() - t0:.0f}s", flush=True)
    torch.save(shrink({"config": name, "T": T, "sched": sched, "ddim": ddim, "seed_weights": seed_w, "seed_data": seed_d,
                       "seed_noise": seed_n, "final": trace[T - 1]["sample"], "mid_index": T // 2,
                       "pred_xstart_mid": trace[T // 2]["pred_xstart"], "sample_mid": trace[T // 2]["sample"],
                       "seconds_reference_cpu": time.time() - t0, "cpu_threads": torch.get_num_threads()},
                      ["final", "pred_xstart_mid", "sample_mid"], 24576),
               os.path.join(OUT, fname))
    print(name, fname, "written,", f"{time.time() - t0:.0f}s")


def golden_adm256_eval_b8():
    model, sd, cfg = build_ref_model("ADM256", seed=7)
    B = 8
    data = synth_batch(B, 256, seed=2)
    g = torch.Generator().manual_seed(3)
    x = torch.randn(B, 3, 256, 256, generator=g)
    t = torch.tensor([61, 0, 99, 17, 42, 5, 88, 73], dtype=torch.int64)
    outs = []
    with torch.no_grad():
        for b in range(B):                       # per-image evaluations are independent (no cross-sample op on the path)
            outs.append(model(x[b:b + 1], t[b:b + 1], masked_image=data["masked_image"][b:b + 1], mask=data["mask"][b:b + 1]))
            print("  adm256 eval image", b, flush=True)
        out = torch.cat(outs)
        mine = uor.inpaint_forward(sd, cfg, x[:1], t[:1], data["masked_image"][:1], data["mask"][:1])
    rel = ((out[:1] - mine).norm() / out[:1].norm()).item()
    print("ADM256 eval: oracle rel-L2 vs reference", rel)
    assert rel < 2e-6, rel
    torch.save(shrink({"seed_weights": 7, "seed_data": 2, "seed_x": 3, "t": t, "stride": 2,
                       "out_sub": out[:, :, ::2, ::2].clone(), "norm_per_image": out.flatten(1).norm(dim=1)},
                      ["out_sub"], 12288, per_image=True), os.path.join(OUT, "adm256_eval_b8.pt"))


def golden_adm256_lora_quad():
    model, sd, cfg = build_ref_model("ADM256", seed=13, lora=True)
    data = synth_batch(1, 256, seed=15)
    gt, keep = data["gt"], data["gt_keep_mask"]
    shape, T, seed = (1, 3, 256, 256), 100, 17
    d = create_gaussian_diffusion(steps=T, learn_sigma=True, noise_schedule="quadratic")
    wrap = _Swallow(model).eval()
    steps = []
    with SeqRandn(draw_order(T), seed, strict=False), torch.no_grad():
        for i, o in enumerate(d.ddim_sample_loop_progressive(wrap, shape, model_kwargs={"gt": gt, "gt_keep_mask": keep},
                                                             device="cpu", use_inpainting_injection=True)):
            steps.append({k: v.clone() for k, v in o.items()})
            if i == 2:
                break
    torch.save(shrink({"seed_weights": 13, "lora": dict(rank=8, alpha=64.0, seed=13), "seed_data": 15, "seed_noise": seed,
                       "T": T, "sched": "quadratic", "n_steps": 3, "sample": steps[-1]["sample"],
                       "pred_xstart": steps[-1]["pred_xstart"], "pred_xstart_first": steps[0]["pred_xstart"]},
                      ["sample", "pred_xstart", "pred_xstart_first"], 24576), os.path.join(OUT, "adm256_lora_quad.pt"))
    print("adm256 lora quadratic written")


if __name__ == "__main__":
    what = sys.argv[1] if len(sys.argv) > 1 else "all"
    os.makedirs(OUT, exist_ok=True)
    if what in ("small", "all"):
        golden_step_modes()
        golden_t64_loop_variants()
    if what in ("ref256", "all"):
        loop_256("REF_FFHQ256", 100, "cosine", ddim=True, seed_w=11, seed_d=12, seed_n=5, fname="ref_ffhq256_ddim100.pt")
        loop_256("REF_FFHQ256", 25, "linear", ddim=False, seed_w=11, seed_d=12, seed_n=6, fname="ref_ffhq256_ddpm25.pt")
    if what in ("adm256", "all"):
        golden_adm256_eval_b8()
        golden_adm256_lora_quad()
        loop_256("ADM256", 25, "linear", ddim=False, seed_w=11, seed_d=12, seed_n=6, fname="adm256_ddpm25.pt")
        loop_256("ADM256", 100, "cosine", ddim=True, seed_w=11, seed_d=12, seed_n=5, fname="adm256_ddim100.pt")
    print("done:", what)
