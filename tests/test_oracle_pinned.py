"""CPU: the oracle restatement (oracle/*.py) against the golden vectors produced by the UNMODIFIED
reference (oracle/make_golden.py).  This is what pins the oracle; the reference has no tests."""
import json
import os

import numpy as np
import torch

import fidm_b200  # noqa: F401
from fidm_b200.arch import CONFIGS, param_shapes, unet_topology
from fidm_b200.utils.schedules import get_named_beta_schedule
from fidm_b200.utils.synth import synth_batch, synth_state_dict
from oracle import diffusion_oracle as dor
from oracle import unet_oracle as uor
from oracle.golden_subset import take

from helpers import psnr, seeded_noise


def test_state_dict_layout_matches_reference(golden_dir):
    ref = json.load(open(os.path.join(golden_dir, "state_dict_layout.json")))
    for name, cfg in CONFIGS.items():
        mine = [["base_model." + k, list(s)] for k, s in param_shapes(unet_topology(**cfg))]
        assert mine == ref[name], name


def test_schedule_tables_match_reference(golden_dir):
    ref = json.load(open(os.path.join(golden_dir, "schedules.json")))
    for key, vals in ref.items():
        sched, T = key.rsplit("_", 1)
        T = int(T)
        with np.errstate(divide="ignore"):
            tab = dor.Tables(get_named_beta_schedule(sched, T))
        idx = [0, 1, T // 2, T - 1]
        for k, v in vals.items():
            got = [float(getattr(tab, k)[i]) for i in idx]
            assert got == v, (key, k)          # float64, exact


def test_oracle_sampler_steps_bit_exact(golden_dir):
    cases = torch.load(os.path.join(golden_dir, "sampler_steps.pt"))
    assert len(cases) == 108
    for c in cases:
        tab = dor.Tables(get_named_beta_schedule(c["sched"], c["T"]))
        g = torch.Generator().manual_seed(c["seed"])
        B, C, H, W = c["sample"].shape
        t, T = c["t"], c["T"]
        x = torch.randn(B, C, H, W, generator=g) * (1.0 + t / T)
        gt = torch.rand(B, C, H, W, generator=g) * 2 - 1
        keep = (torch.rand(B, 1, H, W, generator=g) > 0.4).float()
        mo = torch.randn(B, 2 * C if c["var_type"] == "learned_range" else C, H, W, generator=g)
        n_inj = torch.randn(B, C, H, W, generator=g)
        z = torch.randn(B, C, H, W, generator=g)
        xi = dor.inject(tab, x, t, gt, keep, n_inj, c["cumulative"])
        assert torch.equal(xi, c["x_inj"])
        if c["mode"] == "ddim":
            s, x0 = dor.ddim_update(tab, mo, xi, t, z, c["eta"], c["var_type"])
        else:
            s, x0 = dor.ddpm_update(tab, mo, xi, t, z, c["var_type"])
        assert torch.equal(s, c["sample"]) and torch.equal(x0, c["pred_xstart"])
        # known-region pixels are exactly the noised ground truth
        m = keep.expand_as(xi) == 1
        wg = dor.inject(tab, torch.zeros_like(x), t, gt, torch.ones_like(keep), n_inj, c["cumulative"])
        assert torch.equal(xi[m], wg[m])


def test_oracle_unet_forward_matches_reference(golden_dir):
    gold = torch.load(os.path.join(golden_dir, "t64_forward.pt"))
    cfg = CONFIGS["T64"]
    sd = synth_state_dict(cfg, seed=gold["seed_weights"])
    data = synth_batch(2, 64, seed=gold["seed_data"])
    with torch.no_grad():
        out = uor.inpaint_forward(sd, cfg, gold["x"], gold["t"], data["masked_image"], data["mask"])
    assert torch.allclose(out, gold["out"], rtol=1e-4, atol=1e-5)
    assert ((out - gold["out"]).norm() / gold["out"].norm()).item() < 1e-5


def test_oracle_unet_variants_match_reference(golden_dir):
    gold = torch.load(os.path.join(golden_dir, "t32_variants.pt"))
    for tag, g in gold.items():
        sd = synth_state_dict(g["cfg"], seed=g["seed_weights"])
        data = synth_batch(2, 32, seed=g["seed_data"])
        with torch.no_grad():
            out = uor.inpaint_forward(sd, g["cfg"], g["x"], g["t"], data["masked_image"], data["mask"])
        assert ((out - g["out"]).norm() / g["out"].norm()).item() < 1e-5, tag


def test_oracle_ddim50_loop_matches_reference(golden_dir):
    """BASELINE config #1: T64, DDIM-50 cosine, B=1, injection on -- the full loop on the CPU."""
    gold = torch.load(os.path.join(golden_dir, "t64_ddim50.pt"))
    cfg = CONFIGS["T64"]
    sd = synth_state_dict(cfg, seed=gold["seed_weights"])
    data = synth_batch(1, 64, seed=gold["seed_data"])
    gt, keep = data["gt"], data["gt_keep_mask"]
    tab = dor.Tables(get_named_beta_schedule("cosine", gold["T"]))
    seed, shape = gold["seed_noise"], (1, 3, 64, 64)
    trace = []
    with torch.no_grad():
        out = dor.sample_loop(tab, lambda x, t, **k: uor.inpaint_forward(sd, cfg, x, t, gt * keep, 1 - keep),
                              shape, ddim=True, x_T=seeded_noise("xT", 0, shape, seed), gt=gt, keep=keep,
                              noise_fn=lambda kind, t: seeded_noise(kind, t, shape, seed), trace=trace)
    assert psnr(out, gold["final"]) > 60
    assert psnr(trace[24]["pred_xstart"], gold["pred_xstart_t25"]) > 60


def test_oracle_script_loops_match_reference(golden_dir):
    """The evaluation scripts' strided-DDIM / DDPM loops with post-step injection (SURVEY 8-f row 1)."""
    from oracle import script_oracle as sor
    gold = torch.load(os.path.join(golden_dir, "t64_script_loops.pt"))
    cfg = CONFIGS["T64"]
    sd = synth_state_dict(cfg, seed=1)
    data = synth_batch(1, 64, seed=4)
    gt, masks = data["gt"], data["mask"]
    shape = (1, 3, 64, 64)

    def fn(x, t, gt=None, gt_keep_mask=None):
        return uor.inpaint_forward(sd, cfg, x, t, gt * gt_keep_mask, 1 - gt_keep_mask)

    g = gold["cos100_ddim10_eta"]
    assert list(sor.ddim_timestep_sequence(1000, 100))[:3] == [999, 990, 980] and len(sor.ddim_timestep_sequence(1000, 100)) == 101
    tab = dor.Tables(get_named_beta_schedule(g["sched"], g["steps"]))
    with torch.no_grad():
        out = sor.script_ddim_loop(tab, fn, shape, gt, masks, g["n_ddim"], eta=g["eta"],
                                   x_T=seeded_noise("xT", 0, shape, g["seed_noise"]),
                                   noise_fn=lambda kind, t: seeded_noise(kind, t, shape, g["seed_noise"]))
    assert psnr(out, g["final"]) > 60
    g = gold["cos30_ddpm"]
    tab = dor.Tables(get_named_beta_schedule(g["sched"], g["steps"]))
    with torch.no_grad():
        out = sor.script_ddpm_loop(tab, fn, shape, gt, masks, x_T=seeded_noise("xT", 0, shape, g["seed_noise"]),
                                   noise_fn=lambda kind, t: seeded_noise(kind, t, shape, g["seed_noise"]))
    assert psnr(out, g["final"]) > 60


def test_oracle_mean_and_variance_types_bit_exact(golden_dir):
    """START_X / PREVIOUS_X mean types and LEARNED variance (gaussian_diffusion.py:241-286) against single steps of
    the unmodified reference (oracle/make_golden_r2.py)."""
    cases = torch.load(os.path.join(golden_dir, "sampler_steps_modes.pt"))
    assert len(cases) == 144
    for c in cases:
        tab = dor.Tables(get_named_beta_schedule(c["sched"], c["T"]))
        two = c["var_type"] in ("LEARNED", "LEARNED_RANGE")
        g = torch.Generator().manual_seed(c["seed"])
        B, C, H, W = c["shape"]
        t, T = c["t"], c["T"]
        x = torch.randn(B, C, H, W, generator=g) * (1.0 + t / T)
        gt = torch.rand(B, C, H, W, generator=g) * 2 - 1
        keep = (torch.rand(B, 1, H, W, generator=g) > 0.4).float()
        mo = torch.randn(B, 2 * C if two else C, H, W, generator=g)
        if c["var_type"] == "LEARNED":
            mo[:, C:] = mo[:, C:] * 0.5 - 3.0
        n_inj = torch.randn(B, C, H, W, generator=g)
        z = torch.randn(B, C, H, W, generator=g)
        xi = dor.inject(tab, x, t, gt, keep, n_inj)
        vt, mt = c["var_type"].lower(), c["mean_type"].lower()
        mean, logvar, x0 = dor.mean_variance(tab, mo, xi, t, vt, c["clip"], mt)
        idx = c["sub_idx"]
        assert torch.equal(take(mean, idx), c["mean"]) and torch.equal(take(logvar, idx), c["log_variance"]), (mt, vt, t)
        if c["mode"] == "ddim":
            s, x0 = dor.ddim_update(tab, mo, xi, t, z, c["eta"], vt, c["clip"], mt)
        else:
            s, x0 = dor.ddpm_update(tab, mo, xi, t, z, vt, c["clip"], mt)
        assert torch.equal(take(s, idx), c["sample"]) and torch.equal(take(x0, idx), c["pred_xstart"]), (mt, vt, t, c["mode"])


def test_oracle_loop_switches_match_reference(golden_dir):
    """injection_schedule gating, fresh (non-cumulative) injection noise, predict_xstart and rescale_timesteps through
    the oracle's loop against T64 loops of the unmodified reference (a subset: each is 20 UNet evaluations at batch 2)."""
    gold = torch.load(os.path.join(golden_dir, "t64_loop_variants.pt"))
    meta = gold["_meta"]
    cfg = CONFIGS["T64"]
    sd = synth_state_dict(cfg, seed=meta["seed_weights"])
    data = synth_batch(meta["batch"], 64, seed=meta["seed_data"])
    gt, keep = data["gt"], data["gt_keep_mask"]
    shape = (meta["batch"], 3, 64, 64)
    torch.set_num_threads(os.cpu_count())
    for tag, kw in (("ddim_low", dict(ddim=True, schedule="low")),
                    ("ddpm_fresh_noise", dict(ddim=False, cumulative=False)),
                    ("ddim_predict_xstart", dict(ddim=True, mean_type="start_x")),
                    ("ddim_rescale_t", dict(ddim=True, rescale_timesteps=True))):
        g = gold[tag]
        seed = g["seed_noise"]
        tab = dor.Tables(get_named_beta_schedule("cosine", g["T"]))
        with torch.no_grad():
            out = dor.sample_loop(tab, lambda x, t, **k: uor.inpaint_forward(sd, cfg, x, t, gt * keep, 1 - keep), shape,
                                  x_T=seeded_noise("xT", 0, shape, seed), gt=gt, keep=keep,
                                  noise_fn=lambda kind, t: seeded_noise(kind, t, shape, seed), **kw)
        out = take(out, g["sub_idx"])
        assert psnr(out, g["final"]) > 80, (tag, psnr(out, g["final"]))
