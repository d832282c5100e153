"""CPU: host-side logic of the product (no kernel launches): ABI surface, tables, factories."""
import ctypes
import os
import re

import numpy as np
import pytest
import torch

import fidm_b200 as F
from fidm_b200 import _lib
from fidm_b200.utils.synth import merge_lora, synth_batch, synth_state_dict
from oracle import diffusion_oracle as dor

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "fidm_b200.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(fidm_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    syms = _header_symbols()
    assert len(syms) >= 14
    assert os.path.exists(_lib.LIB_PATH), "run __graft_entry__.build() first"
    handle = ctypes.CDLL(_lib.LIB_PATH)
    for s in syms:
        assert hasattr(handle, s), s
    assert set(syms) == set(_lib.SYMBOLS), set(syms) ^ set(_lib.SYMBOLS)
    assert _lib.lib().fidm_abi_version() == 3


def test_ctypes_structs_match_header_field_order():
    text = open(os.path.join(ROOT, "include", "fidm_b200.h")).read()
    for cname, struct in (("fidm_step_args", _lib.StepArgs), ("fidm_multistep_args", _lib.MultistepArgs),
                          ("fidm_resample_args", _lib.ResampleArgs), ("fidm_gn_args", _lib.GnArgs),
                          ("fidm_conv_args", _lib.ConvArgs), ("fidm_attn_args", _lib.AttnArgs),
                          ("fidm_pack_args", _lib.PackArgs)):
        body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (cname, cname), text, flags=re.S).group(1)
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        names = []
        for decl in body.split(";"):
            decl = decl.strip()
            if not decl:
                continue
            decl = re.sub(r"^(const\s+)?(int32_t|int64_t|float|double|void)\s*\**", "", decl)
            for part in decl.split(","):
                names.append(re.sub(r"\[.*\]", "", part.replace("*", "").strip()))
        assert names == [f[0] for f in struct._fields_], cname
    cols = int(re.search(r"#define FIDM_MS_COLS (\d+)", text).group(1))
    assert cols == _lib.MS_COLS
    for name in ("X0_C1", "X0_C2", "A", "B0", "B1", "INJ_A", "INJ_S"):
        assert int(re.search(r"FIDM_MS_%s = (\d+)" % name, text).group(1)) == getattr(_lib, "MS_" + name)
    assert "fidm_resample_undo" in _lib.SYMBOLS


def test_no_cpu_fallback():
    model = F.DiffusionInpaintingModel(F.UNetModel(**dict(F.CONFIGS["T64"], in_channels=3)))
    z = torch.zeros(1, 3, 64, 64)
    with pytest.raises(_lib.FidmError):
        model(z, torch.zeros(1), masked_image=z, mask=torch.zeros(1, 1, 64, 64))
    d = F.create_gaussian_diffusion(steps=100, learn_sigma=True)
    with pytest.raises(_lib.FidmError):
        d.ddim_sample_loop(lambda x, t, **k: torch.zeros(1, 6, 8, 8), (1, 3, 8, 8), device="cpu")


def test_module_state_dict_is_reference_layout(golden_dir):
    import json
    ref = json.load(open(os.path.join(golden_dir, "state_dict_layout.json")))
    for name in ("T64", "REF_FFHQ256"):
        cfg = dict(F.CONFIGS[name], in_channels=3)
        with torch.device("meta"):
            m = F.DiffusionInpaintingModel(F.UNetModel(**cfg))
        got = [[k, list(v.shape)] for k, v in m.state_dict().items()]
        assert got == ref[name], name
    sd = synth_state_dict(F.CONFIGS["T64"], seed=0)
    m = F.DiffusionInpaintingModel(F.UNetModel(**dict(F.CONFIGS["T64"], in_channels=3)))
    res = m.load_state_dict(sd, strict=True)
    assert not res.missing_keys and not res.unexpected_keys
    lora = merge_lora(sd, rank=8)
    assert list(lora) == list(sd) and all(lora[k].shape == sd[k].shape for k in sd)
    changed = [k for k in sd if not torch.equal(sd[k], lora[k])]
    assert changed and all(k.endswith(("qkv.weight", "proj_out.weight")) for k in changed)


def test_zero_init_matches_reference_convention():
    m = F.UNetModel(**dict(F.CONFIGS["T64"], in_channels=3))
    sd = m.state_dict()
    zero = [k for k, v in sd.items() if v.numel() and not v.any()]
    assert any(k.endswith("out_layers.3.weight") for k in zero)
    assert any(k.endswith("proj_out.weight") for k in zero) and "out.2.weight" in zero
    w = F.DiffusionInpaintingModel(m).state_dict()["base_model.input_blocks.0.0.weight"]
    assert w.shape[1] == 9 and not w[:, 3:].any() and w[:, :3].any()


@pytest.mark.parametrize("sched,T", [("cosine", 100), ("linear", 1000), ("quadratic", 100), ("cosine", 50)])
def test_coefficient_table_is_reference_arithmetic(sched, T):
    d = F.create_gaussian_diffusion(steps=T, learn_sigma=True, noise_schedule=sched)
    tab = dor.Tables(F.get_named_beta_schedule(sched, T))
    for eta in (0.0, 0.7):
        c = d.coefficient_table(eta)
        assert c.shape == (T, _lib.COEF_COLS) and c.dtype == torch.float32
        for t in (0, 1, T // 2, T - 1):
            assert c[t, 0] == dor._c(tab.sqrt_alphas_cumprod, t)
            assert c[t, 5] == dor._c(tab.sqrt_recipm1_alphas_cumprod, t)
            ab, abp = dor._c(tab.alphas_cumprod, t), dor._c(tab.alphas_cumprod_prev, t)
            sigma = eta * torch.sqrt((1 - abp) / (1 - ab)) * torch.sqrt(1 - ab / abp)
            assert c[t, 13] == sigma and c[t, 11] == torch.sqrt(abp)
            assert c[t, 12] == torch.sqrt(1 - abp - sigma ** 2)
            assert c[t, 2] == torch.sqrt(ab) and c[t, 3] == torch.sqrt(1 - ab)
            assert c[t, 14] == float(t != 0)


def test_diffusion_tables_equal_oracle():
    for sched in ("linear", "cosine", "quadratic"):
        d = F.create_gaussian_diffusion(steps=100, noise_schedule=sched)
        tab = dor.Tables(F.get_named_beta_schedule(sched, 100))
        for k in ("betas", "alphas_cumprod", "alphas_cumprod_prev", "sqrt_recip_alphas_cumprod",
                  "posterior_variance", "posterior_log_variance_clipped", "posterior_mean_coef1",
                  "posterior_mean_coef2"):
            assert np.array_equal(getattr(d, k), getattr(tab, k)), (sched, k)
    assert d.num_timesteps == 100 and d.model_var_type == F.ModelVarType.FIXED_LARGE
    assert F.create_gaussian_diffusion(steps=50, noise_schedule="cosine", learn_sigma=True).model_var_type == F.ModelVarType.LEARNED_RANGE
    assert F.create_gaussian_diffusion(steps=50, noise_schedule="cosine", sigma_small=True).model_var_type == F.ModelVarType.FIXED_SMALL
    assert F.create_gaussian_diffusion(steps=50, noise_schedule="cosine", predict_xstart=True).model_mean_type == F.ModelMeanType.START_X
    with pytest.raises(NotImplementedError):
        F.get_named_beta_schedule("nope", 10)


def test_factory_and_checkpoint_sniffing(tmp_path):
    from fidm_b200.train_inpainting import FFHQ_UNET_KWARGS, fold_lora, unwrap_state_dict
    sd = synth_state_dict(dict(FFHQ_UNET_KWARGS, image_size=256, in_channels=3), seed=0, prefix="")
    path = tmp_path / "ckpt.pt"
    torch.save({"state_dict": sd}, path)
    model, diffusion, info = F.create_model_and_diffusion(str(path), "cpu", img_size=256)
    assert info == {"missing_keys": [], "unexpected_keys": []}
    assert diffusion.num_timesteps == 1000 and diffusion.model_var_type == F.ModelVarType.LEARNED_RANGE
    assert len(model.state_dict()) == 362
    assert unwrap_state_dict({"model": 1}) == 1 and unwrap_state_dict({"a": 2}) == {"a": 2}
    assert unwrap_state_dict({"model_state_dict": 3}, keys=("model_state_dict", "state_dict")) == 3
    w = {"q.weight": torch.zeros(4, 3, 1), "q.lora_A.weight": torch.ones(2, 3), "q.lora_B.weight": torch.ones(4, 2)}
    f = fold_lora(w, alpha_over_r=0.5)
    assert list(f) == ["q.weight"] and torch.allclose(f["q.weight"], torch.full((4, 3, 1), 1.0))


def test_procedural_masks_cover_5_to_60_percent():
    d = synth_batch(16, 64, seed=0)
    cov = d["mask"].mean(dim=(1, 2, 3))
    assert (cov >= 0.05).all() and (cov <= 0.75).all()
    assert set(d["mask"].unique().tolist()) <= {0.0, 1.0}
    assert torch.equal(d["masked_image"], d["gt"] * d["gt_keep_mask"])
    assert torch.equal(d["gt_keep_mask"], 1 - d["mask"])


def test_topology_rejects_out_of_scope_arguments():
    with pytest.raises(NotImplementedError):
        F.UNetModel(64, 3, 64, 6, 1, (4,), dims=3)
    with pytest.raises(NotImplementedError):
        F.UNetModel(64, 3, 64, 6, 1, (4,), num_classes=10)


@pytest.mark.parametrize("B,H,W,C,want", [
    (8, 16, 16, 512, 1),      # 512 vectors per (image, group): the plain one-launch kernel
    (8, 64, 64, 512, 2),      # 8192 vectors, 256 blocks: statistics + apply
    (1, 64, 64, 512, 1),      # batch 1: a cluster of 4 blocks shares the (image, group)
    (2, 64, 64, 512, 1),      # batch 2: clusters of 2 (the clustered grid must stay within one wave of 148 blocks)
    (3, 64, 64, 512, 2),
    (1, 128, 128, 256, 1),    # 16384 vectors per group: the reach of 4 blocks x 8 vectors per thread
    (1, 256, 256, 256, 2),
    (4, 8, 8, 96, 2),         # 3 channels per group: no 16-byte vectors
])
def test_groupnorm_launch_plan(B, H, W, C, want):
    """fidm_groupnorm_num_launches is a planning query (no kernel runs): which GroupNorm path a tensor takes.  The
    engine counts launches with it and the one-launch / cluster thresholds of csrc/groupnorm.cu are pinned here."""
    lib = _lib.lib()
    a = _lib.GnArgs()
    a.dtype, a.y_dtype = _lib.BF16, _lib.F16
    a.batch, a.height, a.width, a.channels, a.groups = B, H, W, C, 32
    a.ld_x = a.ld_y = C
    buf = ctypes.create_string_buffer(64)
    a.x = a.y = ctypes.cast((ctypes.addressof(buf) + 15) // 16 * 16, ctypes.c_void_p)     # only alignment is inspected
    assert lib.fidm_groupnorm_num_launches(ctypes.byref(a)) == want
