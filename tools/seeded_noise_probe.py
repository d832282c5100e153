"""Per-image seeded noise on ADM256: one JSON line on stdout.

  * one DDPM step with fresh injection noise, as `randn_like x2 + K4` against the seeded K4 that generates both noise
    tensors in registers, each in a CUDA graph of 20 steps, at batch 8 and 64 (256x256, bf16 stem write); bytes each
    must move computed from the shapes, against a 2 GiB device-to-device copy timed in the same run;
  * ms per step of ddim_sample_loop (100 steps) and p_sample_loop (100-step diffusion) on ADM256 at batch 8, bf16,
    injection on, seeded and unseeded, alternated in the same call; the median of --rounds rounds;
  * peak allocated memory of a 1000-step p_sample_loop at batch 8, seeded against the cumulative noise cache.
The card's name, power limit and clocks are read (not set) in the same call.

    python tools/seeded_noise_probe.py [--rounds 3]
"""
import argparse
import json
import os
import statistics
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from repaint_probe import copy_gbs, event_ms, gpu_info  # noqa: E402


def step_probe(d, B, S, dev):
    """us per DDPM step (CUDA graph of 20), unseeded (two randn_like + K4) and seeded (K4 only)."""
    from fidm_b200 import _lib as L
    from fidm_b200 import seeded
    g = torch.Generator(device=dev).manual_seed(B)
    x = torch.randn(B, 3, S, S, device=dev, generator=g)
    mo = torch.randn(B, 6, S, S, device=dev, generator=g)
    gt = torch.rand(B, 3, S, S, device=dev, generator=g)
    keep = (torch.rand(B, 1, S, S, device=dev, generator=g) > 0.5).float()
    out = torch.empty_like(x)
    x_in = torch.zeros(B, S, S, 16, device=dev, dtype=torch.bfloat16)
    t_in = torch.zeros(B, device=dev)
    seeds = seeded.check_seeds(list(range(B)), B).to(dev)

    def step(z, n):
        d._step(L.STEP_UPDATE_INJECT, x, t=40, t_inject=39, model_out=mo, z=z, gt=gt, keep=keep, inject_noise=n,
                ddim=False, cumulative=False, want_next=True, stem=(x_in, t_in), t_next=39.0, next_buf=out)

    variants = {"randn_x2_k4": lambda: step(torch.randn_like(x), torch.randn_like(gt)),
                "seeded_k4": lambda: step(seeded.Draw(seeds, L.NOISE_STEP, 3), seeded.Draw(seeds, L.NOISE_INJECT_FRESH, 3))}
    px = B * S * S
    # K4, DDPM with learned range: read x 12, model_out 24, gt 12, mask 4 B; write x_next 12 + stem 6 B per pixel;
    # unseeded: + read z and n (24 B) and the two randn writes (24 B)
    base = 12 + 24 + 12 + 4 + 12 + 6
    nbytes = {"randn_x2_k4": px * (base + 48), "seeded_k4": px * base}
    res = {"batch": B}
    for name, fn in variants.items():
        for _ in range(3):
            fn()
        stream = torch.cuda.Stream()
        stream.wait_stream(torch.cuda.current_stream())
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.stream(stream):
            with torch.cuda.graph(graph):
                for _ in range(20):
                    fn()
        torch.cuda.current_stream().wait_stream(stream)
        graph.replay()
        ms = min(event_ms(graph.replay, 10) for _ in range(3)) / 20
        res[name] = {"us_per_step": round(ms * 1e3, 2), "bytes_per_step": nbytes[name],
                     "gbs": round(nbytes[name] / (ms * 1e-3) / 1e9, 1)}
        del graph
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="alternating timing rounds (the median is reported)")
    args = ap.parse_args()
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_batch, synth_state_dict
    dev = torch.device("cuda", 0)
    F._lib.check(F._lib.lib().fidm_device_supported(0), "device")
    info = gpu_info()
    B, S = 8, 256
    cfg = F.CONFIGS["ADM256"]
    model = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
    model.load_state_dict(synth_state_dict(cfg, seed=0), strict=True)
    model.to(dev)
    model.base_model.set_precision("bf16")
    fn = F.InpaintingModelFn(model)
    d = F.create_gaussian_diffusion(steps=100, learn_sigma=True, noise_schedule="cosine")
    data = synth_batch(B, S, seed=100, device=dev)
    mk = {"gt": data["gt"], "gt_keep_mask": data["gt_keep_mask"]}
    shape = (B, 3, S, S)
    seeds = list(range(1000, 1000 + B))
    kw = dict(model_kwargs=mk, device=dev, use_inpainting_injection=True)
    runs = {"ddim100": lambda: d.ddim_sample_loop(fn, shape, **kw),
            "ddim100_seeded": lambda: d.ddim_sample_loop(fn, shape, seeds=seeds, **kw),
            "ddpm100": lambda: d.p_sample_loop(fn, shape, **kw),
            "ddpm100_seeded": lambda: d.p_sample_loop(fn, shape, seeds=seeds, **kw)}
    with torch.no_grad():
        finite = {}
        for name, run in runs.items():                       # warm-up (plans, graphs, tables)
            torch.manual_seed(0)
            finite[name] = bool(torch.isfinite(run()).all())
        ms = {name: [] for name in runs}
        for _ in range(args.rounds):                         # alternate within each round
            for name, run in runs.items():
                torch.manual_seed(0)
                ms[name].append(event_ms(run))
        steps = [step_probe(d, b, S, dev) for b in (8, 64)]
        d1000 = F.create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="linear")
        peak = {}
        for name, extra in (("cumulative_cache", {}), ("seeded", {"seeds": seeds})):
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            torch.manual_seed(0)
            out = d1000.p_sample_loop(fn, shape, **kw, **extra)
            torch.cuda.synchronize()
            peak[name] = {"peak_allocated_mb_above_start": round((torch.cuda.max_memory_allocated() - base) / 1e6, 1),
                          "finite": bool(torch.isfinite(out).all())}
            del out
    cp = copy_gbs(dev)
    for s in steps:
        for name in ("randn_x2_k4", "seeded_k4"):
            s[name]["fraction_of_copy"] = round(s[name]["gbs"] / cp, 3)
    res = {"probe": "seeded_noise", "gpu": info,
           "config": "ADM256 bf16, batch 8, 256x256, injection on, synthetic weights", "copy_gbs": cp,
           "step": steps, "loops": {}, "ddpm1000_peak_memory": peak}
    for name in runs:
        m = statistics.median(ms[name])
        res["loops"][name] = {"ms_per_step": round(m / 100, 3), "all_ms": [round(v, 1) for v in ms[name]],
                              "finite": finite[name]}
    print(json.dumps(res))


if __name__ == "__main__":
    main()
