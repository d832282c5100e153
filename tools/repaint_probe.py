"""RePaint resampling on ADM256: one JSON line on stdout.

  * ms per model evaluation of repaint_sample_loop(jump_length=10, jump_n_sample=10) (910 evaluations) and of
    p_sample_loop (100 evaluations), alternated in the same call on the 100-step cosine diffusion; batch 8 at 256x256,
    bf16, injection on; the median of --rounds rounds;
  * resample_undo_kernel (K7: undo, injection, bf16 stem write) from CUDA events over a CUDA graph of 20 launches at
    batch 8 and 64, with the bytes it must move computed from the shapes, against a 2 GiB device-to-device copy timed
    in the same run.  At batch 8 the kernel's working set (~40 MB) is L2-resident; at batch 64 it is not.
The card's name, power limit and clocks are read (not set) in the same call.

    python tools/repaint_probe.py [--rounds 3]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm,clocks.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock, cur = (v.strip() for v in q[0].split(",")) if q else (torch.cuda.get_device_name(0), "?", "?", "?")
    return {"name": name, "power_limit": power, "max_sm_clock": clock, "sm_clock_at_start": cur}


def event_ms(fn, reps=1):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_probe(d, B, S, dev):
    """ms per resample_undo launch (CUDA graph of 20) and the bytes one launch must move."""
    g = torch.Generator(device=dev).manual_seed(B)
    x, u, n = (torch.randn(B, 3, S, S, device=dev, generator=g) for _ in range(3))
    gt = torch.rand(B, 3, S, S, device=dev, generator=g)
    keep = (torch.rand(B, 1, S, S, device=dev, generator=g) > 0.5).float()
    out = torch.empty_like(x)
    x_in = torch.zeros(B, S, S, 16, device=dev, dtype=torch.bfloat16)
    t_in = torch.zeros(B, device=dev)

    def launch():
        d._resample(x, u, 0.95, 0.3, t_inject=40, gt=gt, keep=keep, inject_noise=n, stem=(x_in, t_in), t_next=40.0,
                    next_buf=out)

    for _ in range(3):
        launch()
    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph):
            for _ in range(20):
                launch()
    torch.cuda.current_stream().wait_stream(stream)
    graph.replay()
    ms = min(event_ms(graph.replay, 10) for _ in range(3)) / 20
    px = B * S * S
    # read x, u, gt, noise: 4 x 12 B; mask 4 B; write x_next 12 B; stem 3 x bf16
    nbytes = px * (4 * 12 + 4 + 12 + 6)
    del graph
    return {"batch": B, "us_per_launch": round(ms * 1e3, 2), "bytes_per_launch": nbytes,
            "gbs": round(nbytes / (ms * 1e-3) / 1e9, 1)}


def copy_gbs(dev, gib=2):
    a = torch.empty(gib << 28, device=dev, dtype=torch.float32)
    b = torch.empty_like(a)
    b.copy_(a)
    ms = min(event_ms(lambda: b.copy_(a), 5) for _ in range(3))
    return round(2 * a.numel() * 4 / (ms * 1e-3) / 1e9, 1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="alternating timing rounds (the median is reported)")
    args = ap.parse_args()
    import fidm_b200 as F
    from fidm_b200 import repaint
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
    n_rp = len(repaint.evaluation_plan(d.alphas_cumprod, 10, 10))
    runs = {"ddpm100_cosine100": (100, lambda: d.p_sample_loop(fn, shape, model_kwargs=mk, device=dev,
                                                               use_inpainting_injection=True)),
            "repaint_10_10_cosine100": (n_rp, lambda: d.repaint_sample_loop(fn, shape, jump_length=10,
                                                                            jump_n_sample=10, model_kwargs=mk,
                                                                            device=dev))}
    with torch.no_grad():
        outs = {}
        for name, (_, run) in runs.items():                 # warm-up (plans, graphs, tables), and the outputs
            torch.manual_seed(0)
            outs[name] = run()
        ms = {name: [] for name in runs}
        for _ in range(args.rounds):                         # alternate the samplers within each round
            for name, (_, run) in runs.items():
                torch.manual_seed(0)
                ms[name].append(event_ms(run))
        kern = [kernel_probe(d, b, S, dev) for b in (8, 64)]
    cp = copy_gbs(dev)
    res = {"probe": "repaint", "gpu": info, "config": "ADM256 bf16, batch 8, 256x256, injection on, synthetic weights",
           "samplers": {}, "kernel": kern, "copy_gbs": cp}
    for name, (N, _) in runs.items():
        m = statistics.median(ms[name])
        res["samplers"][name] = {"evaluations": N, "ms_per_loop": round(m, 2), "ms_per_eval": round(m / N, 4),
                                 "all_ms": [round(v, 2) for v in ms[name]],
                                 "finite": bool(torch.isfinite(outs[name]).all())}
    res["repaint_ms_per_eval_over_ddpm"] = round(res["samplers"]["repaint_10_10_cosine100"]["ms_per_eval"]
                                                 / res["samplers"]["ddpm100_cosine100"]["ms_per_eval"], 4)
    for k in kern:
        k["fraction_of_copy"] = round(k["gbs"] / cp, 3)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
