#!/usr/bin/env python
"""Benchmark of the masked-inpainting sampling path (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload adm256|ref_ffhq256|t64]

A "step" is one complete pass of the hot path over one batch: a full `ddim_sample_loop` (DDIM-100,
cosine schedule, known-region injection on) for `--batch` 256x256 images per GPU on the ADM256
9-channel UNet (BASELINE configs[1]).  Prints ONE JSON line (rank 0).

`value`  : images/s with gt / masks / weights resident in HBM (CUDA-event time, max over ranks).
`e2e`    : the same metric through the public API with HOST buffers: pinned gt + mask -> H2D, the loop,
           D2H of the finished images, all inside the timed region.
`roofline`: the dominant kernel (tcgen05 implicit-GEMM conv, 256->256 @ 256x256) timed alone with CUDA
           events: algorithmic FLOPs per launch / average launch time vs the measured bf16 peak.
`cpu_baseline`: the reference's OWN CPU implementation (oracle/_ref: an unmodified, git-ignored copy of its five
           source files made by __graft_entry__.build(); `kind = "reference"`) timed on the host cores on a bounded
           sample of the same workload; the restatement in oracle/*.py (`kind = "port"`) if no copy exists.
`--impl reference`: the same CPU implementation, all host threads, one JSON line.
`--preset cfg3|cfg4|cfg5`: BASELINE.json configs[2] / [3] / [4] as one reproducible command each (see PRESETS).
`--global-batch G`: strong scaling -- G images split over the ranks (per-GPU batch G / N).
`--dump-outputs DIR`: after the timed steps, the images the last timed step returned go to DIR/samples.npy (float32), so
           that two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = {
    "adm256": dict(cfg="ADM256", size=256, ddim_steps=100, schedule="cosine", gflop_per_image_eval=2241.48,
                   label="ADM256 9-ch UNet (Improved-DDPM 256 config, attn 32/16/8), 256x256, DDIM-100 cosine, "
                         "known-region injection on (BASELINE configs[1])"),
    "ref_ffhq256": dict(cfg="REF_FFHQ256", size=256, ddim_steps=100, schedule="cosine", gflop_per_image_eval=388.84,
                        label="REF-FFHQ256 9-ch UNet (train_inpainting.py:208-224), 256x256, DDIM-100 cosine, "
                              "injection on"),
    "t64": dict(cfg="T64", size=64, ddim_steps=50, schedule="cosine", gflop_per_image_eval=20.03,
                label="T64 9-ch UNet, 64x64, DDIM-50 cosine, injection on (BASELINE configs[0])"),
}


# BASELINE.json configs[2..4] as one reproducible command each: `python bench.py --preset cfgN` (1 GPU) or under
# torchrun with --gpus N.  A preset fixes the GLOBAL batch (split over the ranks) -> "scaling": "strong".
PRESETS = {
    "cfg3": dict(workload="adm256", sampler="ddpm", ddim_steps=1000, schedule="linear", global_batch=32,
                 note="BASELINE configs[2]: ADM256 DDPM-1000 linear schedule, batch 32 batch-sharded over the ranks"),
    "cfg4": dict(workload="adm256", sampler="ddim", ddim_steps=50, schedule="cosine",
                 sweep=[1, 2, 4, 8, 16, 32, 64, 128, 256],
                 note="BASELINE configs[3]: ADM256 DDIM-50 cosine, global batch sweep 1-256, procedural masks 5-60 %"),
    "cfg5": dict(workload="adm256", sampler="ddim", ddim_steps=100, schedule="quadratic", global_batch=64, lora=True,
                 note="BASELINE configs[4]: ADM256 with LoRA-merged qkv / proj_out weights, DDIM-100 quadratic, batch 64 "
                      "batch-sharded over the ranks"),
}


DUMP_MAX_BYTES = 64_000_000 - 4096          # 64 MB (decimal) in all, with room for the .npy header


def dump_samples(path, samples):
    """Write `samples` [N, ...] as float32 to path/samples.npy.  Beyond DUMP_MAX_BYTES a fixed, seeded subset of whole
    images is kept, in batch order, so that runs with the same arguments write the same file."""
    import numpy as np
    samples = samples.detach().float().cpu()
    n = samples.shape[0]
    keep = max(1, DUMP_MAX_BYTES // max(1, samples[:1].numel() * 4))
    if n > keep:
        idx = torch.randperm(n, generator=torch.Generator().manual_seed(0))[:keep].sort().values
        samples = samples[idx]
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "samples.npy"), samples.numpy())


def peaks():
    p = {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "src": "fallback"}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            m = json.load(f)
        p.update(hbm_gbs=m["hbm_gbs"], bf16_tflops=m["bf16_tflops"],
                 bf16_tflops_sustained=m.get("bf16_tflops_sustained", m["bf16_tflops"]), src="measured")
    except Exception:
        pass
    return p


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.stop, self.index = [], threading.Event(), index
        self.th = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        while not self.stop.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([c.strip() for c in out.strip().split(",")])
            except Exception:
                pass
            self.stop.wait(0.2)

    def __enter__(self):
        self.th.start()
        return self

    def __exit__(self, *a):
        self.stop.set()
        self.th.join(timeout=6)

    def summary(self):
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_reference_sample(wl, evals, threads=None):
    """Time `evals` reverse steps (known-region injection + UNet evaluation + DDIM/DDPM update) at batch 1 on the host
    cores.  Runs the reference's own code (oracle/_ref: its GaussianDiffusion.ddim_sample / p_sample driving its
    DiffusionInpaintingModel) when that copy exists, else the oracle restatement.  Returns (seconds per step, cores,
    kind)."""
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_batch, synth_state_dict
    from oracle import ref_loader
    cores = threads or os.cpu_count()
    torch.set_num_threads(cores)
    cfg = F.CONFIGS[wl["cfg"]]
    sd = synth_state_dict(cfg, seed=0)
    data = synth_batch(1, wl["size"], seed=0)
    gt, keep = data["gt"], data["gt_keep_mask"]
    shape = (1, 3, wl["size"], wl["size"])
    x = torch.randn(*shape)
    ddpm = wl.get("sampler", "ddim") == "ddpm"
    times = []
    ref = ref_loader.load()
    if ref is not None:
        model = ref_loader.build_model(cfg, sd)
        d = ref.create_gaussian_diffusion(steps=wl["ddim_steps"], learn_sigma=True, noise_schedule=wl["schedule"])
        masked, mask = gt * keep, 1 - keep

        def model_fn(xx, ts, **kw):                      # the closure of test_inp_ddim_100.py:373-385
            return model(xx, ts, masked_image=masked, mask=mask)

        step = d.p_sample if ddpm else d.ddim_sample
        with torch.no_grad():
            for i in range(evals):
                t = torch.full((1,), wl["ddim_steps"] - 1 - i, dtype=torch.int64)
                t0 = time.perf_counter()
                x = step(model_fn, x, t, model_kwargs={"gt": gt, "gt_keep_mask": keep}, use_inpainting_injection=True)["sample"]
                times.append(time.perf_counter() - t0)
        return times, cores, "reference"
    from oracle import diffusion_oracle as dor
    from oracle import unet_oracle as uor
    tab = dor.Tables(F.get_named_beta_schedule(wl["schedule"], wl["ddim_steps"]))
    with torch.no_grad():
        for i in range(evals):
            t = wl["ddim_steps"] - 1 - i
            t0 = time.perf_counter()
            x = dor.inject(tab, x, t, gt, keep, torch.randn_like(gt))
            out = uor.inpaint_forward(sd, cfg, x, torch.full((1,), t), gt * keep, 1 - keep)
            x, _ = (dor.ddpm_update if ddpm else dor.ddim_update)(tab, out, x, t, torch.randn_like(x))
            times.append(time.perf_counter() - t0)
    return times, cores, "port"


def run_reference(args, wl):
    """--impl reference: the reference's own CPU implementation of the path (oracle/_ref, the unmodified copy that
    travels with the snapshot; the oracle port if absent), each step = one reverse step at batch 1."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n = args.warmup + args.steps
    times, cores, kind = cpu_reference_sample(wl, n)
    t = times[args.warmup:]
    sec = sum(t) / len(t)
    value = 1.0 / (sec * wl["ddim_steps"])
    sample = (f"{len(t)} x one reverse step (injection + UNet eval + update) of the reference's own code at batch 1, "
              f"extrapolated x{wl['ddim_steps']} steps")
    line = {"impl": "reference", "metric": (f"inpainted 256x256 images/s ({wl['sampler'].upper()}-{wl['ddim_steps']})"
                                            if wl["size"] == 256 else "inpainted images/s"), "value": value, "unit": "images/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": wl["label"], "per_gpu_batch": 1},
            "cpu_baseline": {"value": value, "unit": "images/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed sampling loops (default 2)")
    ap.add_argument("--warmup", type=int, default=None, help="untimed sampling loops before them (default 3)")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="adm256", choices=sorted(WORKLOADS))
    ap.add_argument("--batch", type=int, default=8, help="images per GPU")
    ap.add_argument("--ddim-steps", type=int, default=None)
    ap.add_argument("--schedule", default=None, choices=["cosine", "linear", "quadratic"],
                    help="noise schedule (BASELINE configs[2]: linear, configs[4]: quadratic); default: the workload's")
    ap.add_argument("--sampler", default="ddim", choices=["ddim", "ddpm"],
                    help="ddpm: p_sample_loop over all --ddim-steps timesteps (BASELINE configs[2]: DDPM-1000)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--eval-only", action="store_true", help="only time UNet evaluations (ms per eval)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32", "fp8"],
                    help="fp8: opt-in mode, the large GroupNorm-fused 3x3 convs on e4m3 operands (not the headline precision)")
    ap.add_argument("--preset", default=None, choices=sorted(PRESETS))
    ap.add_argument("--global-batch", type=int, default=None,
                    help="strong scaling: this many images split over the ranks (per-GPU batch = G / N)")
    ap.add_argument("--lora", action="store_true", help="LoRA-merged qkv / proj_out weights (same keys and shapes)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the images the last timed step returned to DIR/samples.npy (float32, at most 64 MB: a "
                         "fixed, seeded subset of whole images beyond that)")
    args = ap.parse_args()
    preset = PRESETS.get(args.preset)
    fixed_count = args.eval_only or (preset and "sweep" in preset)       # these modes time a fixed number of runs
    if fixed_count and (args.steps is not None or args.warmup is not None):
        ap.error("--steps / --warmup do not apply to --eval-only (40 timed evaluations) or a sweep (one loop per size)")
    args.steps = 2 if args.steps is None else args.steps
    args.warmup = 3 if args.warmup is None else args.warmup
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (fixed_count or args.impl == "reference"):
        ap.error("--dump-outputs applies to the sampling benchmark only (not --eval-only, --impl reference or a sweep)")
    if preset:
        args.workload, args.sampler, args.ddim_steps, args.schedule = (preset["workload"], preset["sampler"],
                                                                        preset["ddim_steps"], preset["schedule"])
        args.lora = args.lora or preset.get("lora", False)
        if "global_batch" in preset and args.global_batch is None:
            args.global_batch = preset["global_batch"]
    wl = dict(WORKLOADS[args.workload])
    wl["sampler"] = args.sampler
    if args.ddim_steps:
        wl["ddim_steps"] = args.ddim_steps
    if args.schedule:
        wl["schedule"] = args.schedule
    if args.schedule or args.sampler != "ddim" or args.ddim_steps:
        wl["label"] += f" [variant: {args.sampler.upper()}-{wl['ddim_steps']} {wl['schedule']}]"
    if args.lora:
        wl["label"] += " [LoRA-merged attention weights]"
    if preset:
        wl["label"] = preset["note"]
    if args.impl == "reference":
        return run_reference(args, wl)

    import fidm_b200 as F
    from fidm_b200 import ops
    from fidm_b200.parallel import gather_batch
    from fidm_b200.utils.synth import synth_batch, synth_state_dict
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        # The JSON line must be the only thing on stdout, but NCCL printf()s its version banner there while the
        # communicator is created: point fd 1 at stderr for the duration of the (eager) initialisation.
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)
    F._lib.check(F._lib.lib().fidm_device_supported(local), "device")

    cfg = F.CONFIGS[wl["cfg"]]
    strong = args.global_batch is not None
    if strong:
        if args.global_batch % world:
            raise SystemExit(f"--global-batch {args.global_batch} is not a multiple of {world} ranks")
        args.batch = args.global_batch // world
    B, S, T = args.batch, wl["size"], wl["ddim_steps"]
    model = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
    sd = synth_state_dict(cfg, seed=0)
    if args.lora:
        from fidm_b200.utils.synth import merge_lora
        sd = merge_lora(sd, rank=8, alpha=64.0, seed=0)
    model.load_state_dict(sd, strict=True)
    del sd
    model.to(dev)
    model.base_model.set_precision(args.precision)
    fn = F.InpaintingModelFn(model)
    diffusion = F.create_gaussian_diffusion(steps=T, learn_sigma=True, noise_schedule=wl["schedule"])
    if preset and "sweep" in preset:
        return run_sweep(args, preset, wl, model, fn, diffusion, dev, world, rank, local)
    data = synth_batch(B, S, seed=100 + rank, device=dev)
    gt, keep = data["gt"], data["gt_keep_mask"]
    host_gt, host_keep = data["gt"].cpu().pin_memory(), data["gt_keep_mask"].cpu().pin_memory()
    host_out = torch.empty(B * world if False else B, 3, S, S).pin_memory()
    torch.manual_seed(1234 + rank)
    torch.cuda.manual_seed(1234 + rank)

    def loop(g, k):
        # every loop starts from the same generator state: the noise of the last timed step depends on the seed alone,
        # not on --warmup / --steps
        torch.cuda.manual_seed(1234 + rank)
        if args.sampler == "ddpm":
            return diffusion.p_sample_loop(fn, (B, 3, S, S), model_kwargs={"gt": g, "gt_keep_mask": k}, device=dev,
                                           use_inpainting_injection=True)
        return diffusion.ddim_sample_loop(fn, (B, 3, S, S), model_kwargs={"gt": g, "gt_keep_mask": k}, device=dev,
                                          eta=0.0, use_inpainting_injection=True)

    last = {}

    def step_device():
        out = loop(gt, keep)
        last["samples"] = gather_batch(out, B * world) if world > 1 else out
        return last["samples"]

    def step_e2e():
        g = host_gt.to(dev, non_blocking=True)
        k = host_keep.to(dev, non_blocking=True)
        out = loop(g, k)
        host_out.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return out

    def sync_all():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn_step, k):
        sync_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            fn_step()
        e1.record()
        sync_all()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item()

    if args.eval_only:
        xin = torch.randn(B, 3, S, S, device=dev)
        tt = torch.full((B,), T // 2, device=dev)
        for _ in range(5):
            fn(xin, tt, gt=gt, gt_keep_mask=keep)
        with ClockSampler(local) as clk:
            ms_eval = timed(lambda: fn(xin, tt, gt=gt, gt_keep_mask=keep), 40) / 40
        print(json.dumps({"ms_per_unet_eval": ms_eval, "batch": B, "tflops": wl["gflop_per_image_eval"] * B / ms_eval,
                          "norm_dtype": os.environ.get("FIDM_NORM_DTYPE", "fp16"), "clocks": clk.summary()}), flush=True)
        return
    for _ in range(max(args.warmup, 1)):
        step_device()
    with ClockSampler(local) as clk:
        ms = timed(step_device, args.steps)
    if args.dump_outputs and rank == 0:
        dump_samples(args.dump_outputs, last["samples"])
    ms_e2e = timed(step_e2e, args.steps)
    images = B * world * args.steps
    value = images / (ms / 1e3)
    e2e_value = images / (ms_e2e / 1e3)

    plan = model.base_model.plan_for(B, S, S)
    launches_per_loop = T * (plan.n_launches() + 2) + 1          # + pack + K4 per step, + first injection
    # UNet-only timing (ms per eval at this batch)
    xin = torch.randn(B, 3, S, S, device=dev)
    tt = torch.full((B,), T // 2, device=dev)
    for _ in range(3):
        fn(xin, tt, gt=gt, gt_keep_mask=keep)
    ms_eval = timed(lambda: fn(xin, tt, gt=gt, gt_keep_mask=keep), 10) / 10
    tf_eval = wl["gflop_per_image_eval"] * B / ms_eval            # GFLOP / ms == TFLOP/s

    pk = peaks()
    line = {
        "metric": (f"inpainted 256x256 images/s ({args.sampler.upper()}-{T})" if S == 256 else "inpainted images/s"),
        "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if strong else "weak",
        "vs_baseline": None, "dtype": args.precision,
        "dtype_note": ("bf16 residual stream / qkv / attention operands; NORMALIZED conv operands (GroupNorm outputs) and the "
                       "weights they multiply are fp16 -- same width and tensor rate as bf16, 11-bit mantissa, saturating "
                       "converts; fp32 accumulation") if args.precision == "bf16" else
                      ("OPT-IN reduced precision: as bf16, but the large GroupNorm-fused 3x3 convolutions multiply e4m3 "
                       "operands with e4m3 weights (per-output-channel scale); outside the north star's eps bar"
                       if args.precision == "fp8" else "FFMA verification mode"),
        "data": "synthetic",
        "config": {"workload": wl["label"], "preset": args.preset, "per_gpu_batch": B, "global_batch": B * world, "ddim_steps": T,
                   "parallelism": f"batch-sharded x{world}, no collective in the loop, one all_gather of the outputs",
                   "l2": f"no flush: one UNet eval streams {plan.pool.nbytes() / 1e9:.1f}+ GB of activations (>> 126 MB L2)",
                   "cuda_graph": bool(model.base_model.use_cuda_graph)},
        "ms_per_unet_eval": ms_eval,
        "unet_eval": {"batch": B, "tflops": tf_eval, "frac_of_sustained_peak": tf_eval / pk["bf16_tflops_sustained"],
                      "peak_src": pk["src"]},
        "e2e": {"value": e2e_value, "unit": "images/s", "h2d_bytes_per_step": host_gt.numel() * 4 + host_keep.numel() * 4,
                "d2h_bytes_per_step": host_out.numel() * 4},
        "gpu_launches": launches_per_loop * args.steps,
        "clocks": clk.summary(),
    }

    line["config"]["operand_dtypes"] = ("residual stream / qkv / attention bf16; normalized conv operands and their "
                                        "weights fp16; fp32 accumulation, statistics, softmax and sampler state")
    if rank == 0:
        line["roofline"] = dominant_kernel_roofline(ops, dev, pk, B)
        if args.precision == "fp8":
            line["roofline_fp8"] = fp8_kernel_roofline(ops, dev, B)
            line["config"]["fp8_convs_per_eval"] = plan.n_fp8
        line["hbm_kernels"] = hbm_kernel_rooflines(ops, diffusion, dev, pk, B, S)
        if world == 1 and not args.no_cpu_baseline:
            evals = 2 if S == 256 else 5
            times, cores, kind = cpu_reference_sample(wl, evals + 1)
            sec = sum(times[1:]) / len(times[1:])
            line["cpu_baseline"] = {"value": 1.0 / (sec * T), "unit": "images/s", "cores": cores, "kind": kind,
                                    "sample": f"{evals} x one reverse step (injection + UNet eval + update) at batch 1 after 1 "
                                              f"warm-up, extrapolated x{T} steps ({sec:.2f} s per step)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_sweep(args, preset, wl, model, fn, diffusion, dev, world, rank, local):
    """--preset cfg4: one full DDIM loop per global batch size of the sweep (per-GPU batch = max(1, G / N); sizes that
    give the same per-GPU batch as a smaller G are skipped), device-timed, max over ranks."""
    import torch.distributed as dist
    from fidm_b200.utils.synth import synth_batch
    S, T = wl["size"], wl["ddim_steps"]
    rows, seen = [], set()
    for G in preset["sweep"]:
        b = max(1, G // world)
        if b in seen:
            continue
        seen.add(b)
        data = synth_batch(b, S, seed=100 + rank, device=dev)
        gt, keep = data["gt"], data["gt_keep_mask"]
        xin = torch.randn(b, 3, S, S, device=dev)
        tt = torch.full((b,), T // 2, device=dev)
        for _ in range(3):                                    # warm-up: plan build, graph capture, clocks
            fn(xin, tt, gt=gt, gt_keep_mask=keep)
        # ... and the loop's own first-use costs (fused plan inputs, ping-pong buffers from a just-emptied allocator, K4):
        # three steps of the same loop, untimed -- they were ~40 ms of a 190 ms batch-1 loop
        for i, _ in enumerate(diffusion.ddim_sample_loop_progressive(fn, (b, 3, S, S), model_kwargs={"gt": gt, "gt_keep_mask": keep},
                                                                     device=dev, eta=0.0, use_inpainting_injection=True)):
            if i == 2:
                break
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        diffusion.ddim_sample_loop(fn, (b, 3, S, S), model_kwargs={"gt": gt, "gt_keep_mask": keep}, device=dev,
                                   eta=0.0, use_inpainting_injection=True)
        e1.record()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = ms.item()
        hole = float((1 - keep).mean().item())
        rows.append({"global_batch": b * world, "per_gpu_batch": b, "ms_per_loop": ms, "images_per_s": b * world / (ms / 1e3),
                     "unet_tflops_per_gpu": wl["gflop_per_image_eval"] * b * T / ms, "mask_hole_fraction_rank0": hole})
        model.base_model._plans.clear()                       # release this batch size's buffers and graph
        del data, gt, keep, xin
        torch.cuda.empty_cache()
    if rank == 0:
        pk = peaks()
        best = max(rows, key=lambda r: r["images_per_s"])
        for r in rows:
            r["frac_of_sustained_peak"] = r["unet_tflops_per_gpu"] / pk["bf16_tflops_sustained"]
        print(json.dumps({"metric": f"inpainted 256x256 images/s (DDIM-{T}), batch sweep", "value": best["images_per_s"],
                          "unit": "images/s", "n_gpus": world, "steps": 1, "warmup": 3, "ms_per_step": best["ms_per_loop"],
                          "higher_is_better": True, "scaling": "sweep", "vs_baseline": None, "dtype": args.precision,
                          "data": "synthetic", "config": {"workload": wl["label"], "preset": args.preset},
                          "sweep": rows}), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def _time_launches(fn, n=20):
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def hbm_kernel_rooflines(ops, diffusion, dev, pk, B, S):
    """The two HBM-bound kernels against the measured copy bandwidth: K2 GroupNorm+SiLU apply on the largest
    activation (256 channels at full resolution, statistics from the producer's fused column sums) and K4, the
    fused sampler step (DDIM eta=0 update + injection: 64 B per pixel)."""
    from fidm_b200 import _lib as L
    Cc = 256
    x = torch.randn(B, S, S, Cc, device=dev).bfloat16()
    y = torch.empty(B, S, S, Cc, device=dev, dtype=torch.float16)
    gamma, beta = torch.ones(Cc, device=dev), torch.zeros(Cc, device=dev)
    xf = x.float()
    cs = torch.stack([xf.sum(dim=(1, 2)), (xf * xf).sum(dim=(1, 2))], dim=-1).contiguous()
    del xf
    ms_gn = _time_launches(lambda: ops.groupnorm_silu(x, gamma, beta, out=y, chansum=cs))
    by_gn = 2.0 * x.numel() * 2
    xs = torch.randn(B, 3, S, S, device=dev)
    mo = torch.randn(B, 6, S, S, device=dev)
    gt = torch.rand(B, 3, S, S, device=dev)
    keep = (torch.rand(B, 1, S, S, device=dev) > 0.5).float()
    n = torch.randn(B, 3, S, S, device=dev)
    T = diffusion.num_timesteps
    ms_k4 = _time_launches(lambda: diffusion._step(L.STEP_UPDATE_INJECT, xs, t=T // 2, t_inject=T // 2 - 1, model_out=mo,
                                                   gt=gt, keep=keep, inject_noise=n, ddim=True, want_next=True), n=50)
    by_k4 = 64.0 * B * S * S
    # the same launch without the Python launcher: 20 launches captured in a CUDA graph, replayed
    ms_k4_graph = None
    try:
        g = torch.cuda.CUDAGraph()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            outs = [torch.empty_like(xs) for _ in range(2)]
            with torch.cuda.graph(g, stream=side):
                for i in range(20):
                    diffusion._step(L.STEP_UPDATE_INJECT, xs, t=T // 2, t_inject=T // 2 - 1, model_out=mo, gt=gt, keep=keep,
                                    inject_noise=n, ddim=True, want_next=True, next_buf=outs[i & 1])
        torch.cuda.synchronize()
        ms_k4_graph = _time_launches(g.replay, n=10) / 20
    except Exception:          # pragma: no cover
        pass
    # the same kernel on 64 images (268 MB per launch), where the launch latency no longer dominates
    B2 = 64
    xs2, mo2 = torch.randn(B2, 3, S, S, device=dev), torch.randn(B2, 6, S, S, device=dev)
    gt2, n2 = torch.rand(B2, 3, S, S, device=dev), torch.randn(B2, 3, S, S, device=dev)
    keep2 = (torch.rand(B2, 1, S, S, device=dev) > 0.5).float()
    ms_k4b = _time_launches(lambda: diffusion._step(L.STEP_UPDATE_INJECT, xs2, t=T // 2, t_inject=T // 2 - 1, model_out=mo2,
                                                    gt=gt2, keep=keep2, inject_noise=n2, ddim=True, want_next=True), n=50)
    by_k4b = 64.0 * B2 * S * S
    return {"groupnorm_silu_apply": {"bytes_per_launch": by_gn, "ms_per_launch": ms_gn, "achieved_gbs": by_gn / ms_gn / 1e6,
                                     "frac_of_hbm_peak": by_gn / ms_gn / 1e6 / pk["hbm_gbs"]},
            "sampler_step": {"bytes_per_launch": by_k4, "ms_per_launch": ms_k4, "achieved_gbs": by_k4 / ms_k4 / 1e6,
                             "frac_of_hbm_peak": by_k4 / ms_k4 / 1e6 / pk["hbm_gbs"],
                             "note": "34 MB per launch at batch 8: launch-latency bound (includes the Python launcher)",
                             "ms_per_launch_in_cuda_graph": ms_k4_graph,
                             "frac_of_hbm_peak_in_cuda_graph": (by_k4 / ms_k4_graph / 1e6 / pk["hbm_gbs"]) if ms_k4_graph else None},
            "sampler_step_batch64": {"bytes_per_launch": by_k4b, "ms_per_launch": ms_k4b,
                                     "achieved_gbs": by_k4b / ms_k4b / 1e6,
                                     "frac_of_hbm_peak": by_k4b / ms_k4b / 1e6 / pk["hbm_gbs"]},
            "peak_gbs": pk["hbm_gbs"], "peak_src": pk["src"]}


def measured_fp8_peak(dev):
    """Dense e4m3 GEMM throughput of this GPU, measured here (torch._scaled_mm -> cuBLASLt, 8192^3, best of 10):
    the denominator of the FP8 kernel's roofline -- the bf16 peak of MEASURED_PEAKS.json is not reused."""
    n = 8192
    a = torch.randn(n, n, device=dev).to(torch.float8_e4m3fn)
    b = torch.randn(n, n, device=dev).to(torch.float8_e4m3fn).t()          # column-major B, as cuBLASLt wants
    one = torch.ones((), device=dev)
    best = 1e9
    for i in range(13):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        torch._scaled_mm(a, b, scale_a=one, scale_b=one, out_dtype=torch.bfloat16)
        e1.record()
        torch.cuda.synchronize()
        if i >= 3:
            best = min(best, e0.elapsed_time(e1))
    return 2.0 * n ** 3 / (best * 1e-3) / 1e12


def fp8_kernel_roofline(ops, dev, B):
    """The dominant layer (conv 3x3 256->256 @256x256) on the opt-in e4m3 path, timed alone, against the FP8 GEMM
    throughput measured in this run."""
    import math
    Cin = Cout = 256
    H = W = 256
    x = torch.randn(B, H, W, Cin, device=dev).bfloat16()
    w8, scale = ops.quantize_weight_e4m3(ops.repack_weight(torch.randn(Cout, Cin, 3, 3, device=dev) / math.sqrt(Cin * 9),
                                                              torch.float32))
    b = torch.zeros(Cout, device=dev)
    y = torch.empty(B, H, W, Cout, device=dev, dtype=torch.bfloat16)
    coef = ops.groupnorm_silu_coeff(x, torch.ones(Cin, device=dev), torch.zeros(Cin, device=dev))
    ms = _time_launches(lambda: ops.conv2d(x, w8, b, out=y, impl="tc", gn_coef=coef, w_scale=scale))
    flops = 2.0 * B * H * W * Cout * Cin * 9
    ach = flops / (ms * 1e-3) / 1e12
    try:
        peak = measured_fp8_peak(dev)
        src = "torch._scaled_mm e4m3 8192^3, best of 10, measured in this run"
    except Exception as e:          # pragma: no cover
        peak, src = 4500.0, f"nominal dense fp8 (measurement failed: {e})"
    return {"kernel": "conv_halo_kernel<256, e4m3> (GroupNorm+SiLU operand path + 3x3 conv, 256->256, 256x256, batch %d)" % B,
            "bound": "tensor", "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "peak_src": src,
            "ms_per_launch": ms, "flops_per_launch": flops}


def dominant_kernel_roofline(ops, dev, pk, B):
    """The dominant layer, conv3x3 256->256 @ 256x256 (31 % of ADM256 FLOPs, SURVEY Appendix B), as it runs inside the
    UNet: K1h = GroupNorm+SiLU of the raw input applied in the operand path + tcgen05 implicit GEMM + fused output
    statistics; timed alone on this stream.  K1 (same layer on a pre-normalized operand) is reported beside it."""
    import math
    Cin = Cout = 256
    H = W = 256
    x = torch.randn(B, H, W, Cin, device=dev).bfloat16()           # 268 MB at B=8: larger than L2
    x16 = x.half()
    w16 = ops.repack_weight(torch.randn(Cout, Cin, 3, 3, device=dev) / math.sqrt(Cin * 9), torch.float16)
    b = torch.zeros(Cout, device=dev)
    y = torch.empty(B, H, W, Cout, device=dev, dtype=torch.bfloat16)
    coef = ops.groupnorm_silu_coeff(x, torch.ones(Cin, device=dev), torch.zeros(Cin, device=dev))
    ms = _time_launches(lambda: ops.conv2d(x, w16, b, out=y, impl="tc", gn_coef=coef))
    ms_k1 = _time_launches(lambda: ops.conv2d(x16, w16, b, out=y, impl="tc"))
    flops = 2.0 * B * H * W * Cout * Cin * 9
    ach = flops / (ms * 1e-3) / 1e12
    return {"kernel": "conv_halo_kernel<256> (GroupNorm+SiLU operand path + 3x3 conv, 256->256, 256x256, batch %d)" % B,
            "bound": "tensor", "achieved": ach, "peak": pk["bf16_tflops"], "unit": "TFLOP/s", "frac": ach / pk["bf16_tflops"],
            "peak_src": pk["src"] + " burst (kernel timed alone)", "ms_per_launch": ms,
            "flops_per_launch": flops,
            # dram__bytes_read.sum + dram__bytes_write.sum of this kernel at batch 8 from the committed
            # `ncu --set full` capture (profiles/r1d_ncu_full_conv_halo.txt): 269.7 MB + 238.7 MB; the algorithmic
            # minimum is 268.4 MB in + 268.4 MB out + 1.2 MB of weights
            # NOT measured in this run: dram bytes of this kernel at batch 8 from the committed `ncu --set full` capture
            # (profiles/r1d_ncu_full_conv_halo.txt: 269.7 MB read + 238.7 MB written); scaled by batch when it differs
            "traffic": 508.4e6 * B / 8,
            "ncu_capture": {"file": "profiles/r1d_ncu_full_conv_halo.txt", "batch": 8, "dram_bytes": 508.4e6,
                            "tensor_pipe_active_pct": 84.6, "static": True},
            "k1_same_layer_prenormalized_operand": {"ms_per_launch": ms_k1, "achieved": flops / (ms_k1 * 1e-3) / 1e12}}


if __name__ == "__main__":
    main()
