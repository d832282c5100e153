"""Continuous batching on ADM256: one JSON line on stdout.

Workload: ADM256 bf16 (synthetic weights), 256x256, DDIM-50 on a 50-step cosine diffusion, injection on, seeded,
64 requests with procedural masks covering 5-60 % (utils.synth).  Alternated within each of --rounds rounds (the
median is reported):
  (a) each request alone through ddim_sample_loop at batch 1;
  (b) lockstep ddim_sample_loop batches of 8 (the bound when all requests are known up front);
  (c) the continuous sampler, 8 slots, all 64 requests queued at once;
  (d) the continuous sampler fed a deterministic Poisson arrival trace at --load of (b)'s rate.
For each: images/s, per-request latency from submit (or arrival) to result-ready (p50 / p95, CUDA events recorded at
completion), mean slot occupancy, and ms per iteration minus ms per evaluation alone (graph replay of the plan at
that batch), which is the host and sampler-step overhead.  Then K8 (all slots updating, DDIM eta=0, bf16 stem)
against the seeded K4 at batch 8 and 64, each in a CUDA graph of 20 launches, beside a 2 GiB device-to-device copy.
The card's name, power limit and clocks are read (not set) in the same call.

With --sampler dpm_solver the four arms run DPM-Solver++ 2M in --steps evaluations on the 1000-step quadratic diffusion
(as tools/dpm_solver_probe.py; (a) and (b) through dpm_solver_sample_loop, (c) and (d) through
continuous_dpm_solver_sampler), and the step timing is K9 (all slots updating at a second-order grid point, injection,
bf16 stem) against the seeded K6 on the same batch; its checks add the contract on the elementwise stand-in model.

With --sampler repaint the four arms run RePaint(--jump-length, --jump-n-sample) on the 50-step cosine diffusion
((a) and (b) through repaint_sample_loop, (c) and (d) through continuous_repaint_sampler) with 16 requests: at the
default (5, 3) a request takes 140 evaluations, so a round takes seconds rather than minutes.  The step timing is K10
(every slot on a jump evaluation, injection on, bf16 stem) against the seeded K4 STEP_UPDATE_ONLY + K7 pair it
replaces; its checks add the contract on the stand-in model.

    python tools/continuous_probe.py [--rounds 3] [--load 0.8] [--sampler ddim | dpm_solver | repaint] [--steps 20]
                                     [--jump-length 5] [--jump-n-sample 3]
"""
import argparse
import ctypes
import json
import os
import random
import statistics
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from repaint_probe import copy_gbs, event_ms, gpu_info  # noqa: E402

B, S, T, N = 8, 256, 50, 64


class Workload:
    """The sampler the arms run: DDIM-50 on the 50-step cosine diffusion (default), DPM-Solver++ 2M in `steps`
    evaluations on the 1000-step quadratic one, or RePaint(jump_length, jump_n_sample) on the 50-step cosine one.
    evals: model evaluations per request; n: requests per arm."""

    def __init__(self, F, sampler, steps, jump_length=5, jump_n_sample=3):
        from fidm_b200 import repaint
        self.dpm, self.rp, self.steps = sampler == "dpm_solver", sampler == "repaint", steps
        self.jl, self.jn = jump_length, jump_n_sample
        if self.dpm:
            self.d = F.create_gaussian_diffusion(steps=1000, learn_sigma=True, noise_schedule="quadratic")
        else:
            self.d = F.create_gaussian_diffusion(steps=T, learn_sigma=True, noise_schedule="cosine")
        if self.rp:
            self.evals = len(repaint.evaluation_plan(self.d.alphas_cumprod, jump_length, jump_n_sample))
        else:
            self.evals = steps if self.dpm else T
        self.n = 16 if self.rp else N

    def loop(self, fn, gt, keep, seeds):
        kw = dict(model_kwargs={"gt": gt, "gt_keep_mask": keep}, device=gt.device, use_inpainting_injection=True,
                  seeds=seeds)
        if self.dpm:
            return self.d.dpm_solver_sample_loop(fn, tuple(gt.shape), steps=self.steps, **kw)
        if self.rp:
            return self.d.repaint_sample_loop(fn, tuple(gt.shape), jump_length=self.jl, jump_n_sample=self.jn, **kw)
        return self.d.ddim_sample_loop(fn, tuple(gt.shape), **kw)

    def continuous(self, fn):
        if self.dpm:
            return self.d.continuous_dpm_solver_sampler(fn, slots=B, image_size=(S, S), steps=self.steps)
        if self.rp:
            return self.d.continuous_repaint_sampler(fn, slots=B, image_size=(S, S), jump_length=self.jl,
                                                     jump_n_sample=self.jn)
        return self.d.continuous_sampler(fn, slots=B, image_size=(S, S), sampler="ddim")


def _pct(v, q):
    v = sorted(v)
    return v[min(len(v) - 1, int(round(q * (len(v) - 1))))]


class _Clock:
    """GPU time since a synchronised origin, read from events (ms), and the host clock with the same origin (s)."""

    def __init__(self):
        torch.cuda.synchronize()
        self.e0 = torch.cuda.Event(enable_timing=True)
        self.e0.record()
        self.t0 = time.perf_counter()

    def mark(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def ms(self, e):
        return self.e0.elapsed_time(e)


def _standin(x, t, **k):
    """Per-sample elementwise eps model (tests/test_gpu_continuous.py), its value per image batch independent, with the
    variance channels the learned-sigma diffusion expects."""
    eps = torch.tanh(0.7 * x) * torch.cos(t.float().view(-1, 1, 1, 1) * 0.01) + 0.05 * k["gt"]
    return torch.cat([eps, torch.zeros_like(eps)], 1)


def standin_checks(w, gts, keeps, seeds, n=12):
    """The contract on the stand-in model at 256x256: n requests through 8 continuous slots (later ones admitted as
    earlier ones finish) against lockstep batch 8 and against each request alone."""
    cs = w.continuous(_standin)
    tk = [cs.submit(gts[k], keeps[k], seeds[k]) for k in range(n)]
    res = cs.drain()
    cont = torch.cat([res[t] for t in tk])
    lock = w.loop(_standin, gts[:B], keeps[:B], seeds[:B])
    alone = torch.cat([w.loop(_standin, gts[k:k + 1], keeps[k:k + 1], [seeds[k]]) for k in range(n)])
    return {"standin_continuous_equals_lockstep_b8": bool(torch.equal(cont[:B], lock)),
            "standin_continuous_equals_alone_b1": bool(torch.equal(cont, alone))}


def run_alone(w, fn, gts, keeps, seeds):
    clk, done = _Clock(), []
    for k in range(w.n):
        w.loop(fn, gts[k:k + 1], keeps[k:k + 1], [seeds[k]])
        done.append(clk.mark())
    torch.cuda.synchronize()
    lat = [clk.ms(e) for e in done]
    return {"wall_ms": lat[-1], "latency_ms": lat, "occupancy": 1.0, "iterations": w.n * w.evals}


def run_lockstep(w, fn, gts, keeps, seeds):
    clk, done = _Clock(), []
    for j in range(0, w.n, B):
        w.loop(fn, gts[j:j + B], keeps[j:j + B], seeds[j:j + B])
        done += [clk.mark()] * B
    torch.cuda.synchronize()
    lat = [clk.ms(e) for e in done]
    return {"wall_ms": lat[-1], "latency_ms": lat, "occupancy": 1.0, "iterations": w.n // B * w.evals}


def run_continuous(w, fn, gts, keeps, seeds, arrivals_s=None):
    """arrivals_s: host seconds after the origin at which each request arrives (None: all queued at the origin)."""
    cs = w.continuous(fn)
    clk = _Clock()
    arrive_ms, done, tickets = {}, {}, {}
    k, iters, busy = 0, 0, 0
    while k < w.n or cs.pending():
        now = time.perf_counter() - clk.t0
        while k < w.n and (arrivals_s is None or arrivals_s[k] <= now):
            tk = cs.submit(gts[k], keeps[k], seeds[k])
            tickets[tk] = k
            arrive_ms[tk] = 0.0 if arrivals_s is None else arrivals_s[k] * 1e3
            k += 1
        if not cs.pending():
            time.sleep(max(0.0, arrivals_s[k] - now))
            continue
        busy += min(B, cs.pending())          # slots busy in this iteration (admissions included)
        for tk, _ in cs.step():
            done[tk] = clk.mark()
        iters += 1
    torch.cuda.synchronize()
    lat = [clk.ms(done[tk]) - arrive_ms[tk] for tk in tickets]
    return {"wall_ms": max(clk.ms(e) for e in done.values()), "latency_ms": lat, "occupancy": busy / (iters * B),
            "iterations": iters}


def eval_ms(fn, batch):
    """ms per evaluation alone: graph replay of the plan of this batch size."""
    plan = fn.model.base_model.plan_for(batch, S, S)
    plan.run()
    return min(event_ms(plan.run, 20) for _ in range(3))


def k8_probe(d, batch, dev):
    """us per step, DDIM eta=0 update + cumulative injection + bf16 stem write: seeded K4 against K8, CUDA graph of 20."""
    from fidm_b200 import _lib as L
    from fidm_b200 import continuous, seeded
    g = torch.Generator(device=dev).manual_seed(batch)
    x = torch.randn(batch, 3, S, S, device=dev, generator=g)
    mo = torch.randn(batch, 6, S, S, device=dev, generator=g)
    gt = torch.rand(batch, 3, S, S, device=dev, generator=g)
    keep = (torch.rand(batch, 3, S, S, device=dev, generator=g) > 0.5).float()
    nxt = torch.empty_like(x)
    x_in = torch.zeros(batch, S, S, 16, device=dev, dtype=torch.bfloat16)
    t_in = torch.zeros(batch, device=dev)
    seeds = seeded.check_seeds(list(range(batch)), batch).to(dev)
    t = 30

    def k4():
        d._step(L.STEP_UPDATE_INJECT, x, t=t, t_inject=t - 1, model_out=mo, gt=gt, keep=keep,
                inject_noise=seeded.Draw(seeds, L.NOISE_INJECT, t - 1), ddim=True, want_next=True,
                stem=(x_in, t_in), t_next=float(t - 1), next_buf=nxt)

    from fidm_b200.gaussian_diffusion import _MEAN_CODE, _VAR_CODE
    a = L.StepArgs()
    a.batch, a.channels, a.hw = batch, 3, S * S
    a.sampler, a.mean_type, a.var_type = L.SAMPLER_DDIM, _MEAN_CODE[d.model_mean_type], _VAR_CODE[d.model_var_type]
    a.clip_denoised, a.cumulative, a.mask_channels, a.num_timesteps = 1, 1, 3, d.num_timesteps
    coef = d._coef(dev, 0.0)
    tv = torch.tensor([d._t_value(v) for v in range(d.num_timesteps)], dtype=torch.float32, device=dev)
    inj = torch.tensor(continuous.injection_draws(d, "all", True), dtype=torch.int32, device=dev)
    out = torch.empty_like(x)
    a.coef, a.x, a.model_out, a.gt, a.keep_mask, a.x_next = (L.ptr(v) for v in (coef, x, mo, gt, keep, nxt))
    a.stem_out, a.stem_dtype, a.stem_ld, a.t_out = L.ptr(x_in), L.BF16, 16, L.ptr(t_in)
    s = L.SlotArgs()
    s.t_value, s.inject_draw, s.out = L.ptr(tv), L.ptr(inj), L.ptr(out)
    for b in range(batch):
        s.action[b], s.seeds[b] = t, b

    def k8():
        L.check(L.lib().fidm_sampler_step_slots(ctypes.byref(a), ctypes.byref(s), L.stream()), "sampler_step_slots")

    # read x 12, model_out 12 (of 24: the variance half is not read by DDIM), gt 12, keep 12; write x 12, stem 6 B
    nbytes = batch * S * S * (12 + 12 + 12 + 12 + 12 + 6)
    res = {"batch": batch, "bytes_per_step": nbytes}
    for name, fn in (("seeded_k4", k4), ("k8", k8)):
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
        res[name] = {"us_per_step": round(ms * 1e3, 2), "gbs": round(nbytes / (ms * 1e-3) / 1e9, 1)}
        del graph
    k4()
    ref, ref_stem, ref_t = nxt.clone(), x_in.clone(), t_in.clone()
    nxt.zero_(), x_in.zero_(), t_in.zero_()
    k8()
    res["k8_equals_k4"] = bool(torch.equal(nxt, ref) and torch.equal(x_in, ref_stem) and torch.equal(t_in, ref_t))
    return res


def _graph_us(fn):
    """us per call of `fn`, replayed in a CUDA graph of 20 calls."""
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
    del graph
    return ms * 1e3


def k9_probe(d, steps, batch, dev):
    """us per step, order-2 update at grid point 5 + cumulative injection + bf16 stem: seeded K6 against K9 (every slot
    at that point, state and history in place), CUDA graph of 20."""
    from fidm_b200 import _lib as L
    from fidm_b200 import continuous, dpm_solver, seeded
    from fidm_b200.gaussian_diffusion import _MEAN_CODE
    k = 5
    grid = dpm_solver.timestep_grid(d.num_timesteps, steps)
    tab = d._dpm_table(dev, steps, 2, True)
    g = torch.Generator(device=dev).manual_seed(batch)
    x = torch.randn(batch, 3, S, S, device=dev, generator=g)
    mo = torch.randn(batch, 6, S, S, device=dev, generator=g)
    mp = torch.rand(batch, 3, S, S, device=dev, generator=g)
    gt = torch.rand(batch, 3, S, S, device=dev, generator=g)
    keep = (torch.rand(batch, 3, S, S, device=dev, generator=g) > 0.5).float()
    x_in = torch.zeros(batch, S, S, 16, device=dev, dtype=torch.bfloat16)
    t_in = torch.zeros(batch, device=dev)
    seeds = seeded.check_seeds(list(range(batch)), batch).to(dev)
    t_next = d._t_value(int(grid[k + 1]))

    def k6():
        return d._multistep(tab, k, x, mo, m_prev=mp, gt=gt, keep=keep,
                            inject_noise=seeded.Draw(seeds, L.NOISE_INJECT, int(grid[k + 1])), stem=(x_in, t_in),
                            t_next=t_next)

    xs, ms = x.clone(), mp.clone()
    tables = continuous.dpm_slot_tables(d, grid, 2, "all", True)
    tv, inj, order = (torch.tensor(v, dtype=dt, device=dev) for v, dt in
                      zip(tables, (torch.float32, torch.int32, torch.int32)))
    out = torch.empty_like(x)
    a = L.MultistepArgs()
    a.batch, a.channels, a.hw, a.steps = batch, 3, S * S, steps
    a.mean_type, a.out_channels, a.clip_denoised, a.mask_channels = _MEAN_CODE[d.model_mean_type], 6, 1, 3
    a.coef, a.x, a.model_out, a.m_prev, a.m_out, a.x_next, a.gt, a.keep_mask = (
        L.ptr(v) for v in (tab, xs, mo, ms, ms, xs, gt, keep))
    a.stem_out, a.stem_dtype, a.stem_ld, a.t_out = L.ptr(x_in), L.BF16, 16, L.ptr(t_in)
    s = L.MsSlotArgs()
    s.t_value, s.inject_draw, s.order, s.out = L.ptr(tv), L.ptr(inj), L.ptr(order), L.ptr(out)
    s.inject_tag = L.NOISE_INJECT
    for b in range(batch):
        s.action[b], s.seeds[b] = k, b

    def k9():
        L.check(L.lib().fidm_multistep_step_slots(ctypes.byref(a), ctypes.byref(s), L.stream()),
                "multistep_step_slots")

    def k9_fresh():                                  # every timed launch starts from the same state and history
        xs.copy_(x), ms.copy_(mp)
        k9()

    # read x, eps (3 of 6 channels), m_{k-1}, gt, mask: 5 x 12 B; write m_k, x_next: 2 x 12 B; stem 3 x bf16
    nbytes = batch * S * S * (5 * 12 + 2 * 12 + 6)
    res = {"batch": batch, "bytes_per_step": nbytes}
    for name, fn in (("seeded_k6", k6), ("k9", k9)):
        us = _graph_us(fn)
        res[name] = {"us_per_step": round(us, 2), "gbs": round(nbytes / (us * 1e-6) / 1e9, 1)}
    m_ref, x_ref = k6()
    ref_stem, ref_t = x_in.clone(), t_in.clone()
    x_in.zero_(), t_in.zero_()
    k9_fresh()
    res["k9_equals_k6"] = bool(torch.equal(xs, x_ref) and torch.equal(ms, m_ref) and torch.equal(x_in, ref_stem)
                               and torch.equal(t_in, ref_t))
    return res


def k10_probe(d, jl, jn, batch, dev):
    """us per step, every slot on the same jump evaluation (DDPM update, undo, cumulative injection at t_up, bf16 stem):
    the seeded K4 STEP_UPDATE_ONLY + K7 pair against K10, each in a CUDA graph of 20."""
    from fidm_b200 import _lib as L
    from fidm_b200 import continuous, seeded
    from fidm_b200.gaussian_diffusion import _MEAN_CODE, _VAR_CODE
    eval_t, next_t, undo, draws, admit = continuous.repaint_slot_tables(d, jl, jn, "all", True)
    k = next(k for k in range(len(eval_t)) if next_t[k] != eval_t[k] - 1 and draws[k] >= 0)
    t, t_up, (ua, us) = eval_t[k], next_t[k], undo[k]
    g = torch.Generator(device=dev).manual_seed(batch)
    x = torch.randn(batch, 3, S, S, device=dev, generator=g)
    mo = torch.randn(batch, 6, S, S, device=dev, generator=g)
    gt = torch.rand(batch, 3, S, S, device=dev, generator=g)
    keep = (torch.rand(batch, 3, S, S, device=dev, generator=g) > 0.5).float()
    smp, nxt = torch.empty_like(x), torch.empty_like(x)
    x_in = torch.zeros(batch, S, S, 16, device=dev, dtype=torch.bfloat16)
    t_in = torch.zeros(batch, device=dev)
    seeds = seeded.check_seeds(list(range(batch)), batch).to(dev)
    coef = d._coef(dev, 0.0)
    a4 = L.StepArgs()                                # K4 STEP_UPDATE_ONLY as _repaint_loop launches it
    a4.batch, a4.channels, a4.hw, a4.mode, a4.sampler = batch, 3, S * S, L.STEP_UPDATE_ONLY, L.SAMPLER_DDPM
    a4.mean_type, a4.var_type = _MEAN_CODE[d.model_mean_type], _VAR_CODE[d.model_var_type]
    a4.clip_denoised, a4.cumulative, a4.mask_channels, a4.num_timesteps = 1, 1, 1, d.num_timesteps
    a4.t_update, a4.t_inject = t, -1
    a4.coef, a4.x, a4.model_out, a4.sample = L.ptr(coef), L.ptr(x), L.ptr(mo), L.ptr(smp)
    s4 = L.SeededNoise()
    s4.seeds, s4.draw, s4.inject_tag, s4.inject_draw = L.ptr(seeds), k, L.NOISE_INJECT, 0

    def pair():
        L.check(L.lib().fidm_sampler_step_seeded(ctypes.byref(a4), ctypes.byref(s4), L.stream()), "sampler_step_seeded")
        d._resample(smp, seeded.Draw(seeds, L.NOISE_UNDO, k), ua, us, t_inject=t_up, gt=gt, keep=keep,
                    inject_noise=seeded.Draw(seeds, L.NOISE_INJECT, t_up), stem=(x_in, t_in),
                    t_next=d._t_value(t_up), next_buf=nxt)

    tv = torch.tensor([d._t_value(v) for v in range(d.num_timesteps)], dtype=torch.float32, device=dev)
    et, nt, dr = (torch.tensor(v, dtype=torch.int32, device=dev) for v in (eval_t, next_t, draws))
    ud = torch.tensor(undo, dtype=torch.float32, device=dev)
    out = torch.empty_like(x)
    a = L.StepArgs()
    a.batch, a.channels, a.hw, a.sampler = batch, 3, S * S, L.SAMPLER_DDPM
    a.mean_type, a.var_type = a4.mean_type, a4.var_type
    a.clip_denoised, a.cumulative, a.mask_channels, a.num_timesteps = 1, 1, 3, d.num_timesteps
    a.coef, a.x, a.model_out, a.gt, a.keep_mask, a.x_next = (L.ptr(v) for v in (coef, x, mo, gt, keep, nxt))
    a.stem_out, a.stem_dtype, a.stem_ld, a.t_out = L.ptr(x_in), L.BF16, 16, L.ptr(t_in)
    s = L.RpSlotArgs()
    s.t_value, s.eval_t, s.next_t, s.undo, s.inject_draw, s.out = (L.ptr(v) for v in (tv, et, nt, ud, dr, out))
    s.n_evals, s.admit_draw = len(eval_t), admit
    for b in range(batch):
        s.action[b], s.seeds[b] = k, b

    def k10():
        L.check(L.lib().fidm_repaint_step_slots(ctypes.byref(a), ctypes.byref(s), L.stream()), "repaint_step_slots")

    # per pixel, K4 DDPM with learned variance: read x 12, model_out 24, write sample 12; K7: read sample, gt, keep
    # 3 x 12, write x 12, stem 6.  K10 moves the same minus the sample's write and read (read x, model_out, gt, keep;
    # write x, stem): 78 of 102 B
    n_pair = batch * S * S * (12 + 24 + 12 + 3 * 12 + 12 + 6)
    n_k10 = batch * S * S * (12 + 24 + 2 * 12 + 12 + 6)
    res = {"batch": batch, "evaluation": k, "t": t, "t_up": t_up, "bytes_per_step_pair": n_pair,
           "bytes_per_step_k10": n_k10}
    for name, fn, nb in (("seeded_k4_k7", pair, n_pair), ("k10", k10, n_k10)):
        us_ = _graph_us(fn)
        res[name] = {"us_per_step": round(us_, 2), "gbs": round(nb / (us_ * 1e-6) / 1e9, 1)}
    pair()
    ref, ref_stem, ref_t = nxt.clone(), x_in.clone(), t_in.clone()
    nxt.zero_(), x_in.zero_(), t_in.zero_()
    k10()
    res["k10_equals_k4_k7"] = bool(torch.equal(nxt, ref) and torch.equal(x_in, ref_stem) and torch.equal(t_in, ref_t))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3, help="alternating timing rounds (the median is reported)")
    ap.add_argument("--load", type=float, default=0.8, help="Poisson arrival rate of (d) as a fraction of (b)'s rate")
    ap.add_argument("--sampler", choices=("ddim", "dpm_solver", "repaint"), default="ddim",
                    help="the sampler of every arm")
    ap.add_argument("--steps", type=int, default=20, help="model evaluations per request of --sampler dpm_solver")
    ap.add_argument("--jump-length", type=int, default=5, help="RePaint jump length of --sampler repaint")
    ap.add_argument("--jump-n-sample", type=int, default=3, help="RePaint jump_n_sample of --sampler repaint")
    args = ap.parse_args()
    import fidm_b200 as F
    from fidm_b200.utils.synth import synth_batch, synth_state_dict
    dev = torch.device("cuda", 0)
    F._lib.check(F._lib.lib().fidm_device_supported(0), "device")
    info = gpu_info()
    cfg = F.CONFIGS["ADM256"]
    model = F.DiffusionInpaintingModel(F.UNetModel(**dict(cfg, in_channels=3)))
    model.load_state_dict(synth_state_dict(cfg, seed=0), strict=True)
    model.to(dev)
    model.base_model.set_precision("bf16")
    fn = F.InpaintingModelFn(model)
    w = Workload(F, args.sampler, args.steps, args.jump_length, args.jump_n_sample)
    d = w.d
    data = synth_batch(N, S, seed=100, device=dev)
    gts, keeps = data["gt"], data["gt_keep_mask"]
    seeds = list(range(5000, 5000 + N))
    with torch.no_grad():
        # warm-up: plans and graphs of batch 1 and 8, tables; checks that (c) reproduces (a) and (b)
        lock = w.loop(fn, gts[:B], keeps[:B], seeds[:B])
        alone = w.loop(fn, gts[:1], keeps[:1], seeds[:1])
        cs = w.continuous(fn)
        tk = [cs.submit(gts[k], keeps[k], seeds[k]) for k in range(B)]
        res_c = cs.drain()
        cont = torch.cat([res_c[t] for t in tk])
        checks = {"continuous_equals_lockstep_b8": bool(torch.equal(cont, lock)),
                  "continuous_equals_alone_b1": bool(torch.equal(cont[:1], alone)),
                  "lockstep_b8_equals_alone_b1": bool(torch.equal(lock[:1], alone))}
        if w.dpm or w.rp:
            checks.update(standin_checks(w, gts, keeps, seeds))
        ev = {1: eval_ms(fn, 1), B: eval_ms(fn, B)}
        rate_b = None
        runs = {"a_alone_b1": lambda: run_alone(w, fn, gts, keeps, seeds),
                "b_lockstep_b8": lambda: run_lockstep(w, fn, gts, keeps, seeds),
                "c_continuous_all_queued": lambda: run_continuous(w, fn, gts, keeps, seeds),
                "d_continuous_poisson": None}
        got = {name: [] for name in runs}
        for r in range(args.rounds):
            for name, run in runs.items():
                if name == "d_continuous_poisson":
                    rate = args.load * rate_b                       # requests per second
                    rng = random.Random(r)
                    arr, t = [], 0.0
                    for _ in range(w.n):
                        t += rng.expovariate(rate)
                        arr.append(t)
                    got[name].append(run_continuous(w, fn, gts, keeps, seeds, arr))
                else:
                    got[name].append(run())
                if name == "b_lockstep_b8" and rate_b is None:
                    rate_b = w.n / (got[name][-1]["wall_ms"] * 1e-3)
        if w.dpm:
            steps = [k9_probe(d, args.steps, b, dev) for b in (8, 64)]
            checks["k9_equals_k6"] = all(st.pop("k9_equals_k6") for st in steps)
        elif w.rp:
            steps = [k10_probe(d, w.jl, w.jn, b, dev) for b in (8, 64)]
            checks["k10_equals_k4_k7"] = all(st.pop("k10_equals_k4_k7") for st in steps)
        else:
            steps = [k8_probe(d, b, dev) for b in (8, 64)]
    cp = copy_gbs(dev)
    for st in steps:
        for name in (("seeded_k6", "k9") if w.dpm else ("seeded_k4_k7", "k10") if w.rp else ("seeded_k4", "k8")):
            st[name]["fraction_of_copy"] = round(st[name]["gbs"] / cp, 3)
    out = {"probe": "continuous", "gpu": info,
           "config": "ADM256 bf16, 256x256, %s, injection on, seeded, 8 slots, %d requests (5-60 %% holes), "
                     "synthetic weights" % ("DPM-Solver++ 2M-%d quadratic 1000" % args.steps if w.dpm
                                            else "RePaint(%d, %d) cosine 50, %d evaluations per request"
                                            % (w.jl, w.jn, w.evals) if w.rp else "DDIM-50 cosine", w.n),
           "checks": checks, "eval_ms_alone": {str(k): round(v, 3) for k, v in ev.items()},
           "poisson_rate_per_s": round(args.load * rate_b, 3), "copy_gbs": cp, "step": steps, "runs": {}}
    for name, rs in got.items():
        batch = 1 if name == "a_alone_b1" else B
        walls = [r["wall_ms"] for r in rs]
        med = rs[walls.index(statistics.median_low(walls))]
        out["runs"][name] = {
            "images_per_s": round(w.n / (med["wall_ms"] * 1e-3), 3),
            "all_images_per_s": [round(w.n / (v * 1e-3), 3) for v in walls],
            "latency_p50_ms": round(_pct(med["latency_ms"], 0.5), 1),
            "latency_p95_ms": round(_pct(med["latency_ms"], 0.95), 1),
            "mean_slot_occupancy": round(med["occupancy"], 3),
            "iterations": med["iterations"],
            "ms_per_iteration": round(med["wall_ms"] / med["iterations"], 3),
            "overhead_ms_per_iteration": round(med["wall_ms"] / med["iterations"] - ev[batch], 3)}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
