"""Continuous batching for the inpainting loops.

The lockstep loops run a batch of B images from x_T to x_0 together.  Requests that arrive one at a time are served
better by a fixed batch of B *slots*: every iteration is one model evaluation of all slots, each slot holds its own
request at its own timestep, a request that finishes leaves its slot at the end of an iteration and the next queued
request takes that slot in the following iteration.  Every noise value comes from the request's seed (seeded.py), so
a request's result does not depend on its slot, on when it was admitted or on its neighbours: it is bit-identical to
the same request run alone through ddim_sample_loop / p_sample_loop with seeds=[seed].

    cs = diffusion.continuous_sampler(model_fn, slots=8, image_size=(256, 256), sampler="ddim")
    ticket = cs.submit(gt, gt_keep_mask, seed)     # queues; no device work, no synchronisation
    done = cs.step()                               # one iteration -> [(ticket, image [1, C, H, W])]
    results = cs.drain()                           # iterate until queue and slots are empty -> {ticket: image}

An iteration is [admissions] -> model evaluation -> one launch of the per-slot sampler step K8
(fidm_sampler_step_slots).  K8 takes each slot's action (idle, admit, update at t) and seed by value in its launch
parameters, so the schedule lives on the host (SlotSchedule, pure Python) and no iteration copies control data to the
device or synchronises.  With this package's InpaintingModelFn the evaluation is a CUDA-graph replay of the engine plan
whose state channels and timesteps K8 writes, and an iteration without admissions is [graph replay, K8].

diffusion.continuous_dpm_solver_sampler(...) has the same surface for dpm_solver_sample_loop: every request takes
`steps` evaluations on the DPM-Solver++ grid, each slot keeps its own history m_{k-1}, and the per-slot step is K9
(fidm_multistep_step_slots); each result equals dpm_solver_sample_loop run alone with seeds=[seed].

diffusion.continuous_repaint_sampler(...) does the same for repaint_sample_loop: every request takes the
len(repaint.evaluation_plan(...)) evaluations of RePaint's walk, the schedule counts them, and the per-slot step is K10
(fidm_repaint_step_slots): K8's DDPM update, K7's re-noising where a jump follows and the injection at the level the
walk goes on at, from per-evaluation tables built once; each result equals repaint_sample_loop run alone with
seeds=[seed].
"""
import collections
import ctypes as C
import os
from typing import NamedTuple

import torch

from . import _lib as L
from . import dpm_solver, repaint, seeded


def injection_draws(diffusion, schedule, cumulative, inject=True, grid=None):
    """The draw of the injection noise a seeded loop uses at each timestep it visits: t for cumulative noise, for fresh
    noise the number of injections before it; -1 where the loop does not inject (no injection, or t gated by
    `schedule`).  Without `grid`: indexed by t, the visits of ddim_sample_loop / p_sample_loop (T-1 .. 0).  With the
    DPM-Solver++ grid (dpm_solver.timestep_grid): indexed by grid point k, the visits of dpm_solver_sample_loop (x_T's
    injection at grid[0] counts as the first).  Any other list of visited timesteps, in loop order, works the same way
    (repaint_slot_tables)."""
    ts = range(diffusion.num_timesteps - 1, -1, -1) if grid is None else [int(t) for t in grid]
    draws, fresh = [], 0
    for t in ts:
        if inject and not diffusion._injection_gated(t, schedule):
            draws.append(t if cumulative else fresh)
            fresh += 1
        else:
            draws.append(-1)
    return draws[::-1] if grid is None else draws


def dpm_slot_tables(diffusion, grid, order, schedule, cumulative, inject=True):
    """K9's per-grid-point tables (fidm_ms_slot_args) as lists: the timestep value the model sees at t_k, the draw of
    the injection at t_k, and the order of the update out of t_k (dpm_solver.step_orders; 1 at the last point)."""
    return ([diffusion._t_value(int(t)) for t in grid], injection_draws(diffusion, schedule, cumulative, inject, grid),
            dpm_solver.step_orders(len(grid), order) + [1])


def repaint_slot_tables(diffusion, jump_length, jump_n_sample, schedule, cumulative):
    """K10's per-evaluation tables (fidm_rp_slot_args) as lists, from repaint.evaluation_plan: per evaluation k the
    timestep it updates (eval_t), the level of its injection and of the next evaluation (next_t: t_up when a jump
    follows, else t - 1; -1 after the last), the fp32 undo pair (a_u, s_u) (0 without a jump) and the draw of the
    injection at next_t (-1: none); then the draw of the admission's injection at T-1.  The injections are counted in
    repaint_sample_loop's order, x_T's at T-1 first, so fresh noise numbers them as that loop does and cumulative noise
    reuses (INJECT, t) at a revisited level."""
    plan = repaint.evaluation_plan(diffusion.alphas_cumprod, jump_length, jump_n_sample)
    eval_t = [e.t for e in plan]
    next_t = [e.t - 1 if e.t_up is None else e.t_up for e in plan]
    undo = [(e.undo_a, e.undo_s) for e in plan]
    draws = injection_draws(diffusion, schedule, cumulative, grid=[diffusion.num_timesteps - 1] + next_t[:-1])
    return eval_t, next_t, undo, draws[1:] + [-1], draws[0]


class SlotSchedule:
    """Which slot does what in each iteration.  FIFO admission into the lowest free slot; a slot evaluates its request
    at t = T-1 in the iteration it is admitted and at t - 1 in each following one, and is free again after t = 0.
    (For DPM-Solver++ slots T is the number of evaluations and t counts them down: grid point k = T-1-t.)"""

    def __init__(self, slots, num_timesteps):
        self.T = num_timesteps
        self.queue = collections.deque()
        self.t = [None] * slots             # per slot: the timestep of its next evaluation, None when free
        self.owner = [None] * slots         # per slot: the ticket it holds

    def push(self, ticket):
        self.queue.append(ticket)

    def busy(self):
        return sum(t is not None for t in self.t)

    def admit(self):
        """Fill free slots from the queue: [(slot, ticket)] in slot order."""
        out = []
        for b, t in enumerate(self.t):
            if not self.queue:
                break
            if t is None:
                self.t[b], self.owner[b] = self.T - 1, self.queue.popleft()
                out.append((b, self.owner[b]))
        return out

    def advance(self):
        """End of an iteration that evaluated every busy slot at self.t: [(slot, ticket)] of the requests finished."""
        done = []
        for b, t in enumerate(self.t):
            if t == 0:
                done.append((b, self.owner[b]))
                self.t[b] = self.owner[b] = None
            elif t is not None:
                self.t[b] = t - 1
        return done


class _Request(NamedTuple):
    ticket: int
    gt: torch.Tensor        # [1, C, H, W] fp32
    keep: torch.Tensor      # [1, 1 or C, H, W] fp32
    seed: int               # the uint64 seed


class ContinuousSampler:
    """See the module docstring; built by GaussianDiffusion.continuous_sampler.  `model` is called like the loops'
    model (model(x, t, gt=..., gt_keep_mask=...)), here on all slots at once with per-slot timesteps; it sees the keep
    masks as [slots, C, H, W].  With this package's InpaintingModelFn (and FIDM_FUSED_STEP != 0) the sampler uses the
    model's engine plan of batch `slots` and owns its inputs while it has work: a loop of the same batch and image
    size on the same model in between overwrites them."""

    def __init__(self, diffusion, model, slots=8, image_size=(256, 256), sampler="ddim", eta=0.0, clip_denoised=True,
                 use_inpainting_injection=True, injection_schedule="all", use_cumulative_noise=True, channels=3,
                 device=None, denoised_fn=None, cond_fn=None):
        if denoised_fn is not None or cond_fn is not None:
            raise ValueError("continuous batching runs the fused sampler step: denoised_fn / cond_fn are not supported")
        if sampler not in ("ddim", "ddpm"):
            hint = {"dpm_solver": " (DPM-Solver++: diffusion.continuous_dpm_solver_sampler)",
                    "repaint": " (RePaint: diffusion.continuous_repaint_sampler)"}.get(sampler, "")
            raise ValueError(f"sampler must be 'ddim' or 'ddpm', got {sampler!r}{hint}")
        T = diffusion.num_timesteps
        self._setup(diffusion, model, slots, image_size, injection_schedule, channels, device, T)
        ddim = sampler == "ddim"
        self._t_of = self._action_of = list(range(T))     # the schedule counts timesteps
        self._coef = diffusion._coef(self.device, eta if ddim else 0.0)
        self._t_value = torch.tensor([diffusion._t_value(t) for t in range(T)], dtype=torch.float32, device=self.device)
        self._inject_draw = torch.tensor(injection_draws(diffusion, injection_schedule, use_cumulative_noise,
                                                         use_inpainting_injection), dtype=torch.int32, device=self.device)

        from .gaussian_diffusion import _MEAN_CODE, _VAR_CODE
        a = self._args = L.StepArgs()
        a.batch, a.channels, a.hw = slots, channels, self.H * self.W
        a.mode = L.STEP_UPDATE_INJECT
        a.sampler = L.SAMPLER_DDIM if ddim else L.SAMPLER_DDPM
        a.mean_type, a.var_type = _MEAN_CODE[diffusion.model_mean_type], _VAR_CODE[diffusion.model_var_type]
        a.clip_denoised, a.cumulative = int(bool(clip_denoised)), int(bool(use_cumulative_noise))
        a.mask_channels, a.num_timesteps = channels, T
        a.coef, a.x, a.x_next, a.gt, a.keep_mask = (L.ptr(v) for v in (self._coef, self.x, self.x, self.gt, self.keep))
        self._set_stem(a)
        s = self._slot_args = L.SlotArgs()
        s.t_value, s.inject_draw, s.out = L.ptr(self._t_value), L.ptr(self._inject_draw), L.ptr(self.out)
        s.step_noise = int(not ddim or eta != 0.0)
        self._entry = "fidm_sampler_step_slots"

    def _setup(self, diffusion, model, slots, image_size, injection_schedule, channels, device, evaluations):
        """What every solver's sampler shares: the argument checks (before any device work), the slot buffers, the
        schedule of `evaluations` per request, the engine plan and the model's output channels."""
        if isinstance(slots, bool) or not isinstance(slots, int) or not 1 <= slots <= L.MAX_SLOTS:
            raise ValueError(f"slots must be an int in [1, {L.MAX_SLOTS}], got {slots!r}")
        if injection_schedule not in ("all", "high", "low"):
            raise ValueError(f"injection_schedule must be 'all', 'high' or 'low', got {injection_schedule!r}")
        if len(image_size) != 2 or any(isinstance(v, bool) or not isinstance(v, int) or v < 1 for v in image_size):
            raise ValueError(f"image_size must be (H, W) with positive ints, got {image_size!r}")
        if device is None:
            params = getattr(model, "parameters", None)
            device = next(params()).device if params is not None else torch.device("cuda", torch.cuda.current_device())
        device = torch.device(device)
        if device.type != "cuda":
            raise L.FidmError("fidm_b200 runs on sm_100a GPUs only; the continuous sampler needs a CUDA device "
                              "(no CPU fallback exists)")
        self.diffusion, self.model, self.device = diffusion, model, device
        self.B, self.C, (self.H, self.W) = slots, channels, image_size
        self.schedule = SlotSchedule(slots, evaluations)
        self._requests = {}
        self._next_ticket = 0

        shape = (slots, channels) + tuple(image_size)
        self.x = torch.zeros(shape, device=device)                 # slot states, updated in place by the step kernel
        self.gt = torch.zeros(shape, device=device)
        self.keep = torch.zeros(shape, device=device)
        self.out = torch.zeros(shape, device=device)               # the step kernel writes a finished sample here

        self.plan = None
        if getattr(model, "fused_plan", None) is not None and os.environ.get("FIDM_FUSED_STEP", "1") != "0":
            slot_plan = getattr(model, "slot_plan", None)
            self.plan = slot_plan(slots, channels, *image_size) if slot_plan is not None else None
        from .gaussian_diffusion import _VAR_CODE
        self._out_channels = channels if _VAR_CODE[diffusion.model_var_type] == L.VAR_FIXED else 2 * channels
        if self.plan is not None and self.plan.out.shape[1] != self._out_channels:
            raise ValueError(f"the model has {self.plan.out.shape[1]} output channels, the diffusion's variance type "
                             f"needs {self._out_channels}")

    def _set_stem(self, a):
        """With the engine plan the step kernel writes the next evaluation's state channels and timesteps into it."""
        if self.plan is not None:
            a.stem_out, a.stem_dtype, a.stem_ld = (L.ptr(self.plan.x_in), L.dtype_code(self.plan.x_in.dtype),
                                                   self.plan.x_in.shape[-1])
            a.t_out = L.ptr(self.plan.t_in)

    # ------------------------------------------------------------------ requests
    def submit(self, gt, gt_keep_mask, seed):
        """Queue one request: gt [C, H, W] or [1, C, H, W] and its keep mask (1 = known) with 1 or C channels, fp32 on
        the sampler's device, and its uint64 seed.  Returns the request's ticket.  The tensors are copied (on the
        stream, without synchronising): the caller may reuse them."""
        gt = self._image(gt, "gt", (self.C,))
        keep = self._image(gt_keep_mask, "gt_keep_mask", (1, self.C))
        seed = int(seeded.check_seeds([seed], 1)[0]) & ((1 << 64) - 1)
        ticket = self._next_ticket
        self._next_ticket += 1
        self._requests[ticket] = _Request(ticket, gt.clone(), keep.clone(), seed)
        self.schedule.push(ticket)
        return ticket

    def _image(self, t, name, channels):
        if not torch.is_tensor(t):
            raise ValueError(f"{name} must be a tensor, got {type(t)}")
        if t.dim() == 3:
            t = t.unsqueeze(0)
        if t.dim() != 4 or t.shape[0] != 1 or t.shape[1] not in channels or tuple(t.shape[2:]) != (self.H, self.W):
            want = " or ".join(f"[{c}, {self.H}, {self.W}]" for c in channels)
            raise ValueError(f"{name} must be {want} (optionally with a leading 1), got {tuple(t.shape)}")
        if t.device != self.device:
            raise ValueError(f"{name} is on {t.device}, the sampler on {self.device}")
        if t.dtype != torch.float32:
            raise ValueError(f"{name} must be float32, got {t.dtype}")
        return t.detach()

    def pending(self):
        """Requests queued or in a slot."""
        return len(self.schedule.queue) + self.schedule.busy()

    # ------------------------------------------------------------------ iterations
    def step(self):
        """One iteration: admit queued requests into free slots, evaluate every busy slot once, take one K8 (K9, K10) step.
        Returns [(ticket, image [1, C, H, W])] for the requests that finished; each image is a copy enqueued on the
        current stream, ready once the stream reaches it (the caller synchronises when it reads it)."""
        admitted = self.schedule.admit()
        with torch.no_grad():
            if admitted:
                for b, ticket in admitted:
                    self._load(b, self._requests[ticket])
                self._launch({b: L.SLOT_ADMIT for b, _ in admitted}, None)
            ts = list(self.schedule.t)
            if all(t is None for t in ts):
                return []
            model_out = self._evaluate(ts)
            self._launch({b: self._action_of[t] for b, t in enumerate(ts) if t is not None}, model_out)
            done = []
            for b, ticket in self.schedule.advance():
                del self._requests[ticket]
                done.append((ticket, self.out[b:b + 1].clone()))
        return done

    def drain(self):
        """step() until the queue and the slots are empty: {ticket: image}."""
        results = {}
        while self.pending():
            results.update(self.step())
        return results

    def _load(self, b, req):
        """Admission of `req` into slot b: its known region and seed, and with the engine plan its conditioning
        channels (the step kernel's admit action writes the state channels and the timestep)."""
        self.gt[b].copy_(req.gt[0])
        self.keep[b].copy_(req.keep[0].expand(self.C, self.H, self.W))
        self._slot_args.seeds[b] = req.seed
        if self.plan is not None:
            self.model.load_slot(self.plan, b, req.gt, req.keep)

    def _evaluate(self, ts):
        if self.plan is not None:
            return self.plan.run()                   # state channels and timesteps are already in place
        t = torch.tensor([0 if v is None else self._t_of[v] for v in ts], dtype=torch.long).to(self.device,
                                                                                                non_blocking=True)
        out = self.diffusion._call_model(self.model, self.x, t, {"gt": self.gt, "gt_keep_mask": self.keep})
        out = out.detach()
        if out.dtype != torch.float32 or not out.is_contiguous():
            out = out.to(torch.float32).contiguous()
        want = (self.B, self._out_channels, self.H, self.W)
        if tuple(out.shape) != want:
            raise ValueError(f"model output shape {tuple(out.shape)} != {want}")
        return out

    def _launch(self, actions, model_out):
        """One launch of the step kernel: slot b takes actions[b] (SLOT_ADMIT or its grid point: the timestep of a K8
        update, the k of a K9 or K10 one), every other slot idles."""
        s = self._slot_args
        for b in range(self.B):
            s.action[b] = actions.get(b, L.SLOT_IDLE)
        self._args.model_out = L.ptr(model_out)
        L.check(getattr(L.lib(), self._entry)(C.byref(self._args), C.byref(s), L.stream()), self._entry[5:])


class ContinuousDPMSolverSampler(ContinuousSampler):
    """ContinuousSampler for dpm_solver_sample_loop (built by GaussianDiffusion.continuous_dpm_solver_sampler): every
    request takes `steps` evaluations on dpm_solver.timestep_grid, each slot keeps its history m_{k-1} in `self.m`,
    and the per-slot step is K9 (fidm_multistep_step_slots) on K6's coefficient table."""

    def __init__(self, diffusion, model, slots=8, image_size=(256, 256), steps=20, order=2, clip_denoised=True,
                 use_inpainting_injection=True, injection_schedule="all", use_cumulative_noise=True, channels=3,
                 device=None):
        from .gaussian_diffusion import _MEAN_CODE, ModelMeanType
        grid = dpm_solver.timestep_grid(diffusion.num_timesteps, steps)
        tables = dpm_slot_tables(diffusion, grid, order, injection_schedule, use_cumulative_noise,
                                 use_inpainting_injection)
        if diffusion.model_mean_type == ModelMeanType.PREVIOUS_X:
            raise NotImplementedError("DPM-Solver++ needs an eps or x0 prediction; PREVIOUS_X models are not supported")
        self._setup(diffusion, model, slots, image_size, injection_schedule, channels, device, steps)
        # the schedule's counter c runs steps-1 .. 0: grid point k = steps-1-c
        self._t_of = [int(t) for t in grid[::-1]]
        self._action_of = list(range(steps - 1, -1, -1))
        dev = self.device
        self.m = torch.zeros_like(self.x)                          # per-slot history m_{k-1}, updated in place by K9
        self._coef = diffusion._dpm_table(dev, steps, order, use_cumulative_noise)
        self._t_value, self._inject_draw, self._order = (torch.tensor(v, dtype=dt, device=dev) for v, dt in
                                                         zip(tables, (torch.float32, torch.int32, torch.int32)))

        a = self._args = L.MultistepArgs()
        a.batch, a.channels, a.hw = slots, channels, self.H * self.W
        a.mean_type, a.out_channels = _MEAN_CODE[diffusion.model_mean_type], self._out_channels
        a.clip_denoised, a.mask_channels, a.steps = int(bool(clip_denoised)), channels, steps
        a.coef, a.x, a.x_next, a.m_prev, a.m_out, a.gt, a.keep_mask = (
            L.ptr(v) for v in (self._coef, self.x, self.x, self.m, self.m, self.gt, self.keep))
        self._set_stem(a)
        s = self._slot_args = L.MsSlotArgs()
        s.t_value, s.inject_draw, s.order, s.out = (L.ptr(v) for v in (self._t_value, self._inject_draw, self._order,
                                                                        self.out))
        s.inject_tag = L.NOISE_INJECT if use_cumulative_noise else L.NOISE_INJECT_FRESH
        # x_T's injection at t_0 = T-1 is the lockstep loop's K4 STEP_INJECT_ONLY: the K4 table's coefficients
        cls = diffusion.coefficient_table(0.0)
        ia, is_ = (L.C_SQRT_AB, L.C_SQRT_1MAB) if use_cumulative_noise else (L.C_SQRT_AB_F32, L.C_SQRT_1MAB_F32)
        s.admit_inject_a, s.admit_inject_s = float(cls[int(grid[0]), ia]), float(cls[int(grid[0]), is_])
        self._entry = "fidm_multistep_step_slots"


class ContinuousRePaintSampler(ContinuousSampler):
    """ContinuousSampler for repaint_sample_loop (built by GaussianDiffusion.continuous_repaint_sampler): every request
    takes the evaluations of repaint.evaluation_plan(jump_length, jump_n_sample), and the per-slot step is K10
    (fidm_repaint_step_slots) on K4's DDPM coefficient table and the per-evaluation tables of repaint_slot_tables."""

    def __init__(self, diffusion, model, slots=8, image_size=(256, 256), jump_length=10, jump_n_sample=10,
                 clip_denoised=True, use_inpainting_injection=True, injection_schedule="all", use_cumulative_noise=True,
                 channels=3, device=None):
        from .gaussian_diffusion import _MEAN_CODE, _VAR_CODE
        T = diffusion.num_timesteps
        repaint._check(T, jump_length, jump_n_sample)
        if not use_inpainting_injection:
            raise ValueError("RePaint resampling needs the known-region injection (use_inpainting_injection=True)")
        eval_t, next_t, undo, draws, admit_draw = repaint_slot_tables(diffusion, jump_length, jump_n_sample,
                                                                      injection_schedule, use_cumulative_noise)
        n = len(eval_t)
        self._setup(diffusion, model, slots, image_size, injection_schedule, channels, device, n)
        # the schedule's counter c runs n-1 .. 0: evaluation k = n-1-c
        self._t_of = eval_t[::-1]
        self._action_of = list(range(n - 1, -1, -1))
        dev = self.device
        self._coef = diffusion._coef(dev, 0.0)
        self._t_value = torch.tensor([diffusion._t_value(t) for t in range(T)], dtype=torch.float32, device=dev)
        self._eval_t, self._next_t, self._inject_draw = (torch.tensor(v, dtype=torch.int32, device=dev)
                                                         for v in (eval_t, next_t, draws))
        self._undo = torch.tensor(undo, dtype=torch.float32, device=dev)

        a = self._args = L.StepArgs()
        a.batch, a.channels, a.hw = slots, channels, self.H * self.W
        a.mode, a.sampler = L.STEP_UPDATE_INJECT, L.SAMPLER_DDPM
        a.mean_type, a.var_type = _MEAN_CODE[diffusion.model_mean_type], _VAR_CODE[diffusion.model_var_type]
        a.clip_denoised, a.cumulative = int(bool(clip_denoised)), int(bool(use_cumulative_noise))
        a.mask_channels, a.num_timesteps = channels, T
        a.coef, a.x, a.x_next, a.gt, a.keep_mask = (L.ptr(v) for v in (self._coef, self.x, self.x, self.gt, self.keep))
        self._set_stem(a)
        s = self._slot_args = L.RpSlotArgs()
        s.t_value, s.eval_t, s.next_t, s.undo, s.inject_draw, s.out = (
            L.ptr(v) for v in (self._t_value, self._eval_t, self._next_t, self._undo, self._inject_draw, self.out))
        s.n_evals, s.admit_draw = n, admit_draw
        self._entry = "fidm_repaint_step_slots"
