"""CPU: continuous batching of the RePaint loop -- the per-evaluation tables of K10 against the draw order of the
seeded repaint_sample_loop, their reduction to K8's per-timestep draws without jumps, the fidm_rp_slot_args struct
against the header, and the argument errors of the sampler."""
import ctypes
import os
import re

import pytest
import torch

import fidm_b200 as F
from fidm_b200 import _lib, repaint, seeded
from fidm_b200.continuous import injection_draws, repaint_slot_tables

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "fidm_b200.h")


class _Recorder(seeded.SeededDraws):
    """seeded.SeededDraws that records every draw it hands out, in order."""

    def __init__(self, cumulative):
        super().__init__(None, cumulative)
        self.calls = []

    def inject(self, t):
        d = super().inject(t)
        self.calls.append(("inject", int(t), d))
        return d

    def step(self, x, k):
        d = super().step(x, k)
        self.calls.append(("step", int(k), d))
        return d

    def undo(self, x, k):
        d = super().undo(x, k)
        self.calls.append(("undo", int(k), d))
        return d


def _repaint_loop_tables(d, jl, jn, schedule, cumulative):
    """A restatement of _repaint_loop's draws with seeds (_loop_start, then per evaluation the step noise, the undo noise
    when a jump follows and the injection of the next evaluation, each skipped where _repaint_loop skips it), recorded
    in loop order.  Returns K10's tables (eval_t, next_t, undo, inject_draw, admit_draw) read off the record."""
    rng = _Recorder(cumulative)
    T = d.num_timesteps
    plan = repaint.evaluation_plan(d.alphas_cumprod, jl, jn)
    admit = rng.inject(T - 1).draw if not d._injection_gated(T - 1, schedule) else -1
    eval_t, next_t, undo, draws = [], [], [], []
    for k, (i, t_up, ua, us) in enumerate(plan):
        n0 = len(rng.calls)
        rng.step(None, k)
        if t_up is None:
            nxt = i - 1
            if nxt >= 0 and not d._injection_gated(nxt, schedule):
                rng.inject(nxt)
        else:
            nxt = t_up
            rng.undo(None, k)
            if not d._injection_gated(t_up, schedule):
                rng.inject(t_up)
        calls = rng.calls[n0:]
        assert calls[0][0] == "step" and calls[0][2].tag == _lib.NOISE_STEP and calls[0][2].draw == k
        if t_up is not None:
            assert calls[1][0] == "undo" and calls[1][2].tag == _lib.NOISE_UNDO and calls[1][2].draw == k
        inj = [c for c in calls if c[0] == "inject"]
        assert len(inj) <= 1 and all(c[1] == nxt for c in inj)
        for c in inj:
            assert c[2].tag == (_lib.NOISE_INJECT if cumulative else _lib.NOISE_INJECT_FRESH)
        eval_t.append(i)
        next_t.append(nxt)
        undo.append((ua, us))
        draws.append(inj[0][2].draw if inj else -1)
    return eval_t, next_t, undo, draws, admit


CASES = [(10, 3, 3), (10, 1, 4), (12, 5, 2), (20, 4, 3), (20, 19, 2), (20, 3, 1), (50, 5, 3), (100, 10, 10)]


@pytest.mark.parametrize("schedule", ["all", "high", "low"])
@pytest.mark.parametrize("cumulative", [True, False])
@pytest.mark.parametrize("T,jl,jn", CASES)
def test_tables_follow_the_repaint_loop(T, jl, jn, schedule, cumulative):
    d = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine")
    got = repaint_slot_tables(d, jl, jn, schedule, cumulative)
    assert got == _repaint_loop_tables(d, jl, jn, schedule, cumulative)
    eval_t, next_t, undo, draws, admit = got
    plan = repaint.evaluation_plan(d.alphas_cumprod, jl, jn)
    assert len(eval_t) == len(plan) and eval_t[0] == T - 1
    # the walk: evaluation k+1 is at next_t[k]; the last is t = 0 with nothing after it, and t = 0 is visited once
    assert eval_t[1:] == next_t[:-1] and eval_t[-1] == 0 and next_t[-1] == -1 and eval_t.count(0) == 1
    for (t, nt, (ua, us)) in zip(eval_t, next_t, undo):
        assert (nt == t - 1) == (ua == 0.0 and us == 0.0)
        assert nt == t - 1 or nt >= t
    if cumulative:
        assert all(dr in (-1, nt) for dr, nt in zip(draws, next_t))
        assert admit in (-1, T - 1)
    else:                       # fresh: the ungated injections numbered 0, 1, ... in loop order, the admission's first
        used = [dr for dr in [admit] + draws if dr >= 0]
        assert used == list(range(len(used)))


@pytest.mark.parametrize("schedule", ["all", "high", "low"])
@pytest.mark.parametrize("cumulative", [True, False])
@pytest.mark.parametrize("T,jl", [(10, 3), (20, 1), (100, 10)])
def test_without_jumps_the_tables_are_k8s(T, jl, schedule, cumulative):
    """jump_n_sample = 1: the walk is the plain DDPM loop, and the draws are K8's per-timestep ones."""
    d = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine")
    eval_t, next_t, undo, draws, admit = repaint_slot_tables(d, jl, 1, schedule, cumulative)
    k8 = injection_draws(d, schedule, cumulative)
    assert eval_t == list(range(T - 1, -1, -1)) and next_t == [t - 1 for t in eval_t]
    assert undo == [(0.0, 0.0)] * T
    assert draws == [k8[t - 1] if t >= 1 else -1 for t in eval_t]
    assert admit == k8[T - 1]


# ------------------------------------------------------------------------------------------ the C struct
def test_rp_slot_args_match_header():
    text = open(HEADER).read()
    body = re.search(r"typedef struct fidm_rp_slot_args \{(.*?)\} fidm_rp_slot_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names, arrays, types = [], {}, {}
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        ty = re.match(r"^(const\s+)?(u?int32_t|u?int64_t|float|double|void)\s*(\**)", decl)
        decl = decl[ty.end():]
        for part in decl.split(","):
            part = part.replace("*", "").strip()
            m = re.match(r"(\w+)\[(\w+)\]", part)
            if m:
                arrays[m.group(1)] = m.group(2)
            name = re.sub(r"\[.*\]", "", part)
            names.append(name)
            types[name] = "ptr" if ty.group(3) else ty.group(2)
    assert names == [f[0] for f in _lib.RpSlotArgs._fields_]
    assert arrays == {"action": "FIDM_MAX_SLOTS", "seeds": "FIDM_MAX_SLOTS"}
    fields = dict(_lib.RpSlotArgs._fields_)
    assert fields["action"]._length_ == fields["seeds"]._length_ == _lib.MAX_SLOTS
    assert fields["seeds"]._type_ is ctypes.c_uint64 and fields["action"]._type_ is ctypes.c_int32
    for name, ty in types.items():
        if ty == "ptr":
            assert fields[name] is ctypes.c_void_p, name
        elif ty == "int32_t" and name not in arrays:
            assert fields[name] is ctypes.c_int32, name
    # the launch parameters (fidm_step_args + fidm_rp_slot_args) stay inside the classic 4 KB limit
    assert ctypes.sizeof(_lib.StepArgs) + ctypes.sizeof(_lib.RpSlotArgs) <= 4096
    assert "fidm_repaint_step_slots" in _lib.SYMBOLS and "int fidm_repaint_step_slots(" in text
    assert _lib.SYMBOLS["fidm_repaint_step_slots"][1][:2] == [ctypes.POINTER(_lib.StepArgs),
                                                              ctypes.POINTER(_lib.RpSlotArgs)]


# ------------------------------------------------------------------------------------------ argument errors
BAD_CTOR = [(ValueError, dict(jump_length=0)), (ValueError, dict(jump_length=10)), (ValueError, dict(jump_length=True)),
            (ValueError, dict(jump_length=2.0)), (ValueError, dict(jump_n_sample=0)),
            (ValueError, dict(jump_n_sample=True)), (ValueError, dict(jump_n_sample=None)),
            (ValueError, dict(use_inpainting_injection=False)), (ValueError, dict(slots=0)),
            (ValueError, dict(slots=129)), (ValueError, dict(slots=2.0)), (ValueError, dict(injection_schedule="mid")),
            (ValueError, dict(image_size=(8,))), (ValueError, dict(image_size=(0, 8))),
            (_lib.FidmError, dict(device="cpu"))]


@pytest.mark.parametrize("bad", range(len(BAD_CTOR)))
def test_constructor_argument_errors(bad, monkeypatch):
    def no_device(*a, **k):
        raise AssertionError("touched the device before checking the arguments")

    monkeypatch.setattr(torch, "zeros", no_device)
    monkeypatch.setattr(torch, "tensor", no_device)
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    err, kw_bad = BAD_CTOR[bad]
    d = F.create_gaussian_diffusion(steps=10, noise_schedule="cosine")
    kw = dict(slots=2, image_size=(8, 8), jump_length=3, jump_n_sample=3, device="cuda")
    kw.update(kw_bad)
    with pytest.raises(err):
        d.continuous_repaint_sampler(lambda x, t, **k: x, **kw)


def test_cpu_device_is_refused():
    d = F.create_gaussian_diffusion(steps=10, noise_schedule="cosine")
    with pytest.raises(_lib.FidmError):
        d.continuous_repaint_sampler(lambda x, t, **k: x, slots=2, image_size=(8, 8), jump_length=3, device="cpu")


def test_continuous_sampler_points_at_the_repaint_entry():
    d = F.create_gaussian_diffusion(steps=10, noise_schedule="cosine")
    with pytest.raises(ValueError, match="continuous_repaint_sampler"):
        d.continuous_sampler(lambda x, t, **k: x, slots=2, image_size=(8, 8), sampler="repaint", device="cuda")
