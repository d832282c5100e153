"""CPU: continuous batching -- the slot schedule, the per-timestep injection-draw table against the draw order of the
plain seeded loops, the fidm_slot_args struct against the header, and the argument errors of the sampler."""
import os
import random
import re

import pytest
import torch

import fidm_b200 as F
from fidm_b200 import _lib, seeded
from fidm_b200.continuous import SlotSchedule, injection_draws
from helpers import class_draw_order

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "fidm_b200.h")


# ------------------------------------------------------------------------------------------ the schedule
def _drive(slots, T, arrivals, iters):
    """Run a schedule: arrivals[i] requests are pushed before iteration i.  Returns the per-iteration log
    [(admitted, {slot: t evaluated}, finished)] and the tickets pushed."""
    s = SlotSchedule(slots, T)
    log, ticket = [], 0
    for i in range(iters):
        for _ in range(arrivals[i] if i < len(arrivals) else 0):
            s.push(ticket)
            ticket += 1
        admitted = s.admit()
        evals = {b: (s.owner[b], t) for b, t in enumerate(s.t) if t is not None}
        # no idle slot while the queue is non-empty
        assert not s.queue or s.busy() == slots
        finished = s.advance()
        log.append((admitted, evals, finished))
    return log, ticket


@pytest.mark.parametrize("slots,T,seed", [(1, 3, 0), (3, 5, 1), (4, 1, 2), (8, 20, 3)])
def test_schedule_fifo_full_and_exactly_T_evaluations(slots, T, seed):
    rng = random.Random(seed)
    arrivals = [rng.choice([0, 0, 1, 2, 5]) for _ in range(40)]
    log, n = _drive(slots, T, arrivals, 40 + (n_max := sum(arrivals)) * T)
    per_ticket = {k: [] for k in range(n)}
    admit_order, finish_iter = [], {}
    for i, (admitted, evals, finished) in enumerate(log):
        free_before = [b for b in range(slots) if all(b != e for e in evals) or b in dict(admitted)]
        for b, ticket in admitted:
            admit_order.append(ticket)
            assert evals[b] == (ticket, T - 1)
        # admission goes to the lowest free slots
        assert [b for b, _ in admitted] == sorted(b for b, _ in admitted)
        assert all(b in free_before for b, _ in admitted)
        for b, (ticket, t) in evals.items():
            per_ticket[ticket].append((i, b, t))
        for b, ticket in finished:
            finish_iter[ticket] = (i, b)
    assert n == n_max and admit_order == list(range(n))                     # FIFO, everything served
    for ticket, ev in per_ticket.items():
        assert [t for _, _, t in ev] == list(range(T - 1, -1, -1)), ticket   # exactly T evaluations, descending t
        assert len({b for _, b, _ in ev}) == 1                               # never moves
        assert [i for i, _, _ in ev] == list(range(ev[0][0], ev[0][0] + T))  # consecutive iterations
        assert finish_iter[ticket] == (ev[-1][0], ev[-1][1])


def test_schedule_lowest_free_slot():
    s = SlotSchedule(3, 2)
    for k in range(3):
        s.push(k)
    assert s.admit() == [(0, 0), (1, 1), (2, 2)]
    s.t[1] = 0                                   # slot 1 finishes first
    assert s.advance() == [(1, 1)]
    s.push(3)
    s.push(4)
    assert s.admit() == [(1, 3)] and list(s.queue) == [4]


def test_schedule_finish_then_admit_in_the_next_iteration():
    log, _ = _drive(2, 3, [3], 7)
    assert [a for a, _, _ in log] == [[(0, 0), (1, 1)], [], [], [(0, 2)], [], [], []]
    assert [f for _, _, f in log] == [[], [], [(0, 0), (1, 1)], [], [], [(0, 2)], []]
    assert log[3][1] == {0: (2, 2)} and log[6][1] == {}


# ------------------------------------------------------------------------------------------ the injection-draw table
@pytest.mark.parametrize("schedule", ["all", "high", "low"])
@pytest.mark.parametrize("cumulative", [True, False])
@pytest.mark.parametrize("T", [2, 7, 20])
def test_injection_draws_follow_the_plain_loop(schedule, cumulative, T):
    d = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine")
    table = injection_draws(d, schedule, cumulative)
    # the plain loop's injections, in draw order (helpers.class_draw_order), handed out by the seeded draws
    rng = seeded.SeededDraws(None, cumulative)
    want = [-1] * T
    for kind, t in class_draw_order(T, inject=True, schedule=schedule):
        if kind == "inject":
            dr = rng.inject(t)
            assert dr.tag == (_lib.NOISE_INJECT if cumulative else _lib.NOISE_INJECT_FRESH)
            want[t] = dr.draw
    assert table == want
    assert injection_draws(d, schedule, cumulative, inject=False) == [-1] * T


# ------------------------------------------------------------------------------------------ the C struct
def test_slot_args_match_header():
    text = open(HEADER).read()
    body = re.search(r"typedef struct fidm_slot_args \{(.*?)\} fidm_slot_args;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names, arrays = [], {}
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        decl = re.sub(r"^(const\s+)?(u?int32_t|u?int64_t|float|double|void)\s*\**", "", decl)
        for part in decl.split(","):
            part = part.replace("*", "").strip()
            m = re.match(r"(\w+)\[(\w+)\]", part)
            if m:
                arrays[m.group(1)] = m.group(2)
            names.append(re.sub(r"\[.*\]", "", part))
    assert names == [f[0] for f in _lib.SlotArgs._fields_]
    assert arrays == {"action": "FIDM_MAX_SLOTS", "seeds": "FIDM_MAX_SLOTS"}
    max_slots = int(re.search(r"#define FIDM_MAX_SLOTS (\d+)", text).group(1))
    assert max_slots == _lib.MAX_SLOTS == 128
    fields = dict(_lib.SlotArgs._fields_)
    assert fields["action"]._length_ == fields["seeds"]._length_ == max_slots
    assert fields["seeds"]._type_ is __import__("ctypes").c_uint64
    assert int(re.search(r"FIDM_SLOT_IDLE = (-\d+)", text).group(1)) == _lib.SLOT_IDLE
    assert int(re.search(r"FIDM_SLOT_ADMIT = (-\d+)", text).group(1)) == _lib.SLOT_ADMIT
    # the launch parameters (fidm_step_args + fidm_slot_args) stay inside the classic 4 KB kernel-parameter limit
    import ctypes
    assert ctypes.sizeof(_lib.StepArgs) + ctypes.sizeof(_lib.SlotArgs) <= 4096
    assert "fidm_sampler_step_slots" in _lib.SYMBOLS and "fidm_sampler_step_slots" in text


# ------------------------------------------------------------------------------------------ argument errors
BAD_CTOR = [dict(slots=0), dict(slots=129), dict(slots=2.0), dict(slots=True), dict(sampler="dpm_solver"),
            dict(sampler="repaint"), dict(denoised_fn=lambda v: v), dict(cond_fn=lambda x, t, **k: x),
            dict(injection_schedule="mid"), dict(image_size=(8,)), dict(image_size=(0, 8))]


@pytest.mark.parametrize("bad", range(len(BAD_CTOR)))
def test_constructor_argument_errors(bad, monkeypatch):
    def no_device(*a, **k):
        raise AssertionError("touched the device before checking the arguments")

    monkeypatch.setattr(torch, "zeros", no_device)
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    d = F.create_gaussian_diffusion(steps=10, noise_schedule="cosine")
    kw = dict(slots=2, image_size=(8, 8), device="cuda")
    kw.update(BAD_CTOR[bad])
    with pytest.raises(ValueError):
        d.continuous_sampler(lambda x, t, **k: x, **kw)


def test_cpu_device_is_refused():
    d = F.create_gaussian_diffusion(steps=10, noise_schedule="cosine")
    with pytest.raises(_lib.FidmError):
        d.continuous_sampler(lambda x, t, **k: x, slots=2, image_size=(8, 8), device="cpu")
