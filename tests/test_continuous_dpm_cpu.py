"""CPU: continuous batching of the DPM-Solver++ loop -- the per-grid-point injection-draw, timestep and order tables
against the draw order of the seeded dpm_solver_sample_loop, the fidm_ms_slot_args struct against the header, and the
argument errors of the sampler."""
import ctypes
import os
import re

import pytest
import torch

import fidm_b200 as F
from fidm_b200 import _lib, dpm_solver, seeded
from fidm_b200.continuous import dpm_slot_tables, injection_draws

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "fidm_b200.h")


def _dpm_loop_draws(d, grid, schedule, cumulative):
    """The injections of _dpm_solver_loop with seeds, in its order: x_T's at grid[0] (_loop_start), then the one at
    grid[k + 1] after each update, each handed out by seeded.SeededDraws.  Returns the draw per grid point (-1: none)."""
    rng = seeded.SeededDraws(None, cumulative)
    want = [-1] * len(grid)
    for k, t in enumerate(int(v) for v in grid):
        if not d._injection_gated(t, schedule):
            dr = rng.inject(t)
            assert dr.tag == (_lib.NOISE_INJECT if cumulative else _lib.NOISE_INJECT_FRESH)
            want[k] = dr.draw
    return want


@pytest.mark.parametrize("schedule", ["all", "high", "low"])
@pytest.mark.parametrize("cumulative", [True, False])
@pytest.mark.parametrize("T,steps", [(20, 2), (20, 3), (20, 20), (1000, 2), (1000, 3), (1000, 20)])
def test_grid_injection_draws_follow_the_dpm_loop(schedule, cumulative, T, steps):
    d = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine")
    grid = dpm_solver.timestep_grid(T, steps)
    assert injection_draws(d, schedule, cumulative, grid=grid) == _dpm_loop_draws(d, grid, schedule, cumulative)
    assert injection_draws(d, schedule, cumulative, inject=False, grid=grid) == [-1] * steps


@pytest.mark.parametrize("schedule", ["all", "high", "low"])
@pytest.mark.parametrize("cumulative", [True, False])
def test_per_timestep_draws_are_unchanged(schedule, cumulative):
    """Without a grid the table is K8's: indexed by t, the same values as before the grid form existed."""
    T = 1000
    d = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine")
    want, fresh = [-1] * T, 0
    for t in range(T - 1, -1, -1):
        if not d._injection_gated(t, schedule):
            want[t] = t if cumulative else fresh
            fresh += 1
    assert injection_draws(d, schedule, cumulative) == want
    # the full grid visits every timestep in the same order: the same draws, indexed by k = T-1-t
    assert injection_draws(d, schedule, cumulative, grid=dpm_solver.timestep_grid(T, T)) == want[::-1]


@pytest.mark.parametrize("rescale", [False, True])
@pytest.mark.parametrize("T,steps,order", [(20, 2, 2), (20, 3, 2), (20, 20, 1), (1000, 20, 2), (1000, 25, 2)])
def test_slot_tables(T, steps, order, rescale):
    d = F.create_gaussian_diffusion(steps=T, noise_schedule="cosine", rescale_timesteps=rescale)
    grid = dpm_solver.timestep_grid(T, steps)
    t_value, draws, orders = dpm_slot_tables(d, grid, order, "low", False)
    assert t_value == [d._t_value(int(t)) for t in grid]
    assert draws == injection_draws(d, "low", False, grid=grid)
    assert orders == dpm_solver.step_orders(steps, order) + [1]
    assert orders[0] == 1 and orders[-2] == 1 and (order == 1 or steps < 4 or orders[1] == 2)


# ------------------------------------------------------------------------------------------ the C struct
def test_ms_slot_args_match_header():
    text = open(HEADER).read()
    body = re.search(r"typedef struct fidm_ms_slot_args \{(.*?)\} fidm_ms_slot_args;", text, flags=re.S).group(1)
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
    assert names == [f[0] for f in _lib.MsSlotArgs._fields_]
    assert arrays == {"action": "FIDM_MAX_SLOTS", "seeds": "FIDM_MAX_SLOTS"}
    fields = dict(_lib.MsSlotArgs._fields_)
    assert fields["action"]._length_ == fields["seeds"]._length_ == _lib.MAX_SLOTS
    assert fields["seeds"]._type_ is ctypes.c_uint64 and fields["action"]._type_ is ctypes.c_int32
    for name, ty in types.items():
        if ty == "ptr":
            assert fields[name] is ctypes.c_void_p, name
        elif ty == "float":
            assert fields[name] is ctypes.c_float, name
    # the launch parameters (fidm_multistep_args + fidm_ms_slot_args) stay inside the classic 4 KB limit
    assert ctypes.sizeof(_lib.MultistepArgs) + ctypes.sizeof(_lib.MsSlotArgs) <= 4096
    assert "fidm_multistep_step_slots" in _lib.SYMBOLS and "int fidm_multistep_step_slots(" in text


# ------------------------------------------------------------------------------------------ argument errors
BAD_CTOR = [(ValueError, dict(steps=1)), (ValueError, dict(steps=11)), (ValueError, dict(steps=4.0)),
            (ValueError, dict(steps=True)), (ValueError, dict(order=3)), (ValueError, dict(order=0)),
            (ValueError, dict(order=True)), (ValueError, dict(slots=0)), (ValueError, dict(slots=129)),
            (ValueError, dict(slots=2.0)), (ValueError, dict(injection_schedule="mid")),
            (ValueError, dict(image_size=(8,))), (ValueError, dict(image_size=(0, 8))),
            (NotImplementedError, dict(previous_x=True)), (_lib.FidmError, dict(device="cpu"))]


@pytest.mark.parametrize("bad", range(len(BAD_CTOR)))
def test_constructor_argument_errors(bad, monkeypatch):
    def no_device(*a, **k):
        raise AssertionError("touched the device before checking the arguments")

    monkeypatch.setattr(torch, "zeros", no_device)
    monkeypatch.setattr(torch, "tensor", no_device)
    monkeypatch.setattr(torch.cuda, "current_device", no_device)
    err, kw_bad = BAD_CTOR[bad]
    d = F.create_gaussian_diffusion(steps=10, noise_schedule="cosine")
    if kw_bad.pop("previous_x", False):
        d = F.GaussianDiffusion(betas=d.betas, model_mean_type=F.ModelMeanType.PREVIOUS_X,
                                model_var_type=F.ModelVarType.FIXED_LARGE, loss_type=F.LossType.MSE)
    kw = dict(slots=2, image_size=(8, 8), steps=4, device="cuda")
    kw.update(kw_bad)
    with pytest.raises(err):
        d.continuous_dpm_solver_sampler(lambda x, t, **k: x, **kw)


def test_continuous_sampler_points_at_the_dpm_entry():
    d = F.create_gaussian_diffusion(steps=10, noise_schedule="cosine")
    with pytest.raises(ValueError, match="continuous_dpm_solver_sampler"):
        d.continuous_sampler(lambda x, t, **k: x, slots=2, image_size=(8, 8), sampler="dpm_solver", device="cuda")
