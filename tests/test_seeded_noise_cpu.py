"""CPU: per-image seeded noise -- the Philox4x32-10 oracle against the Random123 known-answer vectors, the
fidm_seeded_noise struct against the header, the draw plan of every loop (run with recording stand-ins for the kernel
launchers) and the checks on `seeds`."""
import os
import re

import numpy as np
import pytest
import torch

import fidm_b200 as F
from fidm_b200 import _lib, seeded
from oracle import philox_oracle as P

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "fidm_b200.h")


@pytest.mark.parametrize("ctr,key,want", [
    ([0, 0, 0, 0], [0, 0], "6627e8d5 e169c58d bc57ac4c 9b00dbd8"),
    ([0xFFFFFFFF] * 4, [0xFFFFFFFF] * 2, "408f276d 41c83b0e a20bc7c6 6d5451fd"),
    ([0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344], [0xA4093822, 0x299F31D0], "d16cfe09 94fdcceb 5001e420 24126ea1"),
])
def test_oracle_reproduces_random123_known_answers(ctr, key, want):
    got = P.philox4x32_10(np.array(ctr), np.array(key))
    assert " ".join("%08x" % int(v) for v in got) == want


def test_oracle_layout_and_uniform():
    # element j takes lane j & 3 of group j >> 2: the first 6 elements of a 7-element image are those of an 8-element one
    assert np.array_equal(P.normals(3, 7, 2, 5), P.normals(3, 8, 2, 5)[:7])
    # the key is (seed lo, seed hi): seeds differing only in the high word differ
    assert not np.array_equal(P.normals(1, 8, 0, 0), P.normals(1 + (1 << 32), 8, 0, 0))
    u = P.uniform(np.array([0, 1, 0xFFFFFFFF], dtype=np.uint64))
    assert u[0] == 0.5 * 2.0 ** -32 and 0 < u[1] < 2.0 ** -31 and u[2] == 1.0
    assert np.sqrt(-2 * np.log(u[0])) > 6.6


def test_seeded_noise_struct_matches_header():
    text = open(HEADER).read()
    body = re.search(r"typedef struct fidm_seeded_noise \{(.*?)\} fidm_seeded_noise;", text, flags=re.S).group(1)
    body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
    names = []
    for decl in body.split(";"):
        decl = decl.strip()
        if not decl:
            continue
        decl = re.sub(r"^(const\s+)?(u?int32_t|u?int64_t|float|double|void)\s*\**", "", decl)
        for part in decl.split(","):
            names.append(re.sub(r"\[.*\]", "", part.replace("*", "").strip()))
    assert names == [f[0] for f in _lib.SeededNoise._fields_]
    for name in ("XT", "STEP", "INJECT", "INJECT_FRESH", "UNDO"):
        v = int(re.search(r"FIDM_NOISE_%s = (\d+)" % name, text).group(1))
        assert v == getattr(_lib, "NOISE_" + name) == P.TAGS[name]
    for sym in ("fidm_sampler_step_seeded", "fidm_multistep_step_seeded", "fidm_resample_undo_seeded",
                "fidm_randn_seeded"):
        assert sym in _lib.SYMBOLS


# ------------------------------------------------------------------------------------------ the draw plan
class _Recorder:
    """Stands in for the three kernel launchers of a diffusion and records every seeded draw they receive."""

    def __init__(self, d):
        self.draws = []
        d._step = self.step
        d._multistep = self.multistep
        d._resample = self.resample

    def _note(self, *noise):
        for n in noise:
            if n is not None:
                assert isinstance(n, seeded.Draw), type(n)
                self.draws.append((n.tag, n.draw))

    def step(self, mode, x, *, z=None, inject_noise=None, **kw):
        self._note(z, inject_noise)
        return {"sample": x, "pred_xstart": x, "x_next": x}

    def multistep(self, tab, step, x, model_out, *, inject_noise=None, **kw):
        self._note(inject_noise)
        return x, x

    def resample(self, x, u, undo_a, undo_s, *, inject_noise=None, **kw):
        self._note(u, inject_noise)
        return x


def _run(loop, monkeypatch, cumulative, eta=0.0, order=2, T=20, B=2):
    monkeypatch.setattr(_lib, "require_cuda", lambda *t: None)
    d = F.create_gaussian_diffusion(steps=T, learn_sigma=True, noise_schedule="cosine")
    rec = _Recorder(d)
    shape = (B, 3, 4, 4)
    mk = {"gt": torch.zeros(shape), "gt_keep_mask": torch.ones(B, 1, 4, 4)}
    kw = dict(noise=torch.zeros(shape), model_kwargs=mk, device="cpu", use_inpainting_injection=True,
              use_cumulative_noise=cumulative, seeds=[7, 2 ** 64 - 1])
    model = lambda x, t, **k: torch.zeros(B, 6, 4, 4)  # noqa: E731
    state = torch.get_rng_state()
    if loop == "ddim":
        d.ddim_sample_loop(model, shape, eta=eta, **kw)
    elif loop == "ddpm":
        d.p_sample_loop(model, shape, **kw)
    elif loop == "dpm_solver":
        d.dpm_solver_sample_loop(model, shape, steps=8, order=order, **kw)
    else:
        d.repaint_sample_loop(model, shape, jump_length=3, jump_n_sample=3, **kw)
    assert torch.equal(torch.get_rng_state(), state) and not d._gt_noises_cache
    return rec.draws, d


LOOPS = [("ddim", {}), ("ddim", {"eta": 0.5}), ("ddpm", {}), ("dpm_solver", {"order": 1}),
         ("dpm_solver", {"order": 2}), ("repaint", {})]


@pytest.mark.parametrize("loop,extra", LOOPS)
@pytest.mark.parametrize("cumulative", [True, False])
def test_draw_plan_never_reuses_a_draw(loop, extra, cumulative, monkeypatch):
    draws, d = _run(loop, monkeypatch, cumulative, **extra)
    T = d.num_timesteps
    inject = _lib.NOISE_INJECT if cumulative else _lib.NOISE_INJECT_FRESH
    injections = [x for tag, x in draws if tag == inject]
    steps = [x for tag, x in draws if tag == _lib.NOISE_STEP]
    undos = [x for tag, x in draws if tag == _lib.NOISE_UNDO]
    assert {tag for tag, _ in draws} <= {inject, _lib.NOISE_STEP, _lib.NOISE_UNDO}
    # only a cumulative injection draw may come twice, and only when RePaint revisits its timestep
    once = [dr for dr in draws if not (dr[0] == _lib.NOISE_INJECT and loop == "repaint")]
    assert len(set(once)) == len(once), loop
    if not cumulative:
        assert injections == list(range(len(injections)))           # the i-th fresh injection is draw i
    if loop == "repaint":
        assert cumulative is False or len(set(injections)) < len(injections)
        assert undos and len(set(undos)) == len(undos) and set(undos) < set(steps)
    else:
        assert not undos
    if loop in ("ddim", "ddpm"):
        if cumulative:
            assert injections == list(range(T - 1, -1, -1))         # x_T at T-1, then after every step but the last
        assert steps == ([] if loop == "ddim" and not extra else list(range(T)))
    if loop == "dpm_solver":
        assert not steps and len(injections) == 8                   # on x_T and after each of the 7 updates
    if loop == "repaint":
        assert steps == list(range(len(steps)))


# ------------------------------------------------------------------------------------------ checks on seeds
BAD_SEEDS = [[1], [1, 2, 3], [1, -1], [1, 2 ** 64], [1, 2.0], [1, True], "ab", 5,
             torch.tensor([1.0, 2.0]), torch.tensor([[1, 2]]), torch.tensor([1, -2]), torch.tensor([1, 2, 3])]


@pytest.mark.parametrize("loop", ["ddim", "ddpm", "dpm_solver", "repaint", "ddim_progressive", "repaint_progressive"])
@pytest.mark.parametrize("bad", range(len(BAD_SEEDS)))
def test_bad_seeds_raise_before_any_draw(loop, bad, monkeypatch):
    def no_draw(*a, **k):
        raise AssertionError("drew noise before checking seeds")

    for mod, name in ((torch, "randn"), (torch, "randn_like"), (seeded, "randn")):
        monkeypatch.setattr(mod, name, no_draw)
    d = F.create_gaussian_diffusion(steps=20, learn_sigma=True, noise_schedule="cosine")
    shape = (2, 3, 4, 4)
    mk = {"gt": torch.zeros(shape), "gt_keep_mask": torch.ones(2, 1, 4, 4)}
    model = lambda x, t, **k: torch.zeros(2, 6, 4, 4)  # noqa: E731
    kw = dict(model_kwargs=mk, device="cpu", use_inpainting_injection=True, seeds=BAD_SEEDS[bad])
    with pytest.raises(ValueError):
        if loop == "ddim":
            d.ddim_sample_loop(model, shape, **kw)
        elif loop == "ddpm":
            d.p_sample_loop(model, shape, **kw)
        elif loop == "dpm_solver":
            d.dpm_solver_sample_loop(model, shape, steps=5, **kw)
        elif loop == "repaint":
            d.repaint_sample_loop(model, shape, jump_length=2, jump_n_sample=2, **kw)
        elif loop == "ddim_progressive":
            next(d.ddim_sample_loop_progressive(model, shape, **kw))
        else:
            d.repaint_sample_loop_progressive(model, shape, jump_length=2, jump_n_sample=2, **kw)


def test_good_seeds_are_uint64_bit_patterns():
    assert seeded.check_seeds([0, 2 ** 63, 2 ** 64 - 1, np.uint64(5)], 4).tolist() == [0, -2 ** 63, -1, 5]
    assert seeded.check_seeds(torch.tensor([3, 4]), 2).tolist() == [3, 4]
    assert seeded.check_seeds(torch.tensor([2 ** 64 - 1, 1], dtype=torch.uint64), 2).tolist() == [-1, 1]


def test_seeds_with_denoised_fn_or_cond_fn_are_not_implemented():
    d = F.create_gaussian_diffusion(steps=20, noise_schedule="cosine")
    model = lambda x, t, **k: torch.zeros(1, 3, 4, 4)  # noqa: E731
    for kw in (dict(denoised_fn=lambda v: v), dict(cond_fn=lambda x, t, **k: x)):
        with pytest.raises(NotImplementedError):
            d.ddim_sample_loop(model, (1, 3, 4, 4), device="cpu", seeds=[1], **kw)
        with pytest.raises(NotImplementedError):
            d.p_sample_loop(model, (1, 3, 4, 4), device="cpu", seeds=[1], **kw)



def test_sample_sharded_passes_each_rank_its_slice_of_the_seeds(monkeypatch):
    import fidm_b200.parallel as par
    seen = {}

    class D:
        def p_sample_loop(self, model, shape, seeds=None, **kw):
            seen["seeds"] = seeded.check_seeds(seeds, shape[0]).tolist()
            return torch.zeros(shape)

        ddim_sample_loop = dpm_solver_sample_loop = repaint_sample_loop = p_sample_loop

    monkeypatch.setattr(par.dist, "is_initialized", lambda: True)
    monkeypatch.setattr(par.dist, "get_world_size", lambda: 2)
    monkeypatch.setattr(par, "gather_batch", lambda local, batch: local)
    state = torch.get_rng_state()
    for rank, want in ((0, [5, -3]), (1, [2 ** 63 - 1])):
        monkeypatch.setattr(par.dist, "get_rank", lambda rank=rank: rank)
        par.sample_sharded(D(), None, torch.zeros(3, 3, 4, 4), torch.ones(3, 1, 4, 4), sampler="ddpm",
                           seeds=[5, 2 ** 64 - 3, 2 ** 63 - 1])
        assert seen["seeds"] == want
    assert torch.equal(torch.get_rng_state(), state)                # seed + rank is not used with seeds
    with pytest.raises(ValueError):
        par.sample_sharded(D(), None, torch.zeros(3, 3, 4, 4), torch.ones(3, 1, 4, 4), sampler="ddpm", seeds=[1, 2])
