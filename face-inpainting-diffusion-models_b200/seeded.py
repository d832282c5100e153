"""Per-image seeded noise for the sampling loops.

With `seeds=` a loop takes every Gaussian value from a counter-based generator evaluated inside the sampler kernels
(Philox4x32-10 keyed by the image's own uint64 seed, csrc/philox.cuh), instead of torch's global generator.  An image's
noise is then a function of its seed and of the loop position only, so its result does not depend on the batch it is
sampled in, its position there, or the number of GPUs the batch is sharded over; and no noise tensor is drawn, stored
or cached.  Which draw a loop uses where (include/fidm_b200.h):

    x_T                                           (XT, 0)             unless `noise` is given
    step noise of the k-th model evaluation       (STEP, k)           DDIM eta = 0 and DPM-Solver++ draw none
    cumulative injection noise at timestep t      (INJECT, t)         RePaint revisits of t reuse it
    the i-th fresh injection of the loop          (INJECT_FRESH, i)   use_cumulative_noise=False
    RePaint undo noise after evaluation k         (UNDO, k)
"""
from typing import NamedTuple

import numpy as np
import torch

from . import _lib as L


class Draw(NamedTuple):
    """One seeded draw: the values a `_seeded` launch generates in place of a noise tensor."""
    seeds: torch.Tensor          # device int64 [batch]: the images' uint64 seeds, bit for bit
    tag: int
    draw: int


class SeededDraws:
    """The draws of one seeded loop, handed out in loop order (the counterpart of the torch-generator draws)."""

    def __init__(self, seeds, cumulative):
        self.seeds, self.cumulative, self.fresh = seeds, cumulative, 0

    def inject(self, t):
        if self.cumulative:
            return Draw(self.seeds, L.NOISE_INJECT, int(t))
        self.fresh += 1
        return Draw(self.seeds, L.NOISE_INJECT_FRESH, self.fresh - 1)

    def step(self, x, k):
        return Draw(self.seeds, L.NOISE_STEP, int(k))

    def undo(self, x, k):
        return Draw(self.seeds, L.NOISE_UNDO, int(k))


def check_seeds(seeds, batch):
    """`seeds` (B ints in [0, 2^64), or an int64 / uint64 tensor) as a CPU int64 tensor holding the uint64 bit patterns.
    ValueError for a wrong type, length or range."""
    if torch.is_tensor(seeds):
        if seeds.dtype not in (torch.int64, torch.uint64):
            raise ValueError(f"seeds must be an int64 or uint64 tensor, got {seeds.dtype}")
        if seeds.dim() != 1 or seeds.shape[0] != batch:
            raise ValueError(f"seeds must have shape ({batch},), got {tuple(seeds.shape)}")
        s = seeds.detach().cpu().contiguous()
        if s.dtype == torch.uint64:
            return s.view(torch.int64)
        if bool((s < 0).any()):
            raise ValueError("seeds must be in [0, 2**64); an int64 tensor holds no negative seed")
        return s
    if isinstance(seeds, (str, bytes)) or not hasattr(seeds, "__len__"):
        raise ValueError(f"seeds must be a sequence of {batch} ints or an int64 / uint64 tensor, got {type(seeds)}")
    if len(seeds) != batch:
        raise ValueError(f"seeds must hold one seed per image: {len(seeds)} for a batch of {batch}")
    vals = []
    for v in seeds:
        if isinstance(v, (bool, np.bool_)) or not isinstance(v, (int, np.integer)):
            raise ValueError(f"seeds must be ints, got {type(v)}")
        v = int(v)
        if not 0 <= v < 1 << 64:
            raise ValueError(f"seed {v} is outside [0, 2**64)")
        vals.append(v - (1 << 64) if v >= 1 << 63 else v)
    return torch.tensor(vals, dtype=torch.int64)


def randn(seeds, shape, tag, draw):
    """A new fp32 tensor of `shape` ([B, ...], contiguous) whose image b holds draw (tag, draw) under seeds[b]: the values
    the seeded sampler kernels generate for that draw.  `seeds`: a device int64 tensor from check_seeds."""
    L.require_cuda(seeds)
    B = shape[0]
    assert seeds.dtype == torch.int64 and tuple(seeds.shape) == (B,), (seeds.dtype, tuple(seeds.shape))
    out = torch.empty(tuple(shape), device=seeds.device, dtype=torch.float32)
    L.check(L.lib().fidm_randn_seeded(L.ptr(out), L.ptr(seeds.contiguous()), B, out.numel() // B, int(tag), int(draw),
                                      L.stream()), "randn_seeded")
    return out


def launch_args(noise, inject):
    """The fidm_seeded_noise of a sampler launch whose step / undo noise is `noise` and injection noise `inject` (each
    None when the launch has none), or None when neither is a Draw: the launch reads noise tensors."""
    draws = [d for d in (noise, inject) if isinstance(d, Draw)]
    if not draws:
        return None
    assert len(draws) == sum(d is not None for d in (noise, inject)), "seeded and tensor noise in one launch"
    s = L.SeededNoise()
    s.seeds = L.ptr(draws[0].seeds)
    s.draw = -1 if noise is None else noise.draw
    if inject is not None:
        s.inject_tag, s.inject_draw = inject.tag, inject.draw
    return s
