"""Shared test helpers: seeded noise identical to oracle/make_golden.py, PSNR, torch.randn patching."""
import math

import torch

_REAL_RANDN = torch.randn


def seeded_noise(kind, t, shape, seed):
    g = torch.Generator().manual_seed(seed * 100003 + {"xT": 0, "inject": 1, "step": 2}[kind] * 50021 + int(t))
    return _REAL_RANDN(*shape, generator=g)


class PatchedRandn:
    """Route torch.randn / torch.randn_like to seeded_noise in the sampling loops' known draw order:
    randn(shape) once, then per step [inject noise], step noise (gaussian_diffusion.py:96-101,381,478)."""

    def __init__(self, T, seed, inject=True, device="cpu", first_draw=True):
        self.seq = [("xT", 0)] if first_draw else []
        for t in range(T - 1, -1, -1):
            if inject:
                self.seq.append(("inject", t))
            self.seq.append(("step", t))
        self.i, self.seed, self.device = 0, seed, device

    def _next(self, shape):
        kind, t = self.seq[self.i]
        self.i += 1
        return seeded_noise(kind, t, tuple(shape), self.seed).to(self.device)

    def __enter__(self):
        self._r, self._rl = torch.randn, torch.randn_like
        torch.randn = lambda *s, **k: self._next(s[0] if len(s) == 1 and not isinstance(s[0], int) else s)
        torch.randn_like = lambda x, **k: self._next(x.shape)
        return self

    def __exit__(self, *a):
        torch.randn, torch.randn_like = self._r, self._rl


def psnr(a, b, peak=2.0):
    mse = ((a.double() - b.double()) ** 2).mean().item()
    return 10 * math.log10(peak * peak / max(mse, 1e-30))


def rel_l2(a, b):
    return ((a.double() - b.double()).norm() / b.double().norm()).item()


class SeqRandn:
    """torch.randn / randn_like patched to an explicit [(kind, t), ...] draw sequence."""

    def __init__(self, seq, seed, device="cpu"):
        self.seq, self.i, self.seed, self.device = list(seq), 0, seed, device

    def _next(self, shape):
        kind, t = self.seq[self.i]
        self.i += 1
        return seeded_noise(kind, t, tuple(shape), self.seed).to(self.device)

    def __enter__(self):
        self._r, self._rl = torch.randn, torch.randn_like
        torch.randn = lambda *s, **k: self._next(s[0] if len(s) == 1 and not isinstance(s[0], int) else s)
        torch.randn_like = lambda x, **k: self._next(x.shape)
        return self

    def __exit__(self, *a):
        torch.randn, torch.randn_like = self._r, self._rl


def script_draw_order(seq, eta=0.0, ddpm=False):
    """RNG draw order of the evaluation scripts' loops (test_inp_ddim_100.py:402-576)."""
    order = [("xT", 0)]
    for t in seq:
        t = int(t)
        if ddpm or (t > 0 and eta > 0):
            order.append(("step", t))
        if t > 0:
            order.append(("inject", t))
    return order


def class_draw_order(T, inject=True, schedule="all", first=True):
    """RNG draw order of the class path's loops (gaussian_diffusion.py:96-101,146,381,428,478,521) with the
    high / low gating of :132-135 -- the same function oracle/make_golden_r2.py used."""
    seq = [("xT", 0)] if first else []
    for t in range(T - 1, -1, -1):
        gated = (schedule == "high" and t < T // 2) or (schedule == "low" and t >= T // 2)
        if inject and not gated:
            seq.append(("inject", t))
        seq.append(("step", t))
    return seq


def attention_shapes(cfg):
    """{(tokens, heads, head_dim)} of the attention layers of the UNet built from the constructor arguments `cfg`,
    each at the resolution the forward pass reaches it (arch.all_layers is in execution order)."""
    from fidm_b200.arch import all_layers, unet_topology
    res, shapes = cfg["image_size"], set()
    for layer in all_layers(unet_topology(**cfg)):
        if layer.kind == "attn":
            shapes.add((res * res, layer.heads, layer.channels // layer.heads))
        elif layer.kind == "down" or getattr(layer, "down", False):
            res //= 2
        elif layer.kind == "up" or getattr(layer, "up", False):
            res *= 2
    return shapes


def hole_psnr(a, b, keep):
    """PSNR over the inpainted (hole) pixels only: the known region is bit-exact by construction and would flatter
    a whole-image figure."""
    hole = (keep.expand_as(a) == 0)
    return psnr(a[hole], b[hole])
