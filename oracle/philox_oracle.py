"""Restatement of the per-image seeded noise of csrc/philox.cuh in numpy, from the specification:

  Philox4x32-10 (Salmon, Moraes, Dror, Shaw 2011): multipliers 0xD2511F53 / 0xCD9E8D57, key increments
  0x9E3779B9 / 0xBB67AE85, 10 rounds.
  key      = (seed & 0xffffffff, seed >> 32)
  counter  = (q, draw, tag, 0), q = j >> 2, j = c*hw + p the flat NCHW index of the element within its image
  normals  = Box-Muller on (w0, w1) -> lanes 0, 1 and (w2, w3) -> lanes 2, 3; element j takes lane j & 3
  u        = (w + 0.5) * 2^-32 formed in fp32 as the kernels form it (w rounded to fp32, + 0.5 rounded), never 0;
             r = sqrt(-2 ln u1), theta = 2 pi u2, computed here in float64.

Integer arithmetic is numpy uint64 reduced mod 2^32, so the words are exact; the normals agree with the kernels' fp32
values to their rounding (a few ulp of |n|)."""
import numpy as np

M0, M1 = 0xD2511F53, 0xCD9E8D57
W0, W1 = 0x9E3779B9, 0xBB67AE85
MASK = 0xFFFFFFFF
TAGS = {"XT": 0, "STEP": 1, "INJECT": 2, "INJECT_FRESH": 3, "UNDO": 4}


def philox4x32_10(ctr, key):
    """ctr: [..., 4], key: [..., 2] unsigned ints -> [..., 4] uint64 words (each < 2^32)."""
    c = [np.asarray(ctr, dtype=np.uint64)[..., i] & MASK for i in range(4)]
    k0, k1 = (np.asarray(key, dtype=np.uint64)[..., i] & MASK for i in range(2))
    for r in range(10):
        if r > 0:
            k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
        p0, p1 = c[0] * np.uint64(M0), c[2] * np.uint64(M1)          # < 2^64: exact in uint64
        hi0, lo0 = p0 >> np.uint64(32), p0 & MASK
        hi1, lo1 = p1 >> np.uint64(32), p1 & MASK
        c = [hi1 ^ c[1] ^ k0, lo1, hi0 ^ c[3] ^ k1, lo0]
    return np.stack(c, axis=-1)


def uniform(w):
    """The kernels' u = fl32(fl32(w) + 0.5) * 2^-32, in (0, 1], as float64."""
    return (np.asarray(w, dtype=np.float64).astype(np.float32) + np.float32(0.5)).astype(np.float64) * 2.0 ** -32


def normals(seed, n, tag, draw):
    """The n normals (float64) of elements j = 0 .. n-1 of one image under `seed`, draw (tag, draw)."""
    seed = int(seed) & ((1 << 64) - 1)
    q = np.arange((n + 3) // 4, dtype=np.uint64)
    ctr = np.stack([q, np.full_like(q, draw), np.full_like(q, tag), np.zeros_like(q)], axis=-1)
    key = np.array([seed & MASK, seed >> 32], dtype=np.uint64)
    w = philox4x32_10(ctr, np.broadcast_to(key, (len(q), 2)))
    out = np.empty((len(q), 4))
    for pair in (0, 1):
        r = np.sqrt(-2.0 * np.log(uniform(w[:, 2 * pair])))
        th = 2.0 * np.pi * uniform(w[:, 2 * pair + 1])
        out[:, 2 * pair], out[:, 2 * pair + 1] = r * np.cos(th), r * np.sin(th)
    return out.reshape(-1)[:n]


def randn(seeds, shape, tag, draw):
    """[B, ...] float64: image b holds normals(seeds[b], prod(shape[1:]), tag, draw) in NCHW order."""
    n = int(np.prod(shape[1:]))
    return np.stack([normals(s, n, tag, draw) for s in seeds]).reshape(shape)
