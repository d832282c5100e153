"""Seeded element subsets of large golden arrays.

Every file under tests/golden stays below 1 MB: a large reference output is stored as its elements at a fixed, sorted,
seeded index set, saved next to it as `sub_idx`.  Tests apply the same index to what they compute (`take`) and keep their
bars: PSNR and rel-L2 over tens of thousands of elements, exact equality element by element.
"""
import torch


def subset_index(numel, keep, seed=0):
    """`keep` distinct flat indices in [0, numel), sorted (int32)."""
    return torch.randperm(numel, generator=torch.Generator().manual_seed(seed))[:keep].sort().values.int()


def take(t, idx, per_image=False):
    """The elements of `t` at `idx`: over the whole flattened tensor, or per leading image ([N, len(idx)])."""
    idx = idx.long().to(t.device)
    return t.reshape(t.shape[0], -1)[:, idx] if per_image else t.reshape(-1)[idx]


def shrink(entry, keys, keep, per_image=False):
    """`entry` with each array in `keys` (all of one shape) replaced by its subset; the index is added as `sub_idx` and the
    arrays' full shape as `shape`."""
    ref = entry[keys[0]]
    numel = ref[0].numel() if per_image else ref.numel()
    idx = subset_index(numel, keep)
    out = dict(entry, sub_idx=idx, shape=tuple(ref.shape))
    for k in keys:
        assert entry[k].shape == ref.shape, k
        out[k] = take(entry[k], idx, per_image).clone()
    return out
