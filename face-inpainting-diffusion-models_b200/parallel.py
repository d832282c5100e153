"""Batch sharding across the GPUs of one box.

Every op on the sampling path is per-sample (GroupNorm is per (n, group), attention per (n, head),
injection per pixel), so the image batch is split into contiguous slices, one process per GPU, with
NO collective inside the reverse loop; a single all_gather returns the finished images
(SURVEY.md section 8-e).  Works with any initialised torch.distributed backend (NCCL on GPUs, gloo in
the CPU tests of the host logic).
"""
import torch
import torch.distributed as dist


def shard_bounds(batch, rank, world_size):
    """[start, stop) of `rank`'s contiguous slice; sizes differ by at most one."""
    base, rem = divmod(batch, world_size)
    start = rank * base + min(rank, rem)
    return start, start + base + (1 if rank < rem else 0)


def shard(t, rank=None, world_size=None, dim=0):
    rank = dist.get_rank() if rank is None else rank
    world_size = dist.get_world_size() if world_size is None else world_size
    a, b = shard_bounds(t.shape[dim], rank, world_size)
    return t.narrow(dim, a, b - a)


def gather_batch(local, batch):
    """all_gather of per-rank [b_r, ...] slices into the full [batch, ...] tensor (every rank)."""
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return local
    world = dist.get_world_size()
    sizes = [shard_bounds(batch, r, world) for r in range(world)]
    cap = max(b - a for a, b in sizes)
    pad = torch.zeros((cap,) + tuple(local.shape[1:]), dtype=local.dtype, device=local.device)
    pad[: local.shape[0]] = local
    bufs = [torch.empty_like(pad) for _ in range(world)]
    dist.all_gather(bufs, pad)
    return torch.cat([bufs[r][: b - a] for r, (a, b) in enumerate(sizes)], dim=0)


def sample_sharded(diffusion, model_fn, gt, gt_keep_mask, *, ddim=True, eta=0.0, seed=0, sampler=None, **loop_kwargs):
    """Run the inpainting loop on this rank's slice of (gt, gt_keep_mask) and gather the results.
    Per-rank generator seed = seed + rank (parity is checked shard by shard against the oracle).
    sampler: "ddim" | "ddpm" | "dpm_solver" | "repaint" (None: "ddim" if `ddim` else "ddpm"); `eta` is used by
    "ddim" only, and loop_kwargs go to the chosen loop (steps / order, jump_length / jump_n_sample, ...)."""
    if sampler is None:
        sampler = "ddim" if ddim else "ddpm"
    loops = {"ddim": diffusion.ddim_sample_loop, "ddpm": diffusion.p_sample_loop,
             "dpm_solver": diffusion.dpm_solver_sample_loop, "repaint": diffusion.repaint_sample_loop}
    if sampler not in loops:
        raise ValueError(f"sampler must be one of {sorted(loops)}, got {sampler!r}")
    rank = dist.get_rank() if dist.is_initialized() else 0
    world = dist.get_world_size() if dist.is_initialized() else 1
    if gt.shape[0] < world:
        # an empty shard would make its rank fail in the loop while the others wait in all_gather
        raise ValueError(f"batch {gt.shape[0]} < world size {world}: every rank needs at least one image")
    g, k = shard(gt, rank, world), shard(gt_keep_mask, rank, world)
    torch.manual_seed(seed + rank)
    if g.is_cuda:
        torch.cuda.manual_seed(seed + rank)
    extra = {"eta": eta} if sampler == "ddim" else {}
    out = loops[sampler](model_fn, tuple(g.shape), model_kwargs={"gt": g, "gt_keep_mask": k}, device=g.device,
                         use_inpainting_injection=True, **extra, **loop_kwargs)
    return gather_batch(out, gt.shape[0])
