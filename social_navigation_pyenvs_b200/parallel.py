"""Multi-GPU plumbing (one process per GPU, torch.distributed): how the path shards.

* Independent environments (BASELINE configs 2-4) shard by env with NO data-path collective: rank r owns the contiguous block
  `env_shard(E, r, world)`; only timing / counters are reduced at the end.
* One very large crowd (config 5) shards by agent: rank r owns rows `agent_shard(N, r, world)` and every sub-step all-gathers the
  [5, N] entity view (x, y, vx, vy, r+safety) -- `all_gather_columns` -- over NCCL (NVLink/NVSwitch); gloo on CPU in the tests.
"""
import torch


def env_shard(E, rank, world):
    """Contiguous block of envs owned by `rank` (blocks differ by at most one env)."""
    base, rem = divmod(E, world)
    start = rank * base + min(rank, rem)
    return slice(start, start + base + (1 if rank < rem else 0))


def agent_shard(N, rank, world):
    """(offset, n_local) of the agent rows owned by `rank`; the crowd size must divide evenly so that the all-gather is regular."""
    if N % world:
        raise ValueError(f"crowd of {N} agents cannot be split evenly over {world} ranks")
    n_local = N // world
    return rank * n_local, n_local


def all_gather_columns(buf, offset, n_local, world, group=None):
    """buf [F, N_total] with this rank's columns [offset, offset + n_local) valid -> every rank's columns valid, in place."""
    if world == 1:
        return buf
    import torch.distributed as dist
    F = buf.shape[0]
    local = buf[:, offset:offset + n_local].contiguous()
    parts = torch.empty((world, F, n_local), dtype=buf.dtype, device=buf.device)
    if buf.is_cuda:
        dist.all_gather_into_tensor(parts, local, group=group)
    else:  # gloo has no all_gather_into_tensor
        dist.all_gather(list(parts.unbind(0)), local, group=group)
    buf.copy_(parts.permute(1, 0, 2).reshape(F, world * n_local))
    return buf


def all_gather_columns_packed(bufs, offset, n_local, world, group=None):
    """all_gather_columns for several buffers [F_i, N_total] of any dtypes in ONE collective: this rank's columns of every buffer
    travel as one byte string."""
    if world == 1:
        return bufs
    import torch.distributed as dist
    local = torch.cat([b[:, offset:offset + n_local].contiguous().view(torch.uint8).reshape(-1) for b in bufs])
    parts = torch.empty((world, local.numel()), dtype=torch.uint8, device=local.device)
    if local.is_cuda:
        dist.all_gather_into_tensor(parts, local, group=group)
    else:  # gloo has no all_gather_into_tensor
        dist.all_gather(list(parts.unbind(0)), local, group=group)
    for r in range(world):
        at = 0
        for b in bufs:
            nb = b.shape[0] * n_local * b.element_size()
            b[:, r * n_local:(r + 1) * n_local].copy_(parts[r, at:at + nb].view(b.dtype).view(b.shape[0], n_local))
            at += nb
    return bufs


def max_over_ranks(value, device, world, group=None):
    """Device-timed durations are reported as the max over ranks."""
    if world == 1:
        return float(value)
    import torch.distributed as dist
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())


def sum_over_ranks(value, device, world, group=None):
    if world == 1:
        return float(value)
    import torch.distributed as dist
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return float(t.item())
