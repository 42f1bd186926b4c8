"""Multi-GPU use: intersections are independent units (main.py:230 creates exactly one scene and
scenes share nothing), so the batch is split into contiguous blocks, one process per GPU, with NO
collective on the step path.  The only exchange is the end-of-rollout reduction of the statistics
vector (`pve_counters`, 16 float64), an all-reduce(sum) over NCCL / NVLink."""
import torch
import torch.distributed as dist


def shard_range(n_total, rank, world):
    """Contiguous block [lo, hi) of intersections owned by ``rank`` (sizes differ by at most one).

    With device-generated arrivals a rank passes ``first_env=lo`` to ``BatchedScene.reset_poisson``: the stream is keyed
    by the global intersection index, so every intersection sees the same traffic however the batch is sharded.  With
    per-intersection or per-lane rates it passes its slice ``rates[lo:hi]`` of the whole batch's ``[n_total, lane_num]``
    rates as well (``pve_reset_poisson_rates``)."""
    base, rem = divmod(int(n_total), int(world))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def reduce_stats(counters, group=None):
    """Sum the per-GPU statistics vectors (``BatchedScene.stats_tensor()``) over all ranks."""
    out = counters.clone()
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(out, op=dist.ReduceOp.SUM, group=group)
    return out


def max_over_ranks(value, device, group=None):
    """Timing helper: the slowest rank defines the elapsed time."""
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return float(t.item())
