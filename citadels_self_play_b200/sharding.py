"""How playouts and CFR roots are spread over ranks (one process per GPU).  Games are independent
(SURVEY.md 8(e)): rank r owns a contiguous block of global game ids per step; nothing is exchanged on the step
path.  The only collective is a sum of the outcome statistics (and a max of the times) after the timed region."""
import torch


def first_gid(step, rank, world, games_per_rank):
    """Global id of the first game rank `rank` plays in step `step`; blocks of different (step, rank) are disjoint."""
    return (step * world + rank) * games_per_rank


STAT_KEYS = ("games", "steps", "steps_sq", "errors")


def stats_to_tensor(stats, device="cpu"):
    v = [stats[k] for k in STAT_KEYS] + list(stats["wins"]) + list(stats["points_sum"]) + list(stats["points_sq"])
    return torch.tensor(v, dtype=torch.int64, device=device)


def tensor_to_stats(t):
    v = [int(x) for x in t.tolist()]
    d = dict(zip(STAT_KEYS, v[:4]))
    d["wins"], d["points_sum"], d["points_sq"] = v[4:10], v[10:16], v[16:22]
    return d


def reduce_stats(stats, device="cpu", group=None):
    """all_reduce(SUM) of the outcome statistics over `group` (default: the default process group; no-op for a single process)."""
    import torch.distributed as dist
    t = stats_to_tensor(stats, device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return tensor_to_stats(t)


def reduce_sum(values, device="cpu", group=None):
    """all_reduce(SUM) of integer counts over `group` (no-op for a single process)."""
    import torch.distributed as dist
    t = torch.tensor(list(values), dtype=torch.int64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM, group=group)
    return [int(x) for x in t.tolist()]


def reduce_max(values, device="cpu", group=None):
    import torch.distributed as dist
    t = torch.tensor(list(values), dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX, group=group)
    return [float(x) for x in t.tolist()]
