"""Multi-GPU host logic: games are independent units, so ranks never exchange data on the self-play path
(SURVEY.md 8e).  This module only (1) partitions game ids / seeds across ranks and (2) reduces the
per-rank measurements for reporting (max of times, sum of work) -- through torch.distributed with
whatever backend the caller initialised (NCCL on GPUs, gloo in the CPU tests)."""
from __future__ import annotations

import torch


def shard_games(total_games: int, world: int, rank: int) -> tuple[int, int]:
    """Contiguous partition of `total_games` over `world` ranks: (first game id, count) of `rank`."""
    base, extra = divmod(total_games, world)
    count = base + (1 if rank < extra else 0)
    start = rank * base + min(rank, extra)
    return start, count


def rank_seed(base_seed: int, rank: int) -> int:
    """Distinct random-stream seed per rank (streams inside a context are keyed by tree id)."""
    return (base_seed + 0x9E3779B97F4A7C15 * (rank + 1)) & 0xFFFFFFFFFFFFFFFF


def iteration_seed(seed: int, iteration: int) -> int:
    """The context seed of iteration `iteration` of a run whose previous iteration's context had `seed` (splitmix64's
    finaliser of seed ^ iteration * K: for a given iteration, distinct seeds stay distinct, so the ranks keep distinct
    streams)."""
    m = 0xFFFFFFFFFFFFFFFF
    z = (seed ^ (0xD1B54A32D192ED03 * iteration)) & m
    z = ((z ^ (z >> 30)) * 0xBF58476D1CE4E5B9) & m
    z = ((z ^ (z >> 27)) * 0x94D049BB133111EB) & m
    return z ^ (z >> 31)


def reduce_measurements(times: dict[str, float], work: dict[str, int], device: str = "cpu"):
    """max-over-ranks of every time, sum-over-ranks of every work counter (an int counter stays an int, a float one -- e.g. a
    mean weighted by its rows -- a float).  No-op without a process group."""
    dist = torch.distributed
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return dict(times), dict(work)
    tk, wk = sorted(times), sorted(work)
    t = torch.tensor([times[k] for k in tk], dtype=torch.float64, device=device)
    w = torch.tensor([float(work[k]) for k in wk], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dist.all_reduce(w, op=dist.ReduceOp.SUM)
    return ({k: float(v) for k, v in zip(tk, t.tolist())},
            {k: float(v) if isinstance(work[k], float) else int(round(v)) for k, v in zip(wk, w.tolist())})


def gather_replay(boards: torch.Tensor, policy: torch.Tensor, status: torch.Tensor, dst: int = 0):
    """Merge per-rank transition blocks ([plies, games, ...]) on rank `dst` along the game axis (config 4's host
    replay buffer).  Returns None on other ranks."""
    dist = torch.distributed
    if not (dist.is_available() and dist.is_initialized()) or dist.get_world_size() == 1:
        return boards, policy, status
    world, rank = dist.get_world_size(), dist.get_rank()
    out = []
    for t in (boards, policy, status):
        t = t.contiguous()
        sizes = [torch.zeros(1, dtype=torch.int64, device=t.device) for _ in range(world)]
        dist.all_gather(sizes, torch.tensor([t.shape[1]], dtype=torch.int64, device=t.device))
        bufs = [torch.empty((t.shape[0], int(s.item())) + tuple(t.shape[2:]), dtype=t.dtype, device=t.device) for s in sizes]
        dist.all_gather(bufs, t) if len({int(s.item()) for s in sizes}) == 1 else _uneven_all_gather(dist, bufs, t, rank)
        out.append(torch.cat(bufs, dim=1) if rank == dst else None)
    return tuple(out) if rank == dst else None


def _uneven_all_gather(dist, bufs, t, rank):
    for src in range(len(bufs)):
        if src == rank:
            bufs[src].copy_(t)
        dist.broadcast(bufs[src], src=src)
