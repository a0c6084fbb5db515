"""Batch sharding over the GPUs of one box: one process per GPU, no communication inside the loop,
one all-gather of the code grids at the end (SURVEY.md 8e).

Images are independent, every rank holds a full weight replica and its own KV cache.  The Philox
counter of every draw is (global row, position, slot), so the gathered result is identical to a
single-GPU run of the whole batch, whatever the world size.
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.distributed as dist


def shard_range(global_batch: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Contiguous rows [lo, hi) of rank `rank`; the first `global_batch % world_size` ranks get one extra row."""
    base, rem = divmod(global_batch, world_size)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def gather_codes(codes_top: torch.Tensor, codes_bot: torch.Tensor, global_batch: int,
                 group: Optional[dist.ProcessGroup] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """All-gathers per-rank [b_r, S] / [b_r, S, 4] int64 code grids into [B, S] / [B, S, 4] on every rank.
    One collective on a packed [b_max, S, 5] buffer (2 560 B per image for S = 64)."""
    world = dist.get_world_size(group)
    rank = dist.get_rank(group)
    S = codes_top.shape[1]
    b_max = (global_batch + world - 1) // world
    packed = torch.zeros(b_max, S, 5, dtype=torch.int64, device=codes_top.device)
    n = codes_top.shape[0]
    packed[:n, :, 0] = codes_top
    packed[:n, :, 1:] = codes_bot
    out = torch.empty(world * b_max, S, 5, dtype=torch.int64, device=codes_top.device)
    dist.all_gather_into_tensor(out, packed, group=group)
    parts = []
    for r in range(world):
        lo, hi = shard_range(global_batch, r, world)
        parts.append(out[r * b_max: r * b_max + (hi - lo)])
    full = torch.cat(parts, dim=0)
    assert full.shape[0] == global_batch and shard_range(global_batch, rank, world)[1] - \
        shard_range(global_batch, rank, world)[0] == n
    return full[:, :, 0].contiguous(), full[:, :, 1:].contiguous()


@torch.no_grad()
def sampling_ihqgpt_sharded(model, num_candidates: int, cond, *, gather: bool = True,
                            group: Optional[dist.ProcessGroup] = None, **kw):
    """`sampling_ihqgpt` for a global batch of `num_candidates` rows split over the ranks of `group`.
    cond: class id (int) | int64 [B] per-row classes | int64 [B, ctx_len_txt] text ids | None.
    Returns the full [B, S] / [B, S, 4] grids on every rank (gather=True) or this rank's shard."""
    from .models import fresh_seed
    from .sampling import sampling_ihqgpt
    world = dist.get_world_size(group) if dist.is_initialized() else 1
    rank = dist.get_rank(group) if dist.is_initialized() else 0
    B = num_candidates if not torch.is_tensor(cond) or cond.numel() == 1 else cond.shape[0]
    lo, hi = shard_range(B, rank, world)
    local_cond = cond[lo:hi] if torch.is_tensor(cond) and cond.numel() > 1 else cond
    kw = dict(kw)
    for name in ("prefix_code_top", "prefix_code_bot"):     # image completion: per-row prefixes follow the rows, as cond does
        t = kw.get(name)
        if t is not None and torch.is_tensor(t) and t.shape[0] > 1:
            kw[name] = t[lo:hi]
    if kw.get("seed") is None:
        # one Philox key for the whole global batch: rank 0 draws it from its default generator, everyone uses it
        box = [fresh_seed() if rank == 0 else None]
        if world > 1:
            dist.broadcast_object_list(box, src=dist.get_global_rank(group, 0) if group is not None else 0, group=group)
        kw["seed"] = box[0]
    if hi > lo:
        ct, cb = sampling_ihqgpt(model, hi - lo, local_cond, row_offset=lo, **kw)
    else:
        # more ranks than rows: this rank has nothing to sample but still joins the collective below
        S = kw.get("max_seq_len", 256)
        ct = torch.empty(0, S, dtype=torch.int64, device=model.device)
        cb = torch.empty(0, S, 4, dtype=torch.int64, device=model.device)
    if gather and world > 1:
        return gather_codes(ct, cb, B, group)
    return ct, cb
