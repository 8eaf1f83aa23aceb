"""Data-parallel plumbing of FQLAgent.update (SURVEY 8e): the batch shards by rows, every rank runs the loss/gradient half
of the step on its rows with loss denominators of the GLOBAL batch (FqlDims.global_batch), the flat gradient arena and
the raw metric accumulators are all-reduced, and every rank applies the identical Adam/Polyak step (no parameter
broadcast).  Nothing here touches CUDA directly, so the same functions run under gloo on CPU in the tests.

The reference itself is single-device (no pmap/shard_map anywhere, SURVEY 2.1): this module is new capability, not a port.
"""
from __future__ import annotations

import torch
import torch.distributed as dist

RAW_SUM = slice(0, 9)    # include/fql_b200.h: raw[0..8] are sums
RAW_MAX = slice(9, 11)   # raw[9] = max q, raw[10] = -min q


def shard_rows(batch: dict, rank: int, world: int) -> dict:
    """Rank r takes rows [r*B/R, (r+1)*B/R) of every array of the GLOBAL batch / noise dict (same global index draw on every
    rank, so R ranks reproduce the 1-rank step on the concatenated batch)."""
    out = {}
    for k, v in batch.items():
        n = v.shape[0]
        if n % world:
            raise ValueError(f'batch rows ({n}) must divide evenly over {world} ranks')
        per = n // world
        out[k] = v[rank * per:(rank + 1) * per]
    return out


def allreduce_step(grads: torch.Tensor, raw: torch.Tensor, group=None) -> None:
    """In-place reduction of the gradient arena (all-reduce SUM) and of the raw accumulators (one all-gather of the 16 floats per
    seed, reduced locally: SUM for the sums, MAX for max q / -min q) -- two collectives per step."""
    dist.all_reduce(grads, op=dist.ReduceOp.SUM, group=group)
    world = dist.get_world_size(group)
    flat = raw.contiguous().reshape(-1)
    gathered = torch.empty(world * flat.numel(), dtype=raw.dtype, device=raw.device)
    dist.all_gather_into_tensor(gathered, flat, group=group)
    gathered = gathered.reshape((world,) + tuple(raw.shape))
    raw[..., RAW_SUM] = gathered[..., RAW_SUM].sum(dim=0)
    raw[..., RAW_MAX] = gathered[..., RAW_MAX].max(dim=0).values


def gather_raw(raw: torch.Tensor, group=None) -> torch.Tensor:
    """All-gather of the per-rank accumulators -> [world, S, 16]; the SUM / MAX reduction over ranks happens inside
    fql_step_apply_gathered (one collective, no host-side reduction kernels)."""
    world = dist.get_world_size(group)
    flat = raw.contiguous().reshape(-1)
    out = torch.empty(world * flat.numel(), dtype=raw.dtype, device=raw.device)
    dist.all_gather_into_tensor(out, flat, group=group)
    return out.reshape((world,) + tuple(raw.shape))


def shard_seeds(num_seeds: int, rank: int, world: int) -> range:
    """Multi-seed runs (BASELINE config 4) shard by agent: no collective on the step."""
    if num_seeds % world:
        raise ValueError(f'{num_seeds} seeds do not divide over {world} ranks')
    per = num_seeds // world
    return range(rank * per, (rank + 1) * per)


def shard_per_seed(per_seed, rank: int, world: int):
    """FQLAgent.create(per_seed=...) of rank r under seed sharding: every sequence sliced to the seeds shard_seeds gives the rank, so
    each rank's agents train with their own hyperparameters.  None stays None."""
    if per_seed is None:
        return None
    lengths = {len(v) for v in per_seed.values()}
    if len(lengths) > 1:
        raise ValueError(f'per_seed sequences differ in length: { {k: len(v) for k, v in per_seed.items()} }')
    if not lengths:
        return {}
    r = shard_seeds(lengths.pop(), rank, world)
    return {k: list(v)[r.start:r.stop] for k, v in per_seed.items()}
