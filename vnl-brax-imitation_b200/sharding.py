"""Env sharding over the GPUs of one box.

The hot path has no cross-env coupling: the reference splits `num_envs` evenly over local devices
(`ppo_imitation/train.py:195,216-217`, `pmap` at `:363`) and `env.step` contains no collective.
Here: one process per GPU (torchrun), each owns a contiguous env range; the only communication is
metric / timing reduction through `torch.distributed` (NCCL on GPUs, gloo in the CPU tests).
"""
from __future__ import annotations

import os
from typing import Dict, Tuple


def env_info() -> Tuple[int, int, int]:
    """(rank, local_rank, world_size) from the torchrun environment (1-process defaults)."""
    return int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))


def shard_range(num_envs: int, rank: int, world_size: int) -> Tuple[int, int]:
    """[lo, hi) of the global env ids owned by `rank`; sizes differ by at most one.

    The reference asserts `num_envs % device_count == 0` (`ppo_imitation/train.py:192-195`); when that
    holds this is exactly its `num_envs // device_count` contiguous split."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    base, rem = divmod(int(num_envs), int(world_size))
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def init_process_group(backend: str = "nccl"):
    import torch.distributed as dist

    rank, local_rank, world = env_info()
    if world > 1 and not dist.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("MASTER_PORT", "29500")
        kw = {}
        if backend == "nccl":  # bind the communicator to this rank's GPU (no device guessing at the first barrier)
            import torch
            kw["device_id"] = torch.device("cuda", local_rank)
        dist.init_process_group(backend=backend, rank=rank, world_size=world, **kw)
    return rank, local_rank, world


def group():
    """`torch.distributed` when a process group with more than one rank is initialised, else None: the one test of whether
    there is anybody to exchange with."""
    import torch.distributed as dist

    return dist if dist.is_available() and dist.is_initialized() and dist.get_world_size() > 1 else None


def barrier():
    dist = group()
    if dist is not None:
        dist.barrier()


def reduce_scalars(values: Dict[str, float], op: str = "sum", device=None) -> Dict[str, float]:
    """All-reduce a small dict of python floats (metric / timing reduction); identity at world size 1."""
    import torch

    dist = group()
    if dist is None:
        return dict(values)
    keys = sorted(values)
    t = torch.tensor([float(values[k]) for k in keys], dtype=torch.float64, device=device)
    if dist.get_backend() == "nccl" and t.device.type != "cuda":
        t = t.cuda()
    dist.all_reduce(t, op={"sum": dist.ReduceOp.SUM, "max": dist.ReduceOp.MAX, "min": dist.ReduceOp.MIN}[op])
    return {k: float(v) for k, v in zip(keys, t.cpu().tolist())}
