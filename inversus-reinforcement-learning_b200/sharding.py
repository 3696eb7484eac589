"""Multi-GPU layout of the rollout path: envs shard, nothing else does.

Envs never interact (inversus_rl/env_wrappers.py:505-519 touches only `self.envs[i]`), so rank r
of G owns the contiguous global env range `shard_range(N, r, G)` and the step path has NO
collective. The draw stream is keyed by GLOBAL env id (`env_id_base`), which makes every env's
trajectory independent of the rank count. The only exchange is the four rollout statistics
(episodes, wins, return sum, length sum), reduced with one tiny all-reduce (NCCL on GPUs, gloo in
the CPU tests).
"""
from __future__ import annotations

import os
from typing import Tuple

import torch


def shard_range(total_envs: int, rank: int, world_size: int) -> Tuple[int, int]:
    """[first, first+count) of global env ids owned by `rank`; sizes differ by at most one."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    base, rem = divmod(int(total_envs), int(world_size))
    count = base + (1 if rank < rem else 0)
    first = rank * base + min(rank, rem)
    return first, count


def dist_env() -> Tuple[int, int, int]:
    """(rank, local_rank, world_size) from the torchrun environment (1 process per GPU)."""
    return (int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)),
            int(os.environ.get("WORLD_SIZE", 1)))


def init_distributed() -> Tuple[int, int, int]:
    """Join the NCCL process group when started by torchrun with more than one process (one GPU each)."""
    rank, local_rank, world = dist_env()
    if world > 1 and not torch.distributed.is_initialized():
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        torch.distributed.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    return rank, local_rank, world


def finish_distributed() -> None:
    """End a torchrun command-line run (no-op without a process group). CUDA graphs may hold NCCL
    kernels: drop them, then give the communicator teardown a bounded time on a side thread (it has
    been seen to block with captured collectives) and leave."""
    if not torch.distributed.is_initialized():
        return
    import gc
    import sys
    import threading
    gc.collect()
    torch.cuda.synchronize()
    torch.distributed.barrier()
    t = threading.Thread(target=torch.distributed.destroy_process_group, daemon=True)
    t.start()
    t.join(20.0)
    sys.stdout.flush()
    sys.stderr.flush()
    os._exit(0)


def reduce_rollout_stats(episodes, wins, return_sum, length_sum, device=None) -> Tuple[float, float, float, float]:
    """Sum the four rollout statistics over ranks (no-op without an initialised process group)."""
    t = torch.tensor([float(episodes), float(wins), float(return_sum), float(length_sum)],
                     dtype=torch.float64, device=device)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM)
    e, w, r, l = t.tolist()
    return e, w, r, l


def max_over_ranks(value: float, device=None) -> float:
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())
