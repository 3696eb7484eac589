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
from fractions import Fraction
from typing import Dict, List, Tuple

import torch


def shard_range(total_envs: int, rank: int, world_size: int) -> Tuple[int, int]:
    """[first, first+count) of global env ids owned by `rank`; sizes differ by at most one."""
    if not (0 <= rank < world_size):
        raise ValueError("rank out of range")
    base, rem = divmod(int(total_envs), int(world_size))
    count = base + (1 if rank < rem else 0)
    first = rank * base + min(rank, rem)
    return first, count


OPPONENT_SLOTS = ("easy", "hard", "latest", "pool")


def _largest_remainder(total: int, weights) -> List[int]:
    """Split `total` into integer parts proportional to `weights` (exact fractions): each part gets
    the floor of its quota, and the rest go one each to the largest fractional remainders, ties to
    the earlier part."""
    wsum = sum(weights)
    quotas = [total * w / wsum for w in weights]
    parts = [int(q) for q in quotas]  # floor: quotas are non-negative
    order = sorted(range(len(weights)), key=lambda i: (-(quotas[i] - parts[i]), i))
    for i in order[:total - sum(parts)]:
        parts[i] += 1
    return parts


def parse_opponent_mix(spec) -> Dict[str, Fraction]:
    """"hard=0.25,latest=0.25,pool=0.5" (or a dict) -> {slot: weight}, weights normalised to sum 1.
    Slots: easy, hard (the scripted dummy), latest (the lagged copy of the learner), pool (older
    snapshots). Raises ValueError on an unknown or repeated slot, a negative weight or a zero sum."""
    items = spec.items() if isinstance(spec, dict) else [kv.split("=", 1) if "=" in kv else (kv, None)
                                                         for kv in str(spec).split(",") if kv.strip()]
    mix: Dict[str, Fraction] = {}
    for k, v in items:
        k = str(k).strip()
        if k not in OPPONENT_SLOTS:
            raise ValueError(f"opponent_mix: unknown slot {k!r} (slots: {', '.join(OPPONENT_SLOTS)})")
        if k in mix:
            raise ValueError(f"opponent_mix: slot {k!r} given twice")
        try:
            w = Fraction(str(v).strip())
        except (TypeError, ValueError, ZeroDivisionError):
            raise ValueError(f"opponent_mix: weight of {k!r} is not a number: {v!r}") from None
        if w < 0:
            raise ValueError(f"opponent_mix: weight of {k!r} is negative")
        mix[k] = w
    total = sum(mix.values())
    if not mix or total <= 0:
        raise ValueError("opponent_mix: the weights must sum to more than 0")
    return {k: w / total for k, w in mix.items()}


def opponent_ranges(num_envs: int, mix, pool_size: int = 4) -> List[Tuple[str, int, int]]:
    """The static opponent of every global env id: [(opponent, lo, hi)] in the fixed slot order easy,
    hard, latest, pool[0] .. pool[M-1], contiguous, covering [0, num_envs) once. Slot sizes follow
    the largest-remainder rule over the normalised weights; the pool range is split into `pool_size`
    equal parts the same way. A slot (or pool snapshot) with weight > 0 but no env is a ValueError.
    The map does not depend on the GPU count: each rank intersects it with its shard_range."""
    mix = parse_opponent_mix(mix)
    if int(pool_size) < 1:
        raise ValueError("pool_size must be at least 1")
    weights = [mix.get(k, Fraction(0)) for k in OPPONENT_SLOTS]
    sizes = _largest_remainder(int(num_envs), weights)
    out, lo = [], 0
    for slot, w, size in zip(OPPONENT_SLOTS, weights, sizes):
        if w == 0:
            continue
        parts = _largest_remainder(size, [1] * int(pool_size)) if slot == "pool" else [size]
        if min(parts) == 0:
            raise ValueError(f"opponent_mix: slot {slot!r} gets {size} of {num_envs} envs"
                             + (f", fewer than pool_size={pool_size}" if slot == "pool" else ""))
        for j, m in enumerate(parts):
            out.append((f"pool[{j}]" if slot == "pool" else slot, lo, lo + m))
            lo += m
    return out


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


def sum_over_ranks(t: torch.Tensor) -> torch.Tensor:
    """All-reduce (sum) `t` in place over ranks (no-op without an initialised process group)."""
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.SUM)
    return t


def max_over_ranks(value: float, device=None) -> float:
    t = torch.tensor([float(value)], dtype=torch.float64, device=device)
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    return float(t.item())
