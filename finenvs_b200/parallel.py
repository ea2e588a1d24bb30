"""Env sharding across the GPUs of one box (one process per GPU, torch.distributed).

The step itself needs NO communication: envs are independent (every op of the reference's
time_series_env.py:277-521 is elementwise over the env dimension), the series is replicated on
every GPU, and redraws are keyed by GLOBAL env id so results do not depend on the sharding.
Collectives (NCCL over NVLink; gloo in the CPU tests) appear only where the reference reduces
over envs:

  * episode statistics at log points  (replaces the means/stds of PPO_agent.py:143-145 and
    evo_agent.py:116-123)                    -> all_reduce(sum) of a 5-vector
  * per-episode trading metrics (TimeSeriesEnv.metrics_summary)  -> all_reduce(sum) + all_reduce(max)
  * evaluate mode's "all envs terminated"    (time_series_env.py:531)  -> all_reduce(min)
  * ES fitness (evo_agent.py:173-191: a GLOBAL argsort -> centred ranks)  -> all_gather
"""
from __future__ import annotations

import os
from typing import Dict, Optional, Tuple

import torch
import torch.distributed as dist


def init_distributed(backend: Optional[str] = None) -> Tuple[int, int, int]:
    """(rank, world_size, local_rank) from the torchrun environment; single process without it."""
    if "RANK" not in os.environ or int(os.environ.get("WORLD_SIZE", "1")) == 1:
        return 0, 1, int(os.environ.get("LOCAL_RANK", "0"))
    rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
    local_rank = int(os.environ.get("LOCAL_RANK", rank))
    if not dist.is_initialized():
        if backend is None:
            backend = "nccl" if torch.cuda.is_available() else "gloo"
        kwargs = {}
        if backend == "nccl":
            torch.cuda.set_device(local_rank)
            kwargs["device_id"] = torch.device("cuda", local_rank)
        dist.init_process_group(backend=backend, rank=rank, world_size=world, **kwargs)
    return rank, world, local_rank


def bind_to_gpu_numa(device_index: int):
    """Pin this process to the CPUs NVML reports as local to GPU `device_index` (its NUMA node), so that the pinned host
    buffers it allocates afterwards (first touch) and its driver threads sit next to the GPU's PCIe root.  One process
    per GPU makes this the natural placement; without it every rank's buffers tend to land on one socket and the
    host-buffer step (fe_step_host) of 8 ranks shares that socket's memory and inter-socket links.
    Returns the previous affinity set (hand it to os.sched_setaffinity(0, ...) to undo) or None if nothing was done."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
        ncpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (ncpu + 63) // 64)
        cpus = {64 * w + b for w, word in enumerate(words) for b in range(64) if (int(word) >> b) & 1}
        prev = os.sched_getaffinity(0)
        cpus &= prev
        if not cpus:
            return None
        os.sched_setaffinity(0, cpus)
        return prev
    except Exception:
        return None


def shard_bounds(total_envs: int, rank: int, world_size: int) -> Tuple[int, int]:
    """Contiguous block of global env ids owned by `rank`: (first id, count).  The remainder goes to
    the lowest ranks, so the global last env (the reference's evaluation env) is on the last rank."""
    if not (0 <= rank < world_size) or total_envs < world_size:
        raise ValueError("need 0 <= rank < world_size <= total_envs")
    q, r = divmod(total_envs, world_size)
    count = q + (1 if rank < r else 0)
    base = rank * q + min(rank, r)
    return base, count


def make_sharded_env(total_envs: int, rank: int, world_size: int, *args, **kwargs):
    """TimeSeriesEnv holding this rank's block of a `total_envs` population (device = local GPU)."""
    from .environments.time_series_env import TimeSeriesEnv

    base, count = shard_bounds(total_envs, rank, world_size)
    return TimeSeriesEnv(*args, num_envs=count, env_id_base=base, total_envs=total_envs, **kwargs)


def stats_vector(stats: Dict[str, torch.Tensor]) -> torch.Tensor:
    """[n_done, n_terminated, sum_len, sum_return, sum_return_sq] as one f64 vector (exact for counts < 2^53)."""
    keys = ("n_done", "n_terminated", "sum_len", "sum_return", "sum_return_sq")
    return torch.stack([stats[k].to(torch.float64) for k in keys])


def all_reduce_episode_stats(vec: torch.Tensor, group=None) -> Dict[str, float]:
    """Sum the per-rank statistics vectors and derive the global episode count / mean / std / length."""
    vec = vec.clone()
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(vec, op=dist.ReduceOp.SUM, group=group)
    n, nt, sl, sr, sq = (float(x) for x in vec.tolist())
    mean = sr / n if n else 0.0
    var = max(sq / n - mean * mean, 0.0) if n else 0.0
    return {"episodes": n, "terminated": nt, "mean_return": mean, "std_return": var ** 0.5,
            "mean_length": sl / n if n else 0.0}


def all_reduce_episode_metrics(summary: Dict[str, torch.Tensor], group=None) -> Dict[str, float]:
    """TimeSeriesEnv.metrics_summary() of every rank combined: the sums add, max_mdd is the maximum.  Counts come
    back as ints (exact below 2^53)."""
    keys = [k for k in summary if k != "max_mdd"]
    vec = torch.stack([summary[k].to(torch.float64) for k in keys])
    mx = summary["max_mdd"].to(torch.float64).reshape(1).clone()
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(vec, op=dist.ReduceOp.SUM, group=group)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX, group=group)
    out = {k: (int(v) if k in ("episodes", "sum_len") else v) for k, v in zip(keys, vec.tolist())}
    out["max_mdd"] = float(mx.item())
    return out


def all_terminated(local_flag: torch.Tensor, group=None) -> bool:
    """time_series_env.py:531 torch.all(terminated) over every shard."""
    flag = local_flag.to(torch.int32).reshape(1).clone()
    if dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    return bool(flag.item())


def all_gather_fitness(local: torch.Tensor, total_envs: int, group=None) -> torch.Tensor:
    """Per-env fitness of every shard, in global env-id order, on every rank ((total_envs,) tensor).
    Shards differ by at most one env, so each is padded to the largest block for one all_gather."""
    if not (dist.is_initialized() and dist.get_world_size(group) > 1):
        return local.clone()
    world, rank = dist.get_world_size(group), dist.get_rank(group)
    counts = [shard_bounds(total_envs, r, world)[1] for r in range(world)]
    width = max(counts)
    padded = torch.zeros(width, dtype=local.dtype, device=local.device)
    padded[: counts[rank]] = local
    out = torch.empty(world * width, dtype=local.dtype, device=local.device)
    dist.all_gather_into_tensor(out, padded, group=group)
    return torch.cat([out[r * width: r * width + counts[r]] for r in range(world)])


def centered_ranks(fitness: torch.Tensor) -> torch.Tensor:
    """evo_agent.py:173-186: rank transform to [-0.5, 0.5] from ONE global argsort."""
    order = fitness.argsort()
    ranks = torch.empty(order.shape, dtype=torch.float32, device=fitness.device)
    ranks[order] = torch.arange(0, order.shape[0], dtype=torch.float32, device=fitness.device)
    return ranks / (len(ranks) - 1) - 0.5


def global_centered_ranks(local_fitness: torch.Tensor, total_envs: int, group=None) -> torch.Tensor:
    """This rank's slice of the globally computed centred ranks (identical to the single-GPU result)."""
    full = centered_ranks(all_gather_fitness(local_fitness, total_envs, group))
    if not (dist.is_initialized() and dist.get_world_size(group) > 1):
        return full
    base, count = shard_bounds(total_envs, dist.get_rank(group), dist.get_world_size(group))
    return full[base: base + count]
