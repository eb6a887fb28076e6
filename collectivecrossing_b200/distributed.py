"""Sharding of N independent envs over the GPUs of one node (one process per GPU, torchrun).

Envs never interact, so the data path needs no collective: every rank owns a contiguous block of
envs and runs the same fused kernel on it.  The counter-based RNG is keyed on the GLOBAL env
index (``global_env_offset``), hence a sharded run reproduces the single-GPU run env by env.
The only exchange is the episode-statistics reduction: one ``all_reduce(SUM)`` of eight float64
scalars per rollout chunk (NCCL over NVLink on GPUs, gloo in the CPU tests).
"""

from __future__ import annotations

from typing import Any, Callable

import torch
import torch.distributed as dist

STAT_KEYS = ("env_steps", "episodes", "terminated_all", "truncated_all", "arrivals", "episode_length_sum",
             "episode_return_sum", "reward_sum")


def world() -> tuple[int, int]:
    """(rank, world_size) of the default process group, (0, 1) when none is initialised."""
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


def shard_range(total_envs: int, rank: int, world_size: int) -> tuple[int, int]:
    """Contiguous block of rank ``rank``: (first global env, number of envs).  The remainder goes
    to the lowest ranks, so block sizes differ by at most one."""
    if not 0 <= rank < world_size:
        raise ValueError(f"rank {rank} outside world of {world_size}")
    base, extra = divmod(int(total_envs), world_size)
    count = base + (1 if rank < extra else 0)
    offset = rank * base + min(rank, extra)
    return offset, count


def reduce_stats(local: dict, device: Any = "cpu") -> dict:
    """Sum the per-rank statistics dicts over the default process group (counts stay exact: they
    are far below 2**53)."""
    rank, size = world()
    if size == 1:
        return dict(local)
    t = torch.tensor([float(local[k]) for k in STAT_KEYS], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    out = {k: (int(round(v)) if k not in ("episode_return_sum", "reward_sum") else v) for k, v in zip(STAT_KEYS, t.tolist())}
    return out


def derived_stats(stats: dict) -> dict:
    """Mean episode return / length and outcome fractions (what RLlib reports as
    episode_return_mean etc., reference examples/training_script.py:92-98)."""
    ep = max(1, stats["episodes"])
    return {
        "episode_return_mean": stats["episode_return_sum"] / ep,
        "episode_len_mean": stats["episode_length_sum"] / ep,
        "terminated_fraction": stats["terminated_all"] / ep,
        "truncated_fraction": stats["truncated_all"] / ep,
        "reward_per_env_step": stats["reward_sum"] / max(1, stats["env_steps"]),
    }


def host_threads_per_rank() -> int:
    """Host threads one rank may use for the host-buffer path when several ranks share a node (torchrun sets
    LOCAL_WORLD_SIZE); 0 = alone on the node, keep the library's automatic choice."""
    import os

    local_world = int(os.environ.get("LOCAL_WORLD_SIZE", "1"))
    if local_world <= 1:
        return 0
    return max(2, (os.cpu_count() or 1) // local_world)


class ShardedCollectiveCrossing:
    """``total_envs`` envs split over the ranks of the default process group.

    ``env_factory(config, num_envs, global_env_offset=..., seed=..., **kw)`` builds the rank-local
    env; by default the CUDA ``BatchedCollectiveCrossing`` on ``cuda:LOCAL_RANK``.  ``env_kwargs`` (``obs_dtype``,
    ``reset_rng``, ...) go to every rank's env.
    """

    def __init__(self, config: Any, total_envs: int, *, seed: int = 0, device: Any = None,
                 env_factory: Callable[..., Any] | None = None, **env_kwargs: Any):
        self.rank, self.world_size = world()
        self.total_envs = int(total_envs)
        self.offset, self.count = shard_range(self.total_envs, self.rank, self.world_size)
        if self.count == 0:
            raise ValueError(f"rank {self.rank} would own no env: use at most {self.total_envs} ranks")
        if env_factory is None:
            from .batched import BatchedCollectiveCrossing

            if device is None:
                # one process per GPU under torchrun: the rank's own device, not whatever happens to be current
                import os

                local = os.environ.get("LOCAL_RANK")
                if local is not None:
                    torch.cuda.set_device(int(local))
                elif self.world_size > 1:
                    raise ValueError("world_size > 1 without LOCAL_RANK: pass device=... (every rank would land on cuda:0)")
                device = torch.device("cuda", torch.cuda.current_device())
            env_factory = lambda cfg, n, **kw: BatchedCollectiveCrossing(cfg, n, device, **kw)  # noqa: E731
        self.device = device
        self.env = env_factory(config, self.count, global_env_offset=self.offset, seed=seed, **env_kwargs)
        self.host_threads = host_threads_per_rank()
        od = getattr(self.env, "obs_dtype", None)
        if self.host_threads and hasattr(self.env, "set_host_expand") and (od == "float32" or (od == "int8" and self.env.num_agents == 8)):
            # the ranks of a node share its cores AND its PCIe / memory paths: each rebuilds its rows with its share of the threads
            # (the formats for which the library's automatic choice does so on a single GPU)
            self.env.set_host_expand(self.host_threads)

    def __getattr__(self, name: str) -> Any:  # reset / step / rollout / policy_actions / observe ...
        return getattr(self.env, name)

    def local_stats(self) -> dict:
        st = self.env.stats
        return st() if callable(st) else st

    def global_stats_device(self) -> torch.Tensor:
        """Episode statistics summed over the ranks as a float64 [8] DEVICE tensor (``STAT_KEYS`` order): the per-rank block is
        copied on the device and all-reduced (NCCL) behind the step kernels — nothing waits on the host, so a rollout loop can
        call this once per chunk.  ``stats_from_tensor`` turns the result into the dict ``global_stats`` returns."""
        t = self.env.stats_device()
        if self.world_size > 1:
            dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t

    @staticmethod
    def stats_from_tensor(t: torch.Tensor) -> dict:
        out = {k: (int(round(v)) if k not in ("episode_return_sum", "reward_sum") else v) for k, v in zip(STAT_KEYS, t.tolist())}
        out.update(derived_stats(out))
        return out

    def global_stats(self) -> dict:
        dev = self.device if (self.device is not None and dist.is_initialized() and dist.get_backend() == "nccl") else "cpu"
        out = reduce_stats(self.local_stats(), dev)
        out.update(derived_stats(out))
        return out
