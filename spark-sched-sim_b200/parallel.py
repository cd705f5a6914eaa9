"""Multi-GPU plumbing: environments shard over ranks, nothing else crosses GPUs.

The reference parallelises rollouts as `num_sequences x num_rollouts` CPU processes
(trainers/trainer.py:264-293): worker `i` uses `base_seed = seed + i // num_rollouts` and re-seeds
with `base_seed + num_sequences * reset_count` (trainers/rollout_worker.py:118-120), then sends its
statistics to the learner over a Pipe (rollout_worker.py:122-129).  Here one process per GPU owns a
contiguous block of environments; the only exchange step is an all-reduce (sum) of the statistics
vector -- NCCL on device tensors in production, gloo on CPU tensors in the tests.
"""
from __future__ import annotations

import numpy as np
import torch
import torch.distributed as dist

STAT_KEYS = ("decisions", "events", "sched_scans", "sum_nodes", "sum_edges", "sum_jobs",
             "observations", "episodes")


def shard_range(total_envs: int, rank: int, world: int) -> tuple[int, int]:
    """[lo, hi) of the global environment ids owned by `rank` (contiguous, sizes differ by <= 1)."""
    base, rem = divmod(total_envs, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


def shard_seeds(base_seed: int, envs_per_rank: int, rank: int, world: int) -> tuple[np.ndarray, int]:
    """Seeds of this rank's environments and the auto-reset seed step: env g (global id) plays
    episodes seeded base_seed + g + (envs_per_rank * world) * k, k = 0, 1, ... -- disjoint over
    ranks, envs and resets."""
    g = rank * envs_per_rank + np.arange(envs_per_rank, dtype=np.uint64)
    return (np.uint64(base_seed) + g).astype(np.uint64), envs_per_rank * world


def reference_worker_seeds(seed: int, num_sequences: int, num_rollouts: int) -> tuple[np.ndarray, int]:
    """The reference trainer's scheme for `num_sequences * num_rollouts` environments: rollouts of
    the same job sequence share a seed (trainer.py:268-270); seed step = num_sequences."""
    i = np.arange(num_sequences * num_rollouts)
    return (seed + i // num_rollouts).astype(np.uint64), num_sequences


def allreduce_stats(stats: dict, device: torch.device | str = "cpu", group=None) -> dict:
    """Sums the per-rank statistics dict over all ranks (no-op without an initialised group)."""
    vec = torch.tensor([float(stats[k]) for k in STAT_KEYS], dtype=torch.float64, device=device)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(vec, op=dist.ReduceOp.SUM, group=group)
    return {k: float(v) for k, v in zip(STAT_KEYS, vec.tolist())}


def allreduce_gradients(grads: torch.Tensor, num_samples: int, group=None) -> tuple[torch.Tensor, int]:
    """Data-parallel policy update: every rank holds d(sum of its samples' loss terms)/d(theta) as one flat vector
    (the layout of ssb_set_decima_weights / ssb_adam_step; = its mini-batch size x the gradient that follows from
    ssb_ppo_loss's adjoint seeds, which carry the local 1/n).  Sums the vectors and the sample counts over the ranks in
    ONE all-reduce (the count rides as a last element) and divides, so that every rank steps Adam with the gradient
    of the mean loss over all ranks' samples -- what the reference's single learner computes over all workers'
    rollouts (trainers/ppo.py:52-70).  In place on `grads`; returns (grads, total samples)."""
    assert grads.dim() == 1 and grads.is_floating_point()
    buf = torch.empty(grads.numel() + 1, dtype=grads.dtype, device=grads.device)
    buf[:-1] = grads
    buf[-1] = float(num_samples)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    total = int(round(float(buf[-1].item())))
    grads.copy_(buf[:-1] / max(total, 1))
    return grads, total


def allreduce_weighted_mean(value: torch.Tensor, weight: float, group=None) -> float:
    """Mean of a per-rank scalar weighted by the ranks' sample counts (one all-reduce of two numbers): the collective
    form of a statistic that decides control flow, e.g. PPO's approximate-KL early stop -- every rank gets the same
    number, so every rank takes the same branch."""
    buf = torch.empty(2, dtype=torch.float64, device=value.device)
    buf[0] = value.reshape(-1)[0].double() * float(weight)
    buf[1] = float(weight)
    if dist.is_available() and dist.is_initialized() and dist.get_world_size(group) > 1:
        dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    s, w = buf.tolist()
    return s / w if w else 0.0


def rollout_summary(sum_job_time: float, sum_wall_time: float, num_completed: float,
                    num_arrived: float, sum_completed_duration: float) -> dict:
    """collect_stats (rollout_worker.py:122-129) from sums that can be all-reduced:
    avg_num_jobs = total job-time / total wall time (metrics.py:15-16)."""
    return {
        "avg_job_duration": (sum_completed_duration / num_completed * 1e-3) if num_completed else float("nan"),
        "avg_num_jobs": (sum_job_time / sum_wall_time) if sum_wall_time else float("nan"),
        "num_completed_jobs": num_completed,
        "num_job_arrivals": num_arrived,
    }


def stats_from_sums(vec) -> dict:
    """The reference's per-iteration statistics (trainer.py:310-320 averages the workers' collect_stats dicts)
    from the (all-reduced) ssb_collect_stats vector.  With an episode log attached ([7] > 0: envs that have a
    completed job in their window), avg_job_duration is the mean over those envs of their window's mean -- the
    trainer's mean over workers of env.avg_job_duration (the last 200 completions, across resets); otherwise the
    mean duration of the jobs completed in the live episodes."""
    v = [float(x) for x in (vec.tolist() if hasattr(vec, "tolist") else vec)]
    n = max(v[1], 1.0)
    if len(v) > 7 and v[7] > 0:
        avg_dur = v[6] / v[7] * 1e-3
    else:
        avg_dur = (v[4] / v[2] * 1e-3) if v[2] else float("nan")
    return {"avg_num_jobs": v[0] / n, "num_completed_jobs": v[2] / n, "num_job_arrivals": v[3] / n,
            "avg_job_duration": avg_dur}
